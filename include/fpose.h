/* fpose.h — C ABI of libfpose.so, the B200-native (sm_100a) render-and-compare hot path behind
 * NVlabs/FoundationPose's Python surfaces.
 *
 * Every entry point is `extern "C"`, takes plain pointers and sizes, returns 0 on success or a
 * negative error code (fp_last_error() returns a thread-local message); nothing throws or aborts.
 * All `void* stream` arguments are a cudaStream_t (pass torch.cuda.current_stream().cuda_stream);
 * all work is enqueued on that stream and is asynchronous unless stated otherwise.
 * Device pointers are owned by the caller; the library owns only what it allocates inside an
 * fp_ctx (packed weights, mesh copy, frame copy, workspaces).
 *
 * Each declaration cites the reference interface it replaces (paths relative to the
 * FoundationPose repository root).
 */
#ifndef FPOSE_H_
#define FPOSE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------------------------ */
/* errors / counters                                                                          */
/* ------------------------------------------------------------------------------------------ */
const char* fp_last_error(void);
/* Number of CUDA kernels this library has launched so far in this process (bench.py's
 * `gpu_launches`). */
unsigned long long fp_launch_count(void);

/* Per-launch device timing of the two roofline kernels (CUDA events on the launching stream):
 * kind 0 = tcgen05 implicit-GEMM kernel (work = algorithmic FLOPs), kind 1 = crop producer
 * (work = algorithmic output bytes).  fp_prof_collect synchronises the device, returns and clears
 * the sums accumulated since fp_prof_enable(1). */
int fp_prof_enable(int on);
int fp_prof_collect(int kind, double* total_ms, double* total_work, int* launches);

/* ------------------------------------------------------------------------------------------ */
/* single operators (parity-test hooks; the product path below calls the same code)           */
/* ------------------------------------------------------------------------------------------ */

/* kinds of dense layer the tcgen05 implicit-GEMM kernel executes */
#define FP_LAYER_LINEAR 0   /* torch.nn.Linear / in_proj / out_proj (refine_network.py:56-70)      */
#define FP_LAYER_CONV3_S1 1 /* 3x3 s1 p1 conv of ResnetBasicBlock (network_modules.py:73-111)       */
#define FP_LAYER_CONV3_S2 2 /* 3x3 s2 p1 ConvBNReLU (refine_network.py:37, :45)                      */
#define FP_LAYER_CONV7_S2 3 /* 7x7 s2 p3 stem ConvBNReLU (refine_network.py:36)                      */

typedef struct fp_gemm_layer {
  int kind;
  int n_img;          /* images in the batch (LINEAR: 1)                                          */
  int Hin, Win;       /* un-padded input size (LINEAR: Hin = 1, Win = number of rows M)           */
  int Cin;            /* input channels (LINEAR: K; CONV7_S2: 8 = 6 real + 2 zero)                */
  int Cout;           /* output channels, multiple of 64                                          */
  const void* in;     /* fp16; NHWC.  CONV7_S2: [n][Hin+6][2][(Win+8)/2][8] = a zero-bordered
                         (Hin+6) x (Win+8) canvas, image at (3,3), every row stored as its even
                         columns then its odd columns (packing.pad_image_c8)                      */
  const void* w;      /* fp16 [Cout][taps*Cin] (tap-major, channel-minor); CONV7_S2:
                         [7 rows][4 tap pairs][2][64][8] (packing.pack_conv7)                     */
  const float* bias;  /* fp32 [Cout] (BatchNorm folded in)                                        */
  const void* res;    /* optional fp16 residual, same indexing as the output, leading dim res_ld  */
  int res_ld;
  void* out;          /* fp16 NHWC output                                                         */
  int out_ld;         /* elements between consecutive output pixels                               */
  int out_split;      /* >0: image n goes to image n % out_split at channel (n / out_split)*Cout;
                         must be a multiple of the tile's image count (2 for >= 8x8 outputs, else 8)  */
  const float* post_add; /* optional fp32 [Ho*Wo][Cout], added after the activation               */
  int relu;
} fp_gemm_layer_t;

/* Runs one layer: out = act(in (*) w + bias [+ res]) [+ post_add]. */
int fp_op_gemm_layer(const fp_gemm_layer_t* layer, void* stream);

/* softmax(Q K^T / sqrt(128)) V of nn.MultiheadAttention (refine_network.py:56-70, score_network.py:53):
 * qkv fp16 [B*400][1536] (q | k | v, 4 heads of 128 each), out fp16 [B*400][512].
 * `impl` is ignored (kept for ABI stability): there is one implementation, the tcgen05 kernel. */
int fp_op_attention(const void* qkv, void* out, int B, int impl, void* stream);
/* The same attention in the two layouts the product runs: n_groups = 1 is the scorer's (score_network.py:53;
 * qkv [B*400][1536], out [B*400][512]), n_groups = 2 the refiner's two heads in one launch (refine_network.py:56-70;
 * qkv [B*400][3072] = head 0's q | k | v then head 1's, out [2][B*400][512]). */
int fp_op_attention_grouped(const void* qkv, void* out, int B, int n_groups, void* stream);

/* What the last fp_op_gemm_layer / product GEMM launch on the calling thread chose (host-side record, no
 * synchronisation).  Writes min(n, FP_GEMM_PLAN_FIELDS) ints:
 *   [0] kernel: 0 = gemm_tile_kernel, 1 = gemm_swap_kernel, 2 = gemm_swap_patch_kernel, 3 = stem_conv_kernel
 *   [1] output channels per tile  [2] CTAs per MMA (cta_group)  [3] epilogue staging slabs (tile kernel, else 0)
 *   [4] patch mode: 0 = one TMA box per filter tap, 1 = one halo'd patch per channel chunk, 2 = column-shifted copies
 *   [5] grid  [6] work tiles: loop iterations summed over the grid (a CTA runs ceil([6] / [5]) of them)
 *   [7..9] one M tile = [7] x [8] pixels (columns x rows) of [9] images (LINEAR: [7] = 128 rows)
 *   [10] M tiles  [11] channel blocks per M tile
 * Returns -1 if this thread has launched no GEMM yet.  Layers that produce nothing (0 images) leave it unchanged. */
#define FP_GEMM_PLAN_FIELDS 12
int fp_op_gemm_last_plan(int* out, int n);


/* ------------------------------------------------------------------------------------------ */
/* product path                                                                               */
/* ------------------------------------------------------------------------------------------ */
typedef struct fp_ctx fp_ctx;

/* Creates a context on the current CUDA device (must be sm_100).  Replaces the implicit global
 * state of the reference predictors (`.cuda()` modules, nvdiffrast `RasterizeCudaContext`,
 * estimater.py:29-41, :166-171). */
int fp_create(fp_ctx** ctx);
int fp_destroy(fp_ctx* ctx);

/* Per-predictor configuration, as each reference predictor reads its own config.yml: which = 0 the refiner's
 * crop_ratio (predict_pose_refine.py:117-118) and rot_normalizer (cfg['rot_normalizer'], :221); which = 1 the
 * scorer's crop_ratio (predict_score.py:137-138; rot_normalizer ignored). */
int fp_set_config(fp_ctx* ctx, int which, float crop_ratio, float rot_normalizer);

/* One named host tensor of a packed network (see foundationpose_b200/engine.py for the packing:
 * BatchNorm folded, conv weights K-major fp16).  dtype: 0 = float32, 1 = float16. */
typedef struct fp_tensor {
  const char* name;
  const void* data; /* HOST pointer */
  int dtype;
  long long numel;
} fp_tensor_t;

/* which: 0 = RefineNet (predict_pose_refine.py:133-143 `load_state_dict`), 1 = ScoreNetMultiPair
 * (predict_score.py:146-156).  Copies to device memory owned by the context; validates names/sizes. */
int fp_load_network(fp_ctx* ctx, int which, const fp_tensor_t* tensors, int n);

/* Replaces Utils.py:104-130 `make_mesh_tensors` (HOST pointers; uv already v-flipped as in :117;
 * texture uint8 RGB [Ht][Wt][3]; pass uv = tex = NULL and vcol (float 0..1, [V][3]) for
 * vertex-coloured meshes).  diameter = estimater.py:54. */
int fp_set_mesh(fp_ctx* ctx, int V, int F, const float* pos, const float* nrm, const float* uv, const float* vcol,
                const int* faces, const unsigned char* tex_rgb, int Ht, int Wt, float diameter);
/* What fp_set_mesh derived (test hook): info[5] = {meshlets, mesh is closed and consistently oriented (0/1),
 * front-face winding sign used for back-face culling (0 = both sides are rendered, as nvdiffrast does), V, F}. */
int fp_mesh_info(fp_ctx* ctx, int* info);

#define FP_FRAME_ON_DEVICE 1    /* rgb/depth are device pointers (default: host, copied on `stream`) */
#define FP_FRAME_FILTER_DEPTH 2 /* erode_depth + bilateral_filter_depth (estimater.py:173-174, :257-258) */
/* Uploads one RGB-D frame (rgb uint8 [H][W][3], depth float32 [H][W] metres, K row-major 3x3), runs
 * the depth filters (Utils.py:304-395) and depth2xyzmap (Utils.py:399-438; zfar as in :426, use
 * INFINITY for register()).  Asynchronous on `stream`. */
int fp_set_frame(fp_ctx* ctx, const unsigned char* rgb, const float* depth, const float* K, int H, int W, int flags,
                 float zfar, void* stream);
/* Replaces the xyz map derived by fp_set_frame with the caller's own (PoseRefinePredictor.predict's `xyz_map`
 * argument, predict_pose_refine.py:150,177): float32 [H][W][3], host or device pointer. */
int fp_set_xyz_map(fp_ctx* ctx, const float* xyz, void* stream);
/* Copies the filtered depth [H][W] and/or the xyz map [H][W][3] to device buffers (test hook). */
int fp_get_depth(fp_ctx* ctx, float* depth_out_dev, float* xyz_out_dev, void* stream);

/* FoundationPose.guess_translation (estimater.py:137-156: centre of the mask's bounding box, median of the
 * masked valid depths of the CURRENT FILTERED frame) and generate_random_pose_hypo (estimater.py:127-134,
 * :203-209) on the device: mask uint8/bool [H][W] (host, or device if mask_on_device), rot_grid [N][16]
 * device -> poses_out [N][16] device (grid rotations, guessed translation) and info_out[4] device =
 * {tx, ty, tz, number of valid masked pixels (the `valid.sum() < 4` test of estimater.py:183)}. */
int fp_start_poses(fp_ctx* ctx, const unsigned char* mask, int mask_on_device, const float* rot_grid, int N,
                   float* poses_out, float* info_out, void* stream);

/* make_crop_data_batch (predict_pose_refine.py:25-89 for mode 0, predict_score.py:56-114 for mode 1):
 * poses [N][16] device.  Fills the context's crop buffer; optionally copies it to crops_out
 * (fp16 [2N][166][2][84][8]: images 0..N-1 rendered, N..2N-1 observed), an fp32 copy of the
 * normalised crops to dbg_out ([N][2][160][160][6]) and the crop windows to win_out
 * ([N][4] = left, top, sx, sy of tf_to_crop). */
int fp_make_crops(fp_ctx* ctx, const float* poses, int N, int mode, void* crops_out, float* dbg_out, float* win_out,
                  void* stream);
/* Tile edge of the crop producer: 0 = chosen from the batch size (80 px for >= 64 hypotheses, 32 px, 16 px for < 4),
 * or force 16 / 32 / 80 (A/B measurements and the tile-size invariance test: the crops do not depend on it). */
int fp_set_crop_tile(fp_ctx* ctx, int tile);
/* Work counters of one crop pass (profiling hook; synchronises): stats_out_host[4] = {meshlet visits, triangles set
 * up, fragments depth-tested, triangles that took the near-plane path}. */
int fp_crop_stats(fp_ctx* ctx, const float* poses, int N, int mode, int* stats_out_host, void* stream);

/* PoseRefinePredictor.predict (predict_pose_refine.py:149-239) without the host round trips: poses
 * in/out are DEVICE [N][16]; last_trans [N][3] / last_rot [N][9] (optional) receive
 * `last_trans_update` / `last_rot_update` (:238-239). */
int fp_refine(fp_ctx* ctx, const float* poses_in, int N, int iterations, float* poses_out, float* last_trans,
              float* last_rot, void* stream);

/* ScorePredictor.predict (predict_score.py:160-214): scores_out DEVICE [N] (= logits + 100),
 * best_out DEVICE int (first index of the maximum = ids[0] of estimater.py:226). */
int fp_score(fp_ctx* ctx, const float* poses, int N, float* scores_out, int* best_out, void* stream);
/* The two halves of fp_score, split where the hypothesis batch shards across GPUs: per-hypothesis
 * features (score_network.py:60-74), then — after an all-gather of the [N][512] features — the
 * cross-hypothesis attention + linear + argmax (score_network.py:84-88). */
int fp_score_features(fp_ctx* ctx, const float* poses, int N, float* feats_out, void* stream);
int fp_score_tail(fp_ctx* ctx, const float* feats, int L, float* scores_out, int* best_out, void* stream);

/* Hot loop of FoundationPose.register (estimater.py:203-235) with HOST buffers: uploads the N
 * start poses, refines `iterations` times, scores, and returns refined poses [N][16], scores [N]
 * and the best index.  Synchronises `stream` before returning. */
int fp_register(fp_ctx* ctx, const float* poses_host, int N, int iterations, float* poses_out_host,
                float* scores_out_host, int* best_out_host, void* stream);

/* FoundationPose.track_one (estimater.py:250-268) as ONE CUDA-graph launch per frame: upload of the frame (HOST rgb
 * uint8 [H][W][3], depth float32 [H][W]; staged through pinned memory owned by the context), erode_depth +
 * bilateral_filter_depth, depth2xyzmap_batch(zfar = inf), `iterations` refiner passes on ONE pose, pose read-back.
 * pose_in_dev: DEVICE [16] ob_in_cam of the centred mesh (pose_last), or NULL = continue from the pose this context's
 * previous fp_track produced.  pose_out_dev (DEVICE [16]) / pose_out_host (HOST [16]) are optional.  Synchronises. */
int fp_track(fp_ctx* ctx, const unsigned char* rgb_host, const float* depth_host, const float* K, int H, int W,
             const float* pose_in_dev, int iterations, float* pose_out_dev, float* pose_out_host, void* stream);

/* ------------------------------------------------------------------------------------------ */
/* one process, several GPUs (the reference's process model: run_demo.py is a single script)  */
/* ------------------------------------------------------------------------------------------ */
typedef struct fp_group fp_group;
/* One fp_ctx per device (dev_ids = NULL: devices 0..ndev-1), each with its own stream; devices 1.. get peer access to
 * device 0, where the gathered features live.  Call from one thread. */
int fp_group_create(int ndev, const int* dev_ids, fp_group** out);
int fp_group_destroy(fp_group* g);
int fp_group_size(fp_group* g);
fp_ctx* fp_group_ctx(fp_group* g, int i); /* for per-device calls of the single-context API */
/* fp_load_network / fp_set_config / fp_set_mesh on every context of the group */
int fp_group_load_network(fp_group* g, int which, const fp_tensor_t* tensors, int n);
int fp_group_set_config(fp_group* g, int which, float crop_ratio, float rot_normalizer);
int fp_group_set_mesh(fp_group* g, int V, int F, const float* pos, const float* nrm, const float* uv, const float* vcol,
                      const int* faces, const unsigned char* tex_rgb, int Ht, int Wt, float diameter);
/* FoundationPose.register (estimater.py:159-240) with the N hypotheses sharded contiguously over the group's devices
 * (BASELINE.json configs[3]): HOST frame, mask (uint8 [H][W]) and rotation grid [N][16]; every device filters the frame,
 * derives the start poses and refines / featurises its slice, writing its feature rows and refined poses straight into
 * device 0's buffers over NVLink peer memory; device 0 runs the cross-hypothesis tail once.  Outputs (HOST): refined
 * poses [N][16], scores [N], best index, optional info[4] = {tx, ty, tz, n_valid} of guess_translation.  Synchronises. */
int fp_group_register(fp_group* g, const unsigned char* rgb_host, const float* depth_host, const float* K, int H, int W,
                      const unsigned char* mask_host, const float* rot_grid_host, int N, int iterations,
                      float* poses_out_host, float* scores_out_host, int* best_out_host, float* info_out_host);

/* parity-test hooks on pre-built crops (fp16 [2N][166][2][84][8], device) */
int fp_op_refine_net(fp_ctx* ctx, const void* crops, int N, float* trans_out, float* rot_out, void* stream);
int fp_op_score_feats(fp_ctx* ctx, const void* crops, int N, float* feats_out, void* stream);
int fp_op_tokens(fp_ctx* ctx, int which, const void* crops, int N, void* tokens_out, void* stream);
/* Host-only hook (no GPU needed) on the mesh preparation fp_set_mesh performs: meshlets of <= 64 triangles / <= 64
 * vertices + closedness / orientation analysis.  info[6] = {meshlets, closed (0/1), front-face winding sign (0 = none),
 * max triangles per meshlet, max vertices per meshlet, total triangles}; face_of_tri_out (optional, [F]) receives the
 * original face id of every meshlet triangle.  Verifies internally that every meshlet triangle maps back to its face. */
int fp_op_build_meshlets(int V, int F, const float* pos, const int* faces, int* info, int* face_of_tri_out,
                         float* meshlets_out /* optional [ceil(F/1)][8]: sphere xyz r, cone axis xyz cutoff */);
/* which: 0 = erode_depth (Utils.py:359-395), 1 = bilateral_filter_depth (Utils.py:304-356) */
int fp_op_depth_filter(const float* depth_dev, float* out_dev, int H, int W, int which, void* stream);
/* egocentric_delta_pose_to_pose with the refiner's output decoding (predict_pose_refine.py:195-231) */
int fp_op_pose_update(const float* poses_in, const float* trans, const float* rot, float* poses_out, int N,
                      float mesh_diameter, float rot_normalizer, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FPOSE_H_ */
