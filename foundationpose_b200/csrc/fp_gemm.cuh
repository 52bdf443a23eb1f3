// fp_gemm.cuh — host-side description of one implicit-GEMM layer (conv / linear) for the
// tcgen05 tile kernel in fp_gemm.cu.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>

namespace fp {

enum LayerKind : int {
  LK_LINEAR = 0,    // out[m, :] = in[m, :] @ W^T            (in: [M, K] fp16 row-major)
  LK_CONV3_S1 = 1,  // 3x3 stride 1 pad 1                      (in: NHWC fp16)
  LK_CONV3_S2 = 2,  // 3x3 stride 2 pad 1                      (in: NHWC fp16, H, W even)
  LK_CONV7_S2 = 3,  // 7x7 stride 2 pad 3, Cin padded to 8     (in: [n][Hin+6][2][(Win+8)/2][8] fp16,
                    //   3-pixel zero border already in memory, even/odd column split: fp_stem.cu)
};

// Geometry + pointers of one layer launch.  All pointers are device pointers.
struct GemmLayer {
  int kind;
  int n_img;        // images (LINEAR: 1)
  int Hin, Win;     // input spatial size, un-padded (LINEAR: Hin = 1, Win = M)
  int Cin;          // input channels (LINEAR: K).  CONV7: 8 (6 real + 2 zero)
  int Cout;         // output channels; multiple of the N tile (64 / 128 / 256)
  const void* in;   // fp16 activations
  const void* w;    // fp16 packed weights [Cout][Ktot], Ktot = taps * Cin (CONV7: [7][4][2][64][8], fp_stem.cu)
  const float* bias;      // [Cout] fp32 (BN folded)
  const void* res;        // optional residual, fp16, indexed like the output with ld = res_ld
  int res_ld;
  void* out;              // fp16 output
  int out_ld;             // elements between consecutive output pixels (>= Cout)
  int out_split;          // if > 0: image n writes to image (n % out_split) at channel offset
                          //         (n / out_split) * Cout   (fuses torch.cat((a, b), 1))
  const float* post_add;  // optional fp32 table [Ho*Wo][Cout] added after the activation (pos. emb.)
  int relu;
};

// Enqueue one layer on `stream`.  Returns 0 or a negative error code (fp_last_error() has text).
int gemm_layer_launch(const GemmLayer& L, cudaStream_t stream);

// What a launch chose (fp_op_gemm_last_plan, include/fpose.h): kept per host thread, a few stores per launch.
enum PlanKernel : int { PK_TILE = 0, PK_SWAP = 1, PK_SWAP_PATCH = 2, PK_STEM = 3 };
struct GemmPlan {
  int kernel;        // PlanKernel
  int bn, cg, slabs; // output channels per tile, CTAs per MMA, epilogue staging slabs (tile kernel only, else 0)
  int patch;         // 0: one TMA box per tap, 1: one halo'd patch per channel chunk, 2: column-shifted copies
  int grid;          // CTAs launched
  int work_tiles;    // loop iterations summed over the grid: a CTA runs ceil(work_tiles / grid) of them
  int bw, bh, bimg;  // one M tile = bw x bh pixels of bimg images (LINEAR: bw = 128 rows)
  int m_tiles, n_tiles;  // M tiles of the launch, channel blocks of `bn` (swap kernels: 128) per M tile
};
void note_plan(const GemmPlan& plan);
bool last_plan(GemmPlan* plan);  // false before this thread's first launch


// Optional per-launch device timing (CUDA events on the launching stream) of the two kernels the
// roofline is reported for: kind 0 = gemm_tile_kernel (work = algorithmic FLOPs), kind 1 = crop_kernel
// (work = algorithmic output bytes).  Off by default; bench.py turns it on for a dedicated pass.
void prof_mark_begin(int kind, double work, cudaStream_t stream);
void prof_mark_end(cudaStream_t stream);
extern std::atomic<bool> g_prof_on;

}  // namespace fp
