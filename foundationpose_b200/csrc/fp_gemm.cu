// fp_gemm.cu — tcgen05 / TMA implicit-GEMM tile kernel for every dense contraction on the hot
// path: the 15 convolutions of RefineNet / ScoreNetMultiPair's encoders and the linear layers of
// their attention heads.
//
// Replaces (reference, via torch -> cuDNN / cuBLAS under fp16 autocast):
//   learning/models/network_modules.py:37-50   ConvBNReLU          (conv + folded BN + ReLU)
//   learning/models/network_modules.py:73-111  ResnetBasicBlock    (conv,BN,ReLU,conv,BN,+id,ReLU)
//   learning/models/refine_network.py:80-92    encodeA / encodeAB / pos_embed / linear layers
//   learning/models/score_network.py:60-74     encoderA / encoderAB / att projections
//
// Design (B200-first, no library GEMM):
//   * D[128 x BN] tiles, fp16 operands, fp32 accumulators in TMEM (double buffered, 2 x BN columns).
//   * Warp-specialised persistent CTA (one per SM, or a CTA pair issuing cta_group::2 MMAs): warp 0 = TMA
//     producer, warp 1 = single-thread tcgen05.mma issuer, warps 2..9 = epilogue (TMEM -> registers ->
//     +bias/+residual/ReLU/+PE -> fp16 -> swizzled smem slab -> TMA tensor store).  smem ring of STAGES x
//     (A 16 KB + B BN*128 B), 128-byte swizzle.
//   * The convolution is an *implicit* GEMM: the A tile for k-block (tap, 64-channel chunk) is one
//     5-D TMA box over the NHWC activation tensor, displaced by the tap offset; out-of-bounds
//     coordinates are zero-filled by the TMA unit, which implements the zero padding.  Stride-2
//     convolutions use a (2C, W/2, 2, H/2, N) view of the same memory so that every tap is again a
//     dense box; the 7x7/s2 stem has its own kernel (fp_stem.cu).  No im2col buffer is ever
//     materialised.
//   * What bounds these main loops on B200 is the SM's 128 B/cycle shared-memory port (TMA fills + MMA
//     operand reads + epilogue staging), hence: CTA pairs (half of B per CTA), the swapped kernel for the
//     128-channel layers, and the PATCH mode, in which the nine taps of a 3x3 convolution are nine shifted
//     descriptors into ONE input patch per 64-channel chunk (see GemmParams).
#include "fp_gemm.cuh"

#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <vector>

#include "fp_common.cuh"

namespace fp {

static std::atomic<unsigned long long> g_launch_count{0};
static thread_local bool t_capturing = false;
void note_launches(int n) {
  if (!t_capturing) g_launch_count.fetch_add((unsigned long long)n, std::memory_order_relaxed);
}
unsigned long long launch_count() { return g_launch_count.load(std::memory_order_relaxed); }
void set_capturing(bool on) { t_capturing = on; }

std::atomic<bool> g_prof_on{false};
static std::mutex g_prof_mu;

struct ProfRec {
  cudaEvent_t e0, e1;
  double work;
  int kind;
};
static std::vector<ProfRec> g_prof_recs;

void prof_mark_begin(int kind, double work, cudaStream_t stream) {
  if (!g_prof_on) return;
  ProfRec r;
  r.kind = kind;
  r.work = work;
  cudaEventCreate(&r.e0);
  cudaEventCreate(&r.e1);
  cudaEventRecord(r.e0, stream);
  std::lock_guard<std::mutex> lk(g_prof_mu);
  g_prof_recs.push_back(r);
}
void prof_mark_end(cudaStream_t stream) {
  if (!g_prof_on) return;
  std::lock_guard<std::mutex> lk(g_prof_mu);
  if (g_prof_recs.empty()) return;
  cudaEventRecord(g_prof_recs.back().e1, stream);
}
// sums and clears the records of `kind`; synchronises the device
int prof_collect(int kind, double* total_ms, double* total_work, int* launches) {
  FP_CUDA_OK(cudaDeviceSynchronize());
  std::lock_guard<std::mutex> lk(g_prof_mu);
  double ms = 0, work = 0;
  int n = 0;
  std::vector<ProfRec> keep;
  for (auto& r : g_prof_recs) {
    if (r.kind != kind) {
      keep.push_back(r);
      continue;
    }
    float t = 0.f;
    cudaEventElapsedTime(&t, r.e0, r.e1);
    ms += t;
    work += r.work;
    ++n;
    cudaEventDestroy(r.e0);
    cudaEventDestroy(r.e1);
  }
  g_prof_recs.swap(keep);
  *total_ms = ms;
  *total_work = work;
  *launches = n;
  return 0;
}

static thread_local char t_last_error[1024] = "";
void set_last_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(t_last_error, sizeof(t_last_error), fmt, ap);
  va_end(ap);
}
const char* get_last_error() { return t_last_error; }

static thread_local GemmPlan t_plan;
static thread_local bool t_plan_set = false;
void note_plan(const GemmPlan& plan) {
  t_plan = plan;
  t_plan_set = true;
}
bool last_plan(GemmPlan* plan) {
  if (t_plan_set) *plan = t_plan;
  return t_plan_set;
}

static thread_local int t_pdl_skip = 0;
void pdl_skip_next() { t_pdl_skip = 1; }

bool pdl_enabled() {
  if (t_pdl_skip) {  // consumed by exactly one launch_pdl
    t_pdl_skip = 0;
    return false;
  }
  static int on = -1;
  if (on < 0) {
    const char* e = getenv("FPOSE_PDL");
    on = (e && e[0] == '0') ? 0 : 1;
  }
  return on != 0;
}

struct GemmParams {
  int lg_bw, lg_bh;  // tile rows m -> (nn, ii, jj): jj = m & (bw-1), ii = (m >> lg_bw) & (bh-1)
  int bw, bh, bn;
  int tiles_w, tiles_h, tiles_n, n_tiles_n, total_tiles;
  int num_kb, chunks_per_tap;
  int dim_w, dim_h, dim_n;
  short tap_off[9][5];
  int Ho, Wo, n_img, Cout;
  const float* bias;
  int has_res;
  int odim_h, odim_n;  // which coordinate of the output / residual maps receives the tile's row / image
  int out_split;
  const float* post_add;
  int relu;
  double alg_flops;  // 2 * M * Cout * K_real of this launch (host-side bookkeeping only)
  // ---- patch mode (3x3 stride-1 convolutions): the A operand of every tap is a shifted VIEW of one shared-memory
  // segment (a halo'd patch of the input tile, 128B-swizzled rows of 64 channels), fetched once per 64-channel
  // chunk instead of once per tap.  tools/umma_probe.cu shows that tcgen05 applies the 128B swizzle to absolute
  // shared-memory address bits, so a descriptor may start at any 128-byte row and use any group stride.
  int seg_count, taps_per_seg;  // segments per channel chunk (1: halo'd patch, 3: one column-shifted copy per s)
  int seg_bytes;                // bytes of one segment's TMA box
  short seg_off[3][5];          // coordinate offsets of segment q relative to the tile origin
  int tap_aoff[9];              // [q * taps_per_seg + t]: byte offset of the tap's first row inside the segment
  short tap_w[9];               // [q * taps_per_seg + t]: filter tap (r * 3 + s) -> which weight k-block
  int a_sbo;                    // bytes between consecutive 8-row groups of the A operand
  int odim_w;                   // coordinate of the output map that receives the tile's column
  int row_mode;                 // tile row -> pixel: 0 = (n, i, j), 1 = (i, n, j), 2 = (i, j, n)   [fastest last]
  int trace_idx;                // -DFP_GEMM_TRACE builds only: slot of this launch in g_gemm_trace
};

// -DFP_GEMM_TRACE (tools/gemm_trace.py): CTA 0 of every gemm_tile_kernel launch stamps its phases with the SM clock
// (slots 0-7) and the global timer (8: entry, 9: exit) so that the fixed cost of a launch at one pose can be read
// phase by phase.  Compiles to nothing in the product build.
#ifdef FP_GEMM_TRACE
__device__ unsigned long long g_gemm_trace[512][10];
__device__ __forceinline__ unsigned long long trace_gtime() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
#define FP_TRACE(slot)                                                              \
  do {                                                                              \
    if (blockIdx.x == 0) g_gemm_trace[p.trace_idx & 511][slot] = (unsigned long long)clock64(); \
  } while (0)
#define FP_TRACE_G(slot)                                                  \
  do {                                                                    \
    if (blockIdx.x == 0) g_gemm_trace[p.trace_idx & 511][slot] = trace_gtime(); \
  } while (0)
#else
#define FP_TRACE(slot)
#define FP_TRACE_G(slot)
#endif

constexpr int kBlockM = 128;
constexpr int kBlockK = 64;
constexpr int kABytes = kBlockM * kBlockK * 2;  // 16 KB
constexpr int kTileThreads = 320;   // tile kernel: producer, MMA, 8 epilogue warps (two per TMEM lane quarter)
constexpr int kSlabBytes = kBlockM * 64 * 2;  // 16 KB: one output slab (128 pixels x 64 channels, 128B-swizzled)

// CG = CTAs per MMA (tcgen05 cta_group): with CG = 2 the CTA pair of a cluster issues one M = 256 MMA; each CTA
// stages its own 128 pixel rows of A and only HALF of the weight tile (BN/2 rows), which halves the B-operand
// shared-memory traffic per SM — the bound of the N <= 128 layers.
// SLABS = epilogue staging slabs (16 KB each).  2: slabs are recycled one by one.  4 (residual layers with
// BN = 256): one slab per 64-channel slice of the tile, so the whole tile's residual is prefetched by TMA
// while the tile's MMAs are still running.
constexpr int kPatchSlot = 26 * 1024;  // one A segment: 10 x 10 x 2 (25,600 B) or 6 x 4 x 8 (24,576 B) rows of 128 B
constexpr int kPatchStages = 3;
constexpr int kSmemBudget = 232448 - 1024 - 256;  // opt-in maximum minus alignment slack and the barrier block

template <int BN, int CG, int SLABS, bool PATCH = false>
struct TileCfg {
  static constexpr int kBBytes = (BN / CG) * kBlockK * 2;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kNumSlabs = (SLABS == 2) ? 2 : 4;  // SLABS = 8: ring of 4 slabs (4 TMA stores in flight)
  static constexpr int kStagingBytes = kNumSlabs * kSlabBytes;
  static constexpr int kRing = 196608 + 2 * kSlabBytes - kStagingBytes;
  static constexpr int kStages = (kRing / kStageBytes) > 8 ? 8 : (kRing / kStageBytes);
  // patch mode: kPatchStages A segments + a ring of weight tiles
  static constexpr int kBRing = kSmemBudget - kPatchStages * kPatchSlot - kStagingBytes;
  static constexpr int kBStages = (kBRing / kBBytes) > 8 ? 8 : (kBRing / kBBytes);
  static constexpr int kOperandBytes = PATCH ? (kPatchStages * kPatchSlot + kBStages * kBBytes) : (kStages * kStageBytes);
  static constexpr int kTmemCols = (2 * BN <= 128) ? 128 : (2 * BN <= 256 ? 256 : 512);
  static constexpr int kSmemBytes = kOperandBytes + kStagingBytes + 1024 /*align slack*/ + 256 /*barriers*/ + 1024 /*bias tile*/;
  static_assert(kSmemBytes <= 232448, "tile configuration exceeds the 227 KB opt-in shared memory");
};

template <int BN, int CG, int SLABS, bool PATCH = false>
__global__ void __launch_bounds__(kTileThreads, 1)
    gemm_tile_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                     const __grid_constant__ CUtensorMap map_out, const __grid_constant__ CUtensorMap map_res,
                     const __grid_constant__ GemmParams p) {
  using Cfg = TileCfg<BN, CG, SLABS, PATCH>;
  constexpr int S = PATCH ? Cfg::kBStages : Cfg::kStages;  // ring of (A+B) stages, or of weight tiles in patch mode
  constexpr int SA = kPatchStages;
  constexpr int NS = Cfg::kNumSlabs;
  constexpr bool PREFETCH = (SLABS == 4);  // whole-tile residual prefetch, one slab per 64-channel slice
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* b_ring = smem + SA * kPatchSlot;        // patch mode: [SA][kPatchSlot] segments, then [S][kBBytes] weights
  uint8_t* staging = smem + Cfg::kOperandBytes;    // [NS][kSlabBytes], 1024-aligned
  uint64_t* bars = reinterpret_cast<uint64_t*>(staging + Cfg::kStagingBytes);
  uint64_t* full = bars;                 // [S]
  uint64_t* empty = bars + S;            // [S]
  uint64_t* tmem_full = bars + 2 * S;    // [2]
  uint64_t* tmem_empty = bars + 2 * S + 2;  // [2]
  uint64_t* res_full = bars + 2 * S + 4;    // [4]
  uint64_t* a_full = bars + 2 * S + 8;      // [SA]  (patch mode)
  uint64_t* a_empty = bars + 2 * S + 8 + SA;  // [SA]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * S + 8 + 2 * SA);
  float* bias_s = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(bars) + 256);  // [BN]: this tile's bias

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int cta_rank = (CG == 2) ? (int)cluster_ctarank() : 0;
  // virtual tiles: (pair of M tiles, N tile) for CG = 2; this CTA owns M tile  vt_m * CG + cta_rank
  const int m_tiles = p.tiles_w * p.tiles_h * p.tiles_n;
  const int total_vt = ((m_tiles + CG - 1) / CG) * p.n_tiles_n;
  const int vt0 = blockIdx.x / CG, vt_step = gridDim.x / CG;

  if (warp == 0 && lane == 0) {
    FP_TRACE(0);
    FP_TRACE_G(8);
    tma_prefetch_desc(&map_a);
    tma_prefetch_desc(&map_b);
    for (int s = 0; s < S; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full[a], 1);
      mbar_init(&tmem_empty[a], 8 * CG);
    }
    for (int a = 0; a < 4; ++a) mbar_init(&res_full[a], 1);
    if (PATCH) {
      for (int a = 0; a < SA; ++a) {
        mbar_init(&a_full[a], 1);
        mbar_init(&a_empty[a], 1);
      }
    }
    tma_prefetch_desc(&map_out);
    if (p.has_res) tma_prefetch_desc(&map_res);
    mbar_fence_init();
  }
  if (CG == 2) cluster_sync_all();  // peer barriers initialised before any remote arrive / multicast commit
  if (warp == 1) {
    if (CG == 2) tmem_alloc_2sm(tmem_slot, Cfg::kTmemCols);
    else tmem_alloc(tmem_slot, Cfg::kTmemCols);
  }
  tc_fence_before();
  if (CG == 2) cluster_sync_all();
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (threadIdx.x == 0) FP_TRACE(1);
  pdl_trigger();
  pdl_wait();  // everything above overlapped the previous kernel's tail; activations are touched only from here on
  if (threadIdx.x == 0) FP_TRACE(2);

  // decode this CTA's tile of virtual tile vt; an odd leftover M tile is parked out of range (TMA zero-fills
  // its loads and clips its stores)
  auto decode = [&](int vt, int& n_tile, int& tw, int& th, int& tn) {
    n_tile = vt % p.n_tiles_n;
    const int m_tile = (vt / p.n_tiles_n) * CG + cta_rank;
    if (m_tile < m_tiles) {
      tw = m_tile % p.tiles_w;
      th = (m_tile / p.tiles_w) % p.tiles_h;
      tn = m_tile / (p.tiles_w * p.tiles_h);
    } else {
      tw = p.tiles_w;
      th = 0;
      tn = 0;
    }
  };

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (PATCH) {
      if (lane == 0) {
        int stage = 0, phase = 0, as = 0, aphase = 0;
        const int tps = p.taps_per_seg;
        for (int vt = vt0; vt < total_vt; vt += vt_step) {
          int n_tile, tw, th, tn;
          decode(vt, n_tile, tw, th, tn);
          int base[5] = {0, 0, 0, 0, 0};
          base[p.dim_w] += tw * p.bw;
          base[p.dim_h] += th * p.bh;
          base[p.dim_n] += tn * p.bn;
          for (int cs = 0; cs < p.chunks_per_tap; ++cs) {
            for (int q = 0; q < p.seg_count; ++q) {
              mbar_wait(&a_empty[as], aphase ^ 1);
              uint8_t* sa = smem + as * kPatchSlot;
              const int c0 = cs * kBlockK, c1 = base[1] + p.seg_off[q][1], c2 = base[2] + p.seg_off[q][2],
                        c3 = base[3] + p.seg_off[q][3], c4 = base[4] + p.seg_off[q][4];
              if (CG == 2) {
                if (cta_rank == 0) mbar_expect_tx(&a_full[as], 2 * p.seg_bytes);
                tma_load_5d_2sm(&map_a, &a_full[as], sa, c0, c1, c2, c3, c4);
              } else {
                mbar_expect_tx(&a_full[as], p.seg_bytes);
                tma_load_5d(&map_a, &a_full[as], sa, c0, c1, c2, c3, c4);
              }
              if (++as == SA) {
                as = 0;
                aphase ^= 1;
              }
              for (int t = 0; t < tps; ++t) {
                mbar_wait(&empty[stage], phase ^ 1);
                uint8_t* sb = b_ring + stage * Cfg::kBBytes;
                const int kcol = (p.tap_w[q * tps + t] * p.chunks_per_tap + cs) * kBlockK;
                if (CG == 2) {
                  if (cta_rank == 0) mbar_expect_tx(&full[stage], 2 * Cfg::kBBytes);
                  tma_load_2d_2sm(&map_b, &full[stage], sb, kcol, n_tile * BN + cta_rank * (BN / 2));
                } else {
                  mbar_expect_tx(&full[stage], Cfg::kBBytes);
                  tma_load_2d(&map_b, &full[stage], sb, kcol, n_tile * BN);
                }
                if (++stage == S) {
                  stage = 0;
                  phase ^= 1;
                }
              }
            }
          }
        }
      }
    } else if (lane == 0) {
      int stage = 0, phase = 0;
      for (int vt = vt0; vt < total_vt; vt += vt_step) {
        int n_tile, tw, th, tn;
        decode(vt, n_tile, tw, th, tn);
        int base[5] = {0, 0, 0, 0, 0};
        base[p.dim_w] += tw * p.bw;
        if (p.dim_h >= 0) base[p.dim_h] += th * p.bh;
        if (p.dim_n >= 0) base[p.dim_n] += tn * p.bn;
        int tap = 0, chunk = 0;
        for (int kb = 0; kb < p.num_kb; ++kb) {
          mbar_wait(&empty[stage], phase ^ 1);
          uint8_t* sa = smem + stage * Cfg::kStageBytes;
          uint8_t* sb = sa + kABytes;
          const int c0 = base[0] + p.tap_off[tap][0] + chunk * kBlockK, c1 = base[1] + p.tap_off[tap][1],
                    c2 = base[2] + p.tap_off[tap][2], c3 = base[3] + p.tap_off[tap][3], c4 = base[4] + p.tap_off[tap][4];
          if (CG == 2) {
            // both CTAs' bytes land on the leader's barrier; the leader alone arms it (for both)
            if (cta_rank == 0) mbar_expect_tx(&full[stage], 2 * Cfg::kStageBytes);
            tma_load_5d_2sm(&map_a, &full[stage], sa, c0, c1, c2, c3, c4);
            tma_load_2d_2sm(&map_b, &full[stage], sb, kb * kBlockK, n_tile * BN + cta_rank * (BN / 2));
          } else {
            mbar_expect_tx(&full[stage], Cfg::kStageBytes);
            tma_load_5d(&map_a, &full[stage], sa, c0, c1, c2, c3, c4);
            tma_load_2d(&map_b, &full[stage], sb, kb * kBlockK, n_tile * BN);
          }
          if (++chunk == p.chunks_per_tap) {
            chunk = 0;
            ++tap;
          }
          if (++stage == S) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    if (PATCH) {
      if (lane == 0 && cta_rank == 0) {
        constexpr uint32_t idesc = umma_idesc_f16(BN, 128u * CG);
        int stage = 0, phase = 0, as = 0, aphase = 0, it = 0;
        const int tps = p.taps_per_seg;
        for (int vt = vt0; vt < total_vt; vt += vt_step, ++it) {
          const int acc = it & 1;
          mbar_wait(&tmem_empty[acc], ((it >> 1) & 1) ^ 1);
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + acc * BN;
          uint32_t accum = 0;
          for (int cs = 0; cs < p.chunks_per_tap; ++cs) {
            for (int q = 0; q < p.seg_count; ++q) {
              mbar_wait(&a_full[as], aphase);
              const uint32_t seg = smem_u32(smem + as * kPatchSlot);
              for (int t = 0; t < tps; ++t) {
                mbar_wait(&full[stage], phase);
                tc_fence_after();
                if (it == 0 && cs == 0 && q == 0 && t == 0) FP_TRACE(3);
                // the tap's rows start tap_aoff bytes into the segment; 8-row groups are a_sbo bytes apart
                const uint64_t da = umma_desc_sw128_sbo(seg + (uint32_t)p.tap_aoff[q * tps + t], (uint32_t)p.a_sbo);
                const uint64_t db = umma_desc_sw128(smem_u32(b_ring + stage * Cfg::kBBytes));
#pragma unroll
                for (int k = 0; k < kBlockK / 16; ++k) {
                  if (CG == 2) umma_f16_2sm(d_tmem, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, accum);
                  else umma_f16(d_tmem, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, accum);
                  accum = 1;
                }
                if (CG == 2) umma_commit_2sm(&empty[stage]);
                else umma_commit(&empty[stage]);
                if (++stage == S) {
                  stage = 0;
                  phase ^= 1;
                }
              }
              if (CG == 2) umma_commit_2sm(&a_empty[as]);
              else umma_commit(&a_empty[as]);
              if (++as == SA) {
                as = 0;
                aphase ^= 1;
              }
            }
          }
          if (CG == 2) umma_commit_2sm(&tmem_full[acc]);
          else umma_commit(&tmem_full[acc]);
        }
        FP_TRACE(4);
      }
    } else if (lane == 0 && cta_rank == 0) {
      constexpr uint32_t idesc = umma_idesc_f16(BN, 128u * CG);
      int stage = 0, phase = 0;
      int it = 0;
      for (int vt = vt0; vt < total_vt; vt += vt_step, ++it) {
        const int acc = it & 1;
        const int acc_phase = (it >> 1) & 1;
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
        for (int kb = 0; kb < p.num_kb; ++kb) {
          mbar_wait(&full[stage], phase);
          tc_fence_after();
          if (it == 0 && kb == 0) FP_TRACE(3);
          const uint32_t sa = smem_u32(smem + stage * Cfg::kStageBytes);
          const uint32_t sb = sa + kABytes;
          const uint64_t da = umma_desc_sw128(sa);
          const uint64_t db = umma_desc_sw128(sb);
#pragma unroll
          for (int k = 0; k < kBlockK / 16; ++k) {
            // advance 16 fp16 = 32 B along K inside the 128 B swizzle atom: +2 in (addr >> 4) units
            if (CG == 2)
              umma_f16_2sm(d_tmem, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (kb > 0 || k > 0) ? 1u : 0u);
            else
              umma_f16(d_tmem, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (kb > 0 || k > 0) ? 1u : 0u);
          }
          // frees the smem slot (in both CTAs) when these MMAs retire
          if (CG == 2) umma_commit_2sm(&empty[stage]);
          else umma_commit(&empty[stage]);
          if (kb == p.num_kb - 1) {
            if (CG == 2) umma_commit_2sm(&tmem_full[acc]);
            else umma_commit(&tmem_full[acc]);
          }
          if (++stage == S) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
      FP_TRACE(4);
    }
  } else {
    // ------------------------------------------------------------------ epilogue (warps 2..9)
    // TMEM -> registers -> (+bias, +residual, ReLU, +pos.emb.) -> fp16 -> 128B-swizzled smem slab ->
    // one TMA tensor store per 128-pixel x 64-channel slab.  The residual slab arrives the same way
    // (TMA load into the slab buffer), so every global access of the epilogue is a bulk, fully
    // coalesced transfer; out-of-range rows are clipped (store) / zero-filled (load) by the TMA unit.
    const int quarter = warp & 3;       // TMEM lanes [32*quarter, +32) are the ones this warp may read
    const int grp = (warp - 2) >> 2;    // which 32-column half of every 64-channel slab this warp handles
    const int row = quarter * 32 + lane;
    int jj, ii;  // tile row -> pixel inside the tile (only the positional-embedding table needs it)
    if (p.row_mode == 1) {  // (i, n, j)
      jj = row & (p.bw - 1);
      ii = row / (p.bw * p.bn);
    } else if (p.row_mode == 2) {  // (i, j, n)
      jj = (row / p.bn) & (p.bw - 1);
      ii = row / (p.bn * p.bw);
    } else {  // (n, i, j)
      jj = row & (p.bw - 1);
      ii = (row >> p.lg_bw) & (p.bh - 1);
    }
    const bool leader = (warp == 2 && lane == 0);
    const uint32_t row_off = (uint32_t)row * 128u;
    const uint32_t sw = (uint32_t)(row & 7);
    int it = 0;
    uint32_t slab_ctr = 0;
    for (int vt = vt0; vt < total_vt; vt += vt_step, ++it) {
      const int acc = it & 1;
      const int acc_phase = (it >> 1) & 1;
      int n_tile, tw, th, tn;
      decode(vt, n_tile, tw, th, tn);
      const int i = th * p.bh + ii, j = min(tw * p.bw + jj, p.Wo - 1);  // j only indexes the pos.-emb. table
      const int n0 = tn * p.bn;
      int n_o0 = n0, coff = 0;
      if (p.out_split > 0) {
        n_o0 = n0 % p.out_split;
        coff = (n0 / p.out_split) * p.Cout;
      }
      // Everything the epilogue reads from global memory is fetched NOW, while the tile's MMAs still run: at one
      // tile per CTA (small batches) the epilogue is exposed and an L2 round trip per 64-channel slab was 2/3 of it
      // (tools/gemm_trace.py: 4.6 -> 1.x us per launch).  The bias goes to shared memory (every row uses the same
      // values; the previous tile's readers are behind that tile's last bar.sync), the positional embedding of the
      // first slab to registers.
      const float* pap = p.post_add ? p.post_add + (size_t)(i * p.Wo + j) * p.Cout + n_tile * BN + grp * 32 : nullptr;
      {
        const int et = (int)threadIdx.x - 64;
        if (et < BN) bias_s[et] = __ldg(p.bias + n_tile * BN + et);
      }
      float4 pe[8];
      if (pap) {
#pragma unroll
        for (int k = 0; k < 8; ++k) pe[k] = __ldg(reinterpret_cast<const float4*>(pap) + k);
      }
      // output / residual box coordinates (dim 0 = channel is added per slab)
      int oc[5] = {0, 0, 0, 0, 0}, rc[5] = {0, 0, 0, 0, 0};
      oc[p.odim_w] = rc[p.odim_w] = tw * p.bw;
      if (p.odim_h >= 0) oc[p.odim_h] = rc[p.odim_h] = th * p.bh;
      if (p.odim_n >= 0) {
        oc[p.odim_n] = n_o0;
        rc[p.odim_n] = n0;
      }

      if (PREFETCH) {
        // one slab per 64-channel slice: fetch the whole tile's residual now, while its MMAs still run
        if (leader) {
          asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");  // last tile's stores have left the slabs
          if (p.has_res) {
            for (int sidx = 0; sidx < BN / 64; ++sidx) {
              mbar_expect_tx(&res_full[sidx], kSlabBytes);
              tma_load_5d(&map_res, &res_full[sidx], staging + sidx * kSlabBytes, n_tile * BN + sidx * 64, rc[1], rc[2], rc[3],
                          rc[4]);
            }
          }
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");
      }
      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
      if (leader && it == 0) FP_TRACE(5);
      const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * BN + grp * 32;
#pragma unroll 1
      for (int c = 0; c < BN; c += 64, ++slab_ctr) {
        const uint32_t buf = PREFETCH ? (uint32_t)(c >> 6) : (slab_ctr % (uint32_t)NS);
        uint8_t* slab = staging + buf * kSlabBytes;
        if (!PREFETCH) {
          // the TMA store that last used this buffer (NS slabs ago) must have finished reading it
          if (leader) {
            if (NS == 2) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
            else asm volatile("cp.async.bulk.wait_group.read 3;" ::: "memory");
          }
          asm volatile("bar.sync 1, 256;" ::: "memory");
          if (p.has_res && leader) {
            mbar_expect_tx(&res_full[buf], kSlabBytes);
            tma_load_5d(&map_res, &res_full[buf], slab, n_tile * BN + c, rc[1], rc[2], rc[3], rc[4]);
          }
        }
        float4 pe_next[8];
        if (pap && c + 64 < BN) {  // the next slab's positional embedding travels under this slab's work
#pragma unroll
          for (int k = 0; k < 8; ++k) pe_next[k] = __ldg(reinterpret_cast<const float4*>(pap + c + 64) + k);
        }
        uint32_t v[32];
        tmem_ld32(taddr + c, v);
        tmem_ld_wait();
        if (c + 64 >= BN) {
          // accumulator fully read: hand the TMEM stage back to the MMA warp before the stores
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {  // one arrival per warp (a remote arrive is a DSMEM transaction)
            if (CG == 2) mbar_arrive_cluster(&tmem_empty[acc], 0);
            else mbar_arrive(&tmem_empty[acc]);
          }
        }
        if (p.has_res) mbar_wait(&res_full[buf], PREFETCH ? (uint32_t)(it & 1) : ((slab_ctr / (uint32_t)NS) & 1u));
#pragma unroll
        for (int q4 = 0; q4 < 4; ++q4) {  // this warp's 4 chunks of 8 channels (16 B)
          const int q = grp * 4 + q4;
          uint4* cell = reinterpret_cast<uint4*>(slab + row_off + (((uint32_t)q ^ sw) << 4));
          float a[8];
          {
            const float4 b0 = *reinterpret_cast<const float4*>(bias_s + c + q * 8);
            const float4 b1 = *reinterpret_cast<const float4*>(bias_s + c + q * 8 + 4);
            const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int k = 0; k < 8; ++k) a[k] = __uint_as_float(v[q4 * 8 + k]) + bb[k];
          }
          if (p.has_res) {
            const uint4 r = *cell;
            const __half2* rh = reinterpret_cast<const __half2*>(&r);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const float2 rf = __half22float2(rh[k]);
              a[2 * k] += rf.x;
              a[2 * k + 1] += rf.y;
            }
          }
          if (p.relu) {
#pragma unroll
            for (int k = 0; k < 8; ++k) a[k] = fmaxf(a[k], 0.f);
          }
          if (pap) {
            const float4 p0 = pe[2 * q4], p1 = pe[2 * q4 + 1];
            a[0] += p0.x; a[1] += p0.y; a[2] += p0.z; a[3] += p0.w;
            a[4] += p1.x; a[5] += p1.y; a[6] += p1.z; a[7] += p1.w;
          }
          *cell = make_uint4(pack_half2(a[0], a[1]), pack_half2(a[2], a[3]), pack_half2(a[4], a[5]), pack_half2(a[6], a[7]));
        }
        if (pap && c + 64 < BN) {
#pragma unroll
          for (int k = 0; k < 8; ++k) pe[k] = pe_next[k];
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> async proxy
        asm volatile("bar.sync 1, 256;" ::: "memory");
        if (leader) {
          tma_store_5d(&map_out, slab, coff + n_tile * BN + c, oc[1], oc[2], oc[3], oc[4]);
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
      }
    }
    if (leader) {
      FP_TRACE(6);
      asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");  // smem must outlive the stores
      FP_TRACE(7);
    }
  }

  tc_fence_before();
  if (CG == 2) cluster_sync_all();
  else __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    if (CG == 2) tmem_dealloc_2sm(tmem_base, Cfg::kTmemCols);
    else tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
  if (threadIdx.x == 0) FP_TRACE_G(9);
}

// ------------------------------------------------------------------------------------------------
// "swap-AB" variant for the 128-output-channel convolutions.
//
// With D[128 pixels x 128 channels] tiles the MMA (128x128x16, 64 cycles) reads 8 KB of operands from shared
// memory while TMA writes the next 32 KB stage: 128 + 128 B/cycle against a 128 B/cycle port — measured 45 %
// tensor-pipe utilisation.  Here the roles are exchanged: the weight tile [128 channels][64 k] is the M side
// and TWO pixel tiles (256 pixels) are the N side, so one 128x256x16 MMA (128 cycles) reads 12 KB and the stage
// is 48 KB per 512 cycles — the same 96 + 96 B/cycle budget as the 256-channel layers.  The accumulator is then
// [channel (TMEM lane)][pixel (TMEM column)]: the epilogue thread owns one channel (bias is a register) and
// scatters fp16 values into the 128B-swizzled [pixel][channel] slabs that the TMA store (and the TMA residual
// load) use; a warp's 32 lanes write 64 contiguous bytes, so the transposition is bank-conflict free.
// ------------------------------------------------------------------------------------------------
constexpr int kSwapStages = 3;
constexpr int kSwapStageBytes = kABytes + 2 * kABytes;  // W 16 KB + X 2 x 16 KB
constexpr int kSwapStaging = 4 * kSlabBytes;            // 2 pixel tiles (one per epilogue warpgroup) x 2 channel halves
constexpr int kSwapSmem = kSwapStages * kSwapStageBytes + kSwapStaging + 1024 + 256;

__global__ void __launch_bounds__(kTileThreads, 1)
    gemm_swap_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_w,
                     const __grid_constant__ CUtensorMap map_out, const __grid_constant__ CUtensorMap map_res,
                     const __grid_constant__ GemmParams p) {
  constexpr int S = kSwapStages;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* staging = smem + S * kSwapStageBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(staging + kSwapStaging);
  uint64_t* full = bars;
  uint64_t* empty = bars + S;
  uint64_t* tmem_full = bars + 2 * S;
  uint64_t* tmem_empty = bars + 2 * S + 2;
  uint64_t* res_full = bars + 2 * S + 4;  // [2]: one per epilogue warpgroup
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * S + 6);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int m_tiles = p.tiles_w * p.tiles_h * p.tiles_n;
  const int c_tiles = p.Cout / 128;
  const int total_vt = ((m_tiles + 1) / 2) * c_tiles;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_a);
    tma_prefetch_desc(&map_w);
    tma_prefetch_desc(&map_out);
    if (p.has_res) tma_prefetch_desc(&map_res);
    for (int s = 0; s < S; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full[a], 1);
      mbar_init(&tmem_empty[a], 256);
      mbar_init(&res_full[a], 1);
    }
    mbar_fence_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_trigger();
  pdl_wait();

  auto decode_m = [&](int m_tile, int& tw, int& th, int& tn) {
    if (m_tile < m_tiles) {
      tw = m_tile % p.tiles_w;
      th = (m_tile / p.tiles_w) % p.tiles_h;
      tn = m_tile / (p.tiles_w * p.tiles_h);
    } else {
      tw = p.tiles_w;  // parked out of range: zero-filled loads, clipped stores
      th = 0;
      tn = 0;
    }
  };

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0, phase = 0;
      for (int vt = blockIdx.x; vt < total_vt; vt += gridDim.x) {
        const int c_tile = vt % c_tiles, pair = vt / c_tiles;
        int base[2][5];
        for (int t = 0; t < 2; ++t) {
          int tw, th, tn;
          decode_m(2 * pair + t, tw, th, tn);
          for (int d = 0; d < 5; ++d) base[t][d] = 0;
          base[t][p.dim_w] += tw * p.bw;
          if (p.dim_h >= 0) base[t][p.dim_h] += th * p.bh;
          if (p.dim_n >= 0) base[t][p.dim_n] += tn * p.bn;
        }
        int tap = 0, chunk = 0;
        for (int kb = 0; kb < p.num_kb; ++kb) {
          mbar_wait(&empty[stage], phase ^ 1);
          uint8_t* sw_ = smem + stage * kSwapStageBytes;
          mbar_expect_tx(&full[stage], kSwapStageBytes);
          tma_load_2d(&map_w, &full[stage], sw_, kb * kBlockK, c_tile * 128);
          for (int t = 0; t < 2; ++t)
            tma_load_5d(&map_a, &full[stage], sw_ + kABytes + t * kABytes, base[t][0] + p.tap_off[tap][0] + chunk * kBlockK,
                        base[t][1] + p.tap_off[tap][1], base[t][2] + p.tap_off[tap][2], base[t][3] + p.tap_off[tap][3],
                        base[t][4] + p.tap_off[tap][4]);
          if (++chunk == p.chunks_per_tap) {
            chunk = 0;
            ++tap;
          }
          if (++stage == S) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc_f16(256, 128);
      int stage = 0, phase = 0, it = 0;
      for (int vt = blockIdx.x; vt < total_vt; vt += gridDim.x, ++it) {
        const int acc = it & 1, acc_phase = (it >> 1) & 1;
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * 256;
        for (int kb = 0; kb < p.num_kb; ++kb) {
          mbar_wait(&full[stage], phase);
          tc_fence_after();
          const uint32_t sw_ = smem_u32(smem + stage * kSwapStageBytes);
          const uint64_t da = umma_desc_sw128(sw_);            // weights: M = 128 channels
          const uint64_t db = umma_desc_sw128(sw_ + kABytes);  // activations: N = 256 pixels
#pragma unroll
          for (int k = 0; k < kBlockK / 16; ++k)
            umma_f16(d_tmem, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (kb > 0 || k > 0) ? 1u : 0u);
          umma_commit(&empty[stage]);
          if (kb == p.num_kb - 1) umma_commit(&tmem_full[acc]);
          if (++stage == S) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else {
    // two independent epilogue warpgroups: group t (warps 2+4t .. 5+4t) owns pixel tile t of every virtual
    // tile (TMEM columns [128 t, 128 t + 128)), its own two staging slabs, named barrier, residual barrier and
    // TMA bulk groups
    const int quarter = warp & 3;
    const int t = (warp - 2) >> 2;
    const int half = quarter >> 1;                      // which 64-channel slab this warp's channels live in
    const int c_local = (quarter & 1) * 32 + lane;      // channel inside the slab
    const bool leader = (((warp - 2) & 3) == 0 && lane == 0);
    const uint32_t c_chunk = (uint32_t)(c_local >> 3), c_byte = (uint32_t)(c_local & 7) * 2u;
    uint8_t* my_staging = staging + t * 2 * kSlabBytes;
    uint8_t* slab = my_staging + half * kSlabBytes;
    int it = 0;
    for (int vt = blockIdx.x; vt < total_vt; vt += gridDim.x, ++it) {
      const int acc = it & 1, acc_phase = (it >> 1) & 1;
      const int c_tile = vt % c_tiles, pair = vt / c_tiles;
      const float bias = __ldg(p.bias + c_tile * 128 + quarter * 32 + lane);
      int oc[5] = {0, 0, 0, 0, 0}, rc[5] = {0, 0, 0, 0, 0}, coff = 0;
      {
        int tw, th, tn;
        decode_m(2 * pair + t, tw, th, tn);
        const int n0 = tn * p.bn;
        int n_o0 = n0;
        if (p.out_split > 0) {
          n_o0 = n0 % p.out_split;
          coff = (n0 / p.out_split) * p.Cout;
        }
        oc[1] = rc[1] = tw * p.bw;
        if (p.odim_h >= 0) oc[p.odim_h] = rc[p.odim_h] = th * p.bh;
        if (p.odim_n >= 0) {
          oc[p.odim_n] = n_o0;
          rc[p.odim_n] = n0;
        }
      }
      // this group's previous stores must have finished reading its two slabs
      if (leader) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
      if (t == 0) asm volatile("bar.sync 1, 128;" ::: "memory");
      else asm volatile("bar.sync 2, 128;" ::: "memory");
      if (p.has_res && leader) {
        mbar_expect_tx(&res_full[t], 2 * kSlabBytes);
        for (int hh = 0; hh < 2; ++hh)
          tma_load_5d(&map_res, &res_full[t], my_staging + hh * kSlabBytes, c_tile * 128 + hh * 64, rc[1], rc[2], rc[3], rc[4]);
      }
      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
      if (p.has_res) mbar_wait(&res_full[t], it & 1);
      const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * 256 + t * 128;
#pragma unroll 1
      for (int c = 0; c < 128; c += 32) {
        uint32_t v[32];
        tmem_ld32(taddr + c, v);
        tmem_ld_wait();
        if (c == 96) {
          tc_fence_before();
          mbar_arrive(&tmem_empty[acc]);
        }
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          const uint32_t px = (uint32_t)(c + i);
          __half* cell = reinterpret_cast<__half*>(slab + px * 128u + ((c_chunk ^ (px & 7u)) << 4) + c_byte);
          float a = __uint_as_float(v[i]) + bias;
          if (p.has_res) a += __half2float(*cell);
          if (p.relu) a = fmaxf(a, 0.f);
          *cell = __float2half_rn(a);
        }
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      if (t == 0) asm volatile("bar.sync 1, 128;" ::: "memory");
      else asm volatile("bar.sync 2, 128;" ::: "memory");
      if (leader) {
        for (int hh = 0; hh < 2; ++hh)
          tma_store_5d(&map_out, my_staging + hh * kSlabBytes, coff + c_tile * 128 + hh * 64, oc[1], oc[2], oc[3], oc[4]);
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      }
    }
    if (leader) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ------------------------------------------------------------------------------------------------
// Patch variant of the swapped kernel (3x3 stride-1, 128 output channels, 8 | H, W).  The N side is ONE tile of
// 4 images x 8 x 8 pixels whose input lives in shared memory as a halo'd patch [10 h][4 n][10 w] of 128-byte
// rows (64 channels, 128B swizzle), fetched once per 64-channel chunk; the B descriptor of filter tap (r, s)
// starts (r * 40 + s) rows into the patch and steps 10 rows per 8-pixel group.  Shared-memory fill per k-block
// drops from 48 KB (W + 2 pixel tiles) to 16 KB + 51.2 KB / 9 — the 128 B/cycle shared-memory port, not the
// tensor pipe, is what bounds these layers.
// ------------------------------------------------------------------------------------------------
constexpr int kSwapPatchBytes = 10 * 4 * 10 * 128;  // 51,200 B
constexpr int kSwapPatchStages = 2;
constexpr int kSwapWStages = 3;
constexpr int kSwapPatchSmem = kSwapPatchStages * kSwapPatchBytes + kSwapWStages * kABytes + kSwapStaging + 1024 + 256;

__global__ void __launch_bounds__(kTileThreads, 1)
    gemm_swap_patch_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_w,
                           const __grid_constant__ CUtensorMap map_out, const __grid_constant__ CUtensorMap map_res,
                           const __grid_constant__ GemmParams p) {
  constexpr int SX = kSwapPatchStages, SW = kSwapWStages;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* w_ring = smem + SX * kSwapPatchBytes;
  uint8_t* staging = w_ring + SW * kABytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(staging + kSwapStaging);
  uint64_t* x_full = bars;                  // [SX]
  uint64_t* x_empty = bars + SX;            // [SX]
  uint64_t* w_full = bars + 2 * SX;         // [SW]
  uint64_t* w_empty = bars + 2 * SX + SW;   // [SW]
  uint64_t* tmem_full = bars + 2 * SX + 2 * SW;
  uint64_t* tmem_empty = tmem_full + 2;
  uint64_t* res_full = tmem_full + 4;  // [2]: one per epilogue warpgroup
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 6);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int m_tiles = p.tiles_w * p.tiles_h * p.tiles_n;
  const int c_tiles = p.Cout / 128;
  const int total_vt = m_tiles * c_tiles;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_a);
    tma_prefetch_desc(&map_w);
    tma_prefetch_desc(&map_out);
    if (p.has_res) tma_prefetch_desc(&map_res);
    for (int s = 0; s < SX; ++s) {
      mbar_init(&x_full[s], 1);
      mbar_init(&x_empty[s], 1);
    }
    for (int s = 0; s < SW; ++s) {
      mbar_init(&w_full[s], 1);
      mbar_init(&w_empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full[a], 1);
      mbar_init(&tmem_empty[a], 256);
      mbar_init(&res_full[a], 1);
    }
    mbar_fence_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_trigger();
  pdl_wait();

  auto decode = [&](int vt, int& c_tile, int& tw, int& th, int& tn) {
    c_tile = vt % c_tiles;
    const int m_tile = vt / c_tiles;
    tw = m_tile % p.tiles_w;
    th = (m_tile / p.tiles_w) % p.tiles_h;
    tn = m_tile / (p.tiles_w * p.tiles_h);
  };

  if (warp == 0) {
    if (lane == 0) {
      int ws = 0, wph = 0, xs = 0, xph = 0;
      for (int vt = blockIdx.x; vt < total_vt; vt += gridDim.x) {
        int c_tile, tw, th, tn;
        decode(vt, c_tile, tw, th, tn);
        for (int cs = 0; cs < p.chunks_per_tap; ++cs) {
          mbar_wait(&x_empty[xs], xph ^ 1);
          mbar_expect_tx(&x_full[xs], kSwapPatchBytes);
          // box (64 ch, 10 w, 4 n, 10 h): halo rows / columns outside the image are zero-filled (= padding)
          tma_load_5d(&map_a, &x_full[xs], smem + xs * kSwapPatchBytes, cs * kBlockK, tw * 8 - 1, tn * 4, th * 8 - 1, 0);
          if (++xs == SX) {
            xs = 0;
            xph ^= 1;
          }
          for (int tap = 0; tap < 9; ++tap) {
            mbar_wait(&w_empty[ws], wph ^ 1);
            mbar_expect_tx(&w_full[ws], kABytes);
            tma_load_2d(&map_w, &w_full[ws], w_ring + ws * kABytes, (tap * p.chunks_per_tap + cs) * kBlockK, c_tile * 128);
            if (++ws == SW) {
              ws = 0;
              wph ^= 1;
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc_f16(256, 128);
      int ws = 0, wph = 0, xs = 0, xph = 0, it = 0;
      for (int vt = blockIdx.x; vt < total_vt; vt += gridDim.x, ++it) {
        const int acc = it & 1, acc_phase = (it >> 1) & 1;
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * 256;
        uint32_t accum = 0;
        for (int cs = 0; cs < p.chunks_per_tap; ++cs) {
          mbar_wait(&x_full[xs], xph);
          const uint32_t patch = smem_u32(smem + xs * kSwapPatchBytes);
          for (int tap = 0; tap < 9; ++tap) {
            mbar_wait(&w_full[ws], wph);
            tc_fence_after();
            const int r = tap / 3, sft = tap - 3 * r;
            const uint64_t da = umma_desc_sw128(smem_u32(w_ring + ws * kABytes));                     // M = 128 channels
            const uint64_t db = umma_desc_sw128_sbo(patch + (uint32_t)((r * 40 + sft) * 128), 1280u);  // N = 256 pixels
#pragma unroll
            for (int k = 0; k < kBlockK / 16; ++k) {
              umma_f16(d_tmem, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, accum);
              accum = 1;
            }
            umma_commit(&w_empty[ws]);
            if (++ws == SW) {
              ws = 0;
              wph ^= 1;
            }
          }
          umma_commit(&x_empty[xs]);
          if (++xs == SX) {
            xs = 0;
            xph ^= 1;
          }
        }
        umma_commit(&tmem_full[acc]);
      }
    }
  } else {
    // two independent epilogue warpgroups: group t owns pixel columns [128 t, 128 t + 128) of the accumulator =
    // rows [4 t, 4 t + 4) of the 8 x 8 tile for all 4 images, i.e. one (64 ch, 8 w, 4 n, 4 h) box per channel half
    const int quarter = warp & 3;
    const int t = (warp - 2) >> 2;
    const int half = quarter >> 1;
    const int c_local = (quarter & 1) * 32 + lane;
    const bool leader = (((warp - 2) & 3) == 0 && lane == 0);
    const uint32_t c_chunk = (uint32_t)(c_local >> 3), c_byte = (uint32_t)(c_local & 7) * 2u;
    uint8_t* my_staging = staging + t * 2 * kSlabBytes;
    uint8_t* slab = my_staging + half * kSlabBytes;
    int it = 0;
    for (int vt = blockIdx.x; vt < total_vt; vt += gridDim.x, ++it) {
      const int acc = it & 1, acc_phase = (it >> 1) & 1;
      int c_tile, tw, th, tn;
      decode(vt, c_tile, tw, th, tn);
      const float bias = __ldg(p.bias + c_tile * 128 + quarter * 32 + lane);
      const int n0 = tn * 4;
      int n_o0 = n0, coff = 0;
      if (p.out_split > 0) {
        n_o0 = n0 % p.out_split;
        coff = (n0 / p.out_split) * p.Cout;
      }
      const int ow = tw * 8, oh = th * 8 + 4 * t;  // map dims: (c, w, n, h)
      if (leader) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
      if (t == 0) asm volatile("bar.sync 1, 128;" ::: "memory");
      else asm volatile("bar.sync 2, 128;" ::: "memory");
      if (p.has_res && leader) {
        mbar_expect_tx(&res_full[t], 2 * kSlabBytes);
        for (int hh = 0; hh < 2; ++hh)
          tma_load_5d(&map_res, &res_full[t], my_staging + hh * kSlabBytes, c_tile * 128 + hh * 64, ow, n0, oh, 0);
      }
      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
      if (p.has_res) mbar_wait(&res_full[t], it & 1);
      const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * 256 + t * 128;
#pragma unroll 1
      for (int c = 0; c < 128; c += 32) {
        uint32_t v[32];
        tmem_ld32(taddr + c, v);
        tmem_ld_wait();
        if (c == 96) {
          tc_fence_before();
          mbar_arrive(&tmem_empty[acc]);
        }
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          const uint32_t px = (uint32_t)(c + i);
          __half* cell = reinterpret_cast<__half*>(slab + px * 128u + ((c_chunk ^ (px & 7u)) << 4) + c_byte);
          float a = __uint_as_float(v[i]) + bias;
          if (p.has_res) a += __half2float(*cell);
          if (p.relu) a = fmaxf(a, 0.f);
          *cell = __float2half_rn(a);
        }
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      if (t == 0) asm volatile("bar.sync 1, 128;" ::: "memory");
      else asm volatile("bar.sync 2, 128;" ::: "memory");
      if (leader) {
        for (int hh = 0; hh < 2; ++hh)
          tma_store_5d(&map_out, my_staging + hh * kSlabBytes, coff + c_tile * 128 + hh * 64, ow, n_o0, oh, 0);
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      }
    }
    if (leader) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
static int g_num_sms = 0;

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

static int encode_map(CUtensorMap* map, const void* base, int rank, const uint64_t* dims,
                      const uint64_t* strides_bytes /*rank-1*/, const uint32_t* box, bool swizzle128 = true) {
  EncodeTiledFn fn = get_encode_fn();
  FP_REQUIRE(fn != nullptr, "cuTensorMapEncodeTiled entry point not available (no CUDA driver?)");
  cuuint64_t gdim[5];
  cuuint64_t gstr[4];
  cuuint32_t bdim[5];
  cuuint32_t estr[5];
  for (int i = 0; i < rank; ++i) {
    gdim[i] = dims[i];
    bdim[i] = box[i];
    estr[i] = 1;
  }
  for (int i = 0; i < rank - 1; ++i) gstr[i] = strides_bytes[i];
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, (cuuint32_t)rank, const_cast<void*>(base), gdim, gstr,
                  bdim, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  FP_REQUIRE(r == CUDA_SUCCESS,
             "cuTensorMapEncodeTiled failed (%d): rank %d dims [%llu %llu %llu %llu %llu] box [%u %u %u %u %u]",
             (int)r, rank, (unsigned long long)dims[0], (unsigned long long)(rank > 1 ? dims[1] : 0),
             (unsigned long long)(rank > 2 ? dims[2] : 0), (unsigned long long)(rank > 3 ? dims[3] : 0),
             (unsigned long long)(rank > 4 ? dims[4] : 0), box[0], rank > 1 ? box[1] : 0, rank > 2 ? box[2] : 0,
             rank > 3 ? box[3] : 0, rank > 4 ? box[4] : 0);
  return 0;
}

int encode_map_f16(CUtensorMap* map, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                   const uint32_t* box) {
  return encode_map(map, base, rank, dims, strides_bytes, box);
}
int encode_map_f16_linear(CUtensorMap* map, const void* base, int rank, const uint64_t* dims,
                          const uint64_t* strides_bytes, const uint32_t* box) {
  return encode_map(map, base, rank, dims, strides_bytes, box, false);
}
int num_sms() {
  if (g_num_sms == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 0;
    if (cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return 0;
  }
  return g_num_sms;
}

static int ilog2(int v) {
  int l = 0;
  while ((1 << l) < v) ++l;
  return l;
}

static int g_cta_group = -1;  // FPOSE_CTA_GROUP=1 falls back to single-CTA MMAs (A/B checks)

#ifdef FP_GEMM_TRACE
struct TraceInfo {
  int bn, cg, slabs, patch, grid, total_vt, num_kb, m_tiles, cout, has_res;
};
static TraceInfo g_trace_info[512];
static int g_trace_next = 0;
static int trace_note(int bn, int cg, int slabs, int patch, int grid, int total_vt, const GemmParams& p) {
  const int i = g_trace_next++ & 511;
  g_trace_info[i] = {bn, cg, slabs, patch, grid, total_vt, p.num_kb, p.tiles_w * p.tiles_h * p.tiles_n, p.Cout, p.has_res};
  return i;
}
}  // namespace fp
extern "C" int fp_op_gemm_trace_reset() {
  fp::g_trace_next = 0;
  return 0;
}
// out: [n][10] stamps, info: [n][10] ints; returns the number of launches noted since the reset
extern "C" int fp_op_gemm_trace_read(unsigned long long* out, int* info, int max_n) {
  const int n = fp::g_trace_next < max_n ? fp::g_trace_next : max_n;
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(out, fp::g_gemm_trace, (size_t)n * 10 * sizeof(unsigned long long));
  memcpy(info, fp::g_trace_info, (size_t)n * sizeof(fp::TraceInfo));
  return n;
}
namespace fp {
#endif

template <int BN, int CG, int SLABS, bool PATCH = false>
static int launch_bn(const CUtensorMap& ma, const CUtensorMap& mb, const CUtensorMap& mo, const CUtensorMap& mr,
                     const GemmParams& p, cudaStream_t stream) {
  using Cfg = TileCfg<BN, CG, SLABS, PATCH>;
  static std::atomic<unsigned long long> attr_mask{0};  // per device: the attribute is device state
  if (!device_bit_test(attr_mask)) {
    FP_CUDA_OK(cudaFuncSetAttribute(gemm_tile_kernel<BN, CG, SLABS, PATCH>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    Cfg::kSmemBytes));
    device_bit_set(attr_mask);
  }
  if (g_num_sms == 0) {
    int dev = 0;
    FP_CUDA_OK(cudaGetDevice(&dev));
    FP_CUDA_OK(cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev));
  }
  const int m_tiles = p.tiles_w * p.tiles_h * p.tiles_n;
  const int total_vt = ((m_tiles + CG - 1) / CG) * p.n_tiles_n;
  const int slots = g_num_sms / CG;
  const int grid = CG * (total_vt < slots ? total_vt : slots);
  note_plan({PK_TILE, BN, CG, SLABS, PATCH ? (p.seg_count == 3 ? 2 : 1) : 0, grid, total_vt * CG, p.bw, p.bh, p.bn, m_tiles,
             p.n_tiles_n});
  prof_mark_begin(0, p.alg_flops, stream);
#ifdef FP_GEMM_TRACE
  GemmParams pt = p;
  pt.trace_idx = trace_note(BN, CG, SLABS, PATCH ? 1 : 0, grid, total_vt, p);
  FP_CUDA_OK(launch_pdl(gemm_tile_kernel<BN, CG, SLABS, PATCH>, dim3(grid), dim3(kTileThreads), Cfg::kSmemBytes, stream, CG, ma, mb,
                        mo, mr, pt));
#else
  FP_CUDA_OK(launch_pdl(gemm_tile_kernel<BN, CG, SLABS, PATCH>, dim3(grid), dim3(kTileThreads), Cfg::kSmemBytes, stream, CG, ma, mb,
                        mo, mr, p));
#endif
  prof_mark_end(stream);
  note_launches(1);
  FP_CUDA_OK(cudaGetLastError());
  return 0;
}


static int launch_swap(const CUtensorMap& ma, const CUtensorMap& mw, const CUtensorMap& mo, const CUtensorMap& mr,
                       const GemmParams& p, cudaStream_t stream) {
  static std::atomic<unsigned long long> attr_mask{0};  // per device: the attribute is device state
  if (!device_bit_test(attr_mask)) {
    FP_CUDA_OK(cudaFuncSetAttribute(gemm_swap_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSwapSmem));
    device_bit_set(attr_mask);
  }
  if (g_num_sms == 0) {
    int dev = 0;
    FP_CUDA_OK(cudaGetDevice(&dev));
    FP_CUDA_OK(cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev));
  }
  const int m_tiles = p.tiles_w * p.tiles_h * p.tiles_n;
  const int total_vt = ((m_tiles + 1) / 2) * (p.Cout / 128);
  const int grid = total_vt < g_num_sms ? total_vt : g_num_sms;
  note_plan({PK_SWAP, 128, 1, 0, 0, grid, total_vt, p.bw, p.bh, p.bn, m_tiles, p.Cout / 128});
  prof_mark_begin(0, p.alg_flops, stream);
  FP_CUDA_OK(launch_pdl(gemm_swap_kernel, dim3(grid), dim3(kTileThreads), kSwapSmem, stream, 1, ma, mw, mo, mr, p));
  prof_mark_end(stream);
  note_launches(1);
  FP_CUDA_OK(cudaGetLastError());
  return 0;
}

static int launch_swap_patch(const CUtensorMap& ma, const CUtensorMap& mw, const CUtensorMap& mo, const CUtensorMap& mr,
                             const GemmParams& p, cudaStream_t stream) {
  static std::atomic<unsigned long long> attr_mask{0};  // per device: the attribute is device state
  if (!device_bit_test(attr_mask)) {
    FP_CUDA_OK(cudaFuncSetAttribute(gemm_swap_patch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSwapPatchSmem));
    device_bit_set(attr_mask);
  }
  const int sms = num_sms();
  FP_REQUIRE(sms > 0, "no CUDA device");
  const int m_tiles = p.tiles_w * p.tiles_h * p.tiles_n;
  const int total_vt = m_tiles * (p.Cout / 128);
  const int grid = total_vt < sms ? total_vt : sms;
  note_plan({PK_SWAP_PATCH, 128, 1, 0, 1, grid, total_vt, p.bw, p.bh, p.bn, m_tiles, p.Cout / 128});
  prof_mark_begin(0, p.alg_flops, stream);
  FP_CUDA_OK(launch_pdl(gemm_swap_patch_kernel, dim3(grid), dim3(kTileThreads), kSwapPatchSmem, stream, 1, ma, mw, mo, mr, p));
  prof_mark_end(stream);
  note_launches(1);
  FP_CUDA_OK(cudaGetLastError());
  return 0;
}

int stem_conv_launch(const GemmLayer& L, cudaStream_t stream);  // fp_stem.cu

static int g_swap_ab = -1;  // FPOSE_SWAP_AB=0 disables the swapped 128-channel kernels (A/B checks)
static int g_patch = -1;    // FPOSE_PATCH=0 falls back to one TMA box per filter tap (A/B checks)

int gemm_layer_launch(const GemmLayer& L, cudaStream_t stream) {
  if (L.kind == LK_CONV7_S2) return stem_conv_launch(L, stream);
  GemmParams p;
  memset(&p, 0, sizeof(p));
  p.odim_w = 1;
  bool patch = false, swap_patch = false;
  int out_bh = 0;  // rows of the output / residual box (0: the tile's bh)
  if (g_swap_ab < 0) {
    const char* e = getenv("FPOSE_SWAP_AB");
    g_swap_ab = (e && e[0] == '0') ? 0 : 1;
  }
  CUtensorMap ma, mb;
  const uint64_t E = 2;  // bytes per fp16
  int Ho, Wo, taps, ktot;
  int BN;
  uint64_t dims[5], str[4];
  uint32_t box[5];
  // Grids far below one wave (a single tracked pose, up to ~8 hypotheses): per-CTA time is the K loop at the MMA
  // rate of the tile (tools/gemm_trace.py: 274 ns per k-block for 256 x 256), so HALVING the tile width doubles the
  // CTAs and halves the layer's latency; the extra operand traffic is irrelevant with most SMs idle.  Decided per
  // convolution before its tiling, because the narrow tiles run on the plain (non-patch) kernel.
  static int g_narrow = -1;
  if (g_narrow < 0) {
    const char* e = getenv("FPOSE_NARROW");
    g_narrow = (e && e[0] == '0') ? 0 : 1;
  }
  bool narrow = false;
  auto is_narrow = [&](int ho, int wo, int bw, int bh, int bn) {
    if (!g_narrow || L.Cout % 256 != 0 || 9 * L.Cin / 64 < 16) return false;
    const int mt = (wo / bw) * (ho / bh) * ((L.n_img + bn - 1) / bn);
    return ((mt + 1) / 2) * (L.Cout / 256) * 4 <= num_sms();  // <= half of the CTA-pair slots
  };

  switch (L.kind) {
    case LK_LINEAR: {
      FP_REQUIRE(L.Cin % 64 == 0, "LINEAR: K=%d not a multiple of 64", L.Cin);
      Ho = 1;
      Wo = L.Win;
      taps = 1;
      p.chunks_per_tap = L.Cin / 64;
      p.bw = 128; p.bh = 1; p.bn = 1;
      p.dim_w = 1; p.dim_h = -1; p.dim_n = -1;
      dims[0] = L.Cin; dims[1] = L.Win; dims[2] = 1; dims[3] = 1; dims[4] = 1;
      str[0] = L.Cin * E; str[1] = str[0] * L.Win; str[2] = str[1]; str[3] = str[1];
      box[0] = 64; box[1] = 128; box[2] = 1; box[3] = 1; box[4] = 1;
      p.tiles_w = (L.Win + 127) / 128; p.tiles_h = 1; p.tiles_n = 1;
      break;
    }
    case LK_CONV3_S1: {
      FP_REQUIRE(L.Cin % 64 == 0, "CONV3_S1: Cin=%d not a multiple of 64", L.Cin);
      Ho = L.Hin; Wo = L.Win;
      taps = 9;
      p.chunks_per_tap = L.Cin / 64;
      if (Wo % 8 == 0 && Ho % 8 == 0) { p.bw = 8; p.bh = 8; p.bn = 2; }
      else if (Wo % 4 == 0 && Ho % 4 == 0) { p.bw = 4; p.bh = 4; p.bn = 8; }
      else FP_REQUIRE(false, "CONV3_S1: unsupported spatial size %dx%d", Ho, Wo);
      if (g_patch < 0) {
        const char* e = getenv("FPOSE_PATCH");
        g_patch = e ? atoi(e) : 1;
      }
      // measured (profiles/r01e_gemm_probe_patch.log): +6 % on the 40 x 40 / 256-channel layers; the 20 x 20 layers
      // (three column-shifted copies, FPOSE_PATCH=2) are 2 % slower than the per-tap boxes and stay on those
      narrow = is_narrow(Ho, Wo, p.bw, p.bh, p.bn);
      patch = !narrow && g_patch && L.Cout % 256 == 0 && (p.bw == 8 || g_patch == 2);
      swap_patch = g_patch && g_swap_ab && L.Cout == 128 && p.bw == 8 && !L.post_add && L.out_split % 4 == 0;
      const uint64_t sw_ = (uint64_t)L.Cin * E, sh_ = sw_ * L.Win, sn_ = sh_ * L.Hin;
      if (swap_patch) {
        // gemm_swap_patch_kernel: the N side is 4 images x 8 x 8 pixels out of one (64 ch, 10 w, 4 n, 10 h) patch
        p.bn = 4;
        p.dim_w = 1; p.dim_n = 2; p.dim_h = 3;
        dims[0] = L.Cin; dims[1] = L.Win; dims[2] = L.n_img; dims[3] = L.Hin; dims[4] = 1;
        str[0] = sw_; str[1] = sn_; str[2] = sh_; str[3] = sn_ * L.n_img;
        box[0] = 64; box[1] = 10; box[2] = 4; box[3] = 10; box[4] = 1;
        p.row_mode = 1;
        out_bh = 4;  // each epilogue warpgroup stores half of the tile's rows
      } else if (patch && p.bw == 8) {
        // one halo'd patch per 64-channel chunk: box (64 ch, 10 w, bn images, 10 h), rows ordered (h, n, w); tap
        // (r, s) starts (r * bn * 10 + s) rows into it and its 8-pixel row groups are 10 rows apart
        p.dim_w = 1; p.dim_n = 2; p.dim_h = 3;
        dims[0] = L.Cin; dims[1] = L.Win; dims[2] = L.n_img; dims[3] = L.Hin; dims[4] = 1;
        str[0] = sw_; str[1] = sn_; str[2] = sh_; str[3] = sn_ * L.n_img;
        box[0] = 64; box[1] = 10; box[2] = p.bn; box[3] = 10; box[4] = 1;
        p.seg_count = 1; p.taps_per_seg = 9;
        p.seg_bytes = 10 * p.bn * 10 * 128;
        p.seg_off[0][1] = -1; p.seg_off[0][3] = -1;
        for (int r = 0; r < 3; ++r)
          for (int s = 0; s < 3; ++s) {
            p.tap_aoff[r * 3 + s] = (r * p.bn * 10 + s) * 128;
            p.tap_w[r * 3 + s] = (short)(r * 3 + s);
          }
        p.a_sbo = 10 * 128;
        p.row_mode = 1;
      } else if (patch) {
        // 20 x 20 maps (tile = 4 x 4 pixels x 8 images): 8 consecutive rows are the 8 images of one pixel, so a
        // halo in w would break the constant group stride; instead one column-shifted copy per filter column s:
        // box (64 ch, 8 images, 4 w, 6 h), rows ordered (h, w, n); tap (r, s) = copy s, r * 32 rows in
        p.dim_n = 1; p.dim_w = 2; p.dim_h = 3;
        dims[0] = L.Cin; dims[1] = L.n_img; dims[2] = L.Win; dims[3] = L.Hin; dims[4] = 1;
        str[0] = sn_; str[1] = sw_; str[2] = sh_; str[3] = sn_ * L.n_img;
        box[0] = 64; box[1] = 8; box[2] = 4; box[3] = 6; box[4] = 1;
        p.seg_count = 3; p.taps_per_seg = 3;
        p.seg_bytes = 8 * 4 * 6 * 128;
        for (int sft = 0; sft < 3; ++sft) {
          p.seg_off[sft][2] = (short)(sft - 1);
          p.seg_off[sft][3] = -1;
          for (int r = 0; r < 3; ++r) {
            p.tap_aoff[sft * 3 + r] = r * 4 * 8 * 128;
            p.tap_w[sft * 3 + r] = (short)(r * 3 + sft);
          }
        }
        p.a_sbo = 1024;
        p.row_mode = 2;
      } else {
        p.dim_w = 1; p.dim_h = 2; p.dim_n = 3;
        dims[0] = L.Cin; dims[1] = L.Win; dims[2] = L.Hin; dims[3] = L.n_img; dims[4] = 1;
        str[0] = sw_; str[1] = sh_; str[2] = sn_; str[3] = sn_ * L.n_img;
        box[0] = 64; box[1] = p.bw; box[2] = p.bh; box[3] = p.bn; box[4] = 1;
        for (int r = 0; r < 3; ++r)
          for (int s = 0; s < 3; ++s) {
            p.tap_off[r * 3 + s][1] = (short)(s - 1);
            p.tap_off[r * 3 + s][2] = (short)(r - 1);
          }
      }
      p.tiles_w = Wo / p.bw; p.tiles_h = Ho / p.bh; p.tiles_n = (L.n_img + p.bn - 1) / p.bn;
      break;
    }
    case LK_CONV3_S2: {
      FP_REQUIRE(L.Cin % 64 == 0, "CONV3_S2: Cin=%d not a multiple of 64", L.Cin);
      FP_REQUIRE(L.Hin % 2 == 0 && L.Win % 2 == 0, "CONV3_S2: odd input size");
      Ho = L.Hin / 2; Wo = L.Win / 2;
      taps = 9;
      p.chunks_per_tap = L.Cin / 64;
      if (Wo % 8 == 0 && Ho % 8 == 0) { p.bw = 8; p.bh = 8; p.bn = 2; }
      else if (Wo % 4 == 0 && Ho % 4 == 0) { p.bw = 4; p.bh = 4; p.bn = 8; }
      else FP_REQUIRE(false, "CONV3_S2: unsupported output size %dx%d", Ho, Wo);
      narrow = is_narrow(Ho, Wo, p.bw, p.bh, p.bn);
      p.dim_w = 1; p.dim_h = 3; p.dim_n = 4;
      // view (N, H, W, C) as (N, H/2, 2, W/2, [2, C]): every (tap, chunk) is a dense box
      dims[0] = 2 * L.Cin; dims[1] = Wo; dims[2] = 2; dims[3] = Ho; dims[4] = L.n_img;
      str[0] = 2 * L.Cin * E; str[1] = (uint64_t)L.Win * L.Cin * E; str[2] = 2 * str[1];
      str[3] = (uint64_t)L.Hin * L.Win * L.Cin * E;
      box[0] = 64; box[1] = p.bw; box[2] = 1; box[3] = p.bh; box[4] = p.bn;
      for (int r = 0; r < 3; ++r)
        for (int s = 0; s < 3; ++s) {
          const int t = r * 3 + s;
          // input row 2i + r - 1: r=0 -> (i-1, phase 1), r=1 -> (i, 0), r=2 -> (i, 1)
          p.tap_off[t][0] = (short)((s == 1 ? 0 : 1) * L.Cin);
          p.tap_off[t][1] = (short)(s == 0 ? -1 : 0);
          p.tap_off[t][2] = (short)(r == 1 ? 0 : 1);
          p.tap_off[t][3] = (short)(r == 0 ? -1 : 0);
        }
      p.tiles_w = Wo / p.bw; p.tiles_h = Ho / p.bh; p.tiles_n = (L.n_img + p.bn - 1) / p.bn;
      break;
    }
    default:
      FP_REQUIRE(false, "unknown layer kind %d", L.kind);
  }
  ktot = taps * L.Cin;
  p.num_kb = ktot / 64;
  p.lg_bw = ilog2(p.bw);
  p.lg_bh = ilog2(p.bh);

  if (narrow) BN = 128;
  else if (L.Cout % 256 == 0) BN = 256;
  else if (L.Cout % 128 == 0) BN = 128;
  else if (L.Cout % 64 == 0) BN = 64;
  else FP_REQUIRE(false, "Cout=%d must be a multiple of 64", L.Cout);
  p.n_tiles_n = L.Cout / BN;
  p.total_tiles = p.tiles_w * p.tiles_h * p.tiles_n * p.n_tiles_n;
  p.Ho = Ho; p.Wo = Wo; p.n_img = L.n_img; p.Cout = L.Cout;
  p.bias = L.bias;
  p.has_res = L.res != nullptr;
  p.out_split = L.out_split;
  p.post_add = L.post_add;
  p.relu = L.relu;
  {
    const double k_real = (double)taps * L.Cin;
    p.alg_flops = 2.0 * (double)L.n_img * Ho * Wo * L.Cout * k_real;
  }
  FP_REQUIRE(L.out_ld % 8 == 0 && (!L.res || L.res_ld % 8 == 0), "out_ld / res_ld must be multiples of 8");
  FP_REQUIRE(L.out_split == 0 || L.out_split % p.bn == 0,
             "out_split=%d must be a multiple of the tile's image count %d (pad the A/B batch boundary)", L.out_split,
             p.bn);
  if (p.total_tiles == 0) return 0;

  int rc = encode_map(&ma, L.in, 5, dims, str, box);
  if (rc) return rc;
  uint64_t wd[2] = {(uint64_t)ktot, (uint64_t)L.Cout};
  uint64_t ws[1] = {(uint64_t)ktot * E};
  if (g_cta_group < 0) {
    const char* e = getenv("FPOSE_CTA_GROUP");
    g_cta_group = (e && e[0] == '1') ? 1 : 2;
  }
  // Measured on B200 (profiles/r01_gemm_probe_cta_pair.log): the CTA-pair MMA (cta_group::2, each CTA stages half
  // of the weight tile) is 8-10 % faster on the 256-wide, deep-K convolutions (up to 1.52 PFLOP/s) and slower on
  // the narrow / shallow-K layers, whose bound is the shared-memory port, not the TMA fill.
  const bool swap_ab = g_swap_ab && BN == 128 && L.Cout == 128 && !L.post_add &&
                       (L.kind == LK_CONV3_S1 || L.kind == LK_CONV3_S2);
  static int cg2_min_kb = -1;
  if (cg2_min_kb < 0) {
    const char* e = getenv("FPOSE_CG2_MIN_KB");
    cg2_min_kb = e ? atoi(e) : 16;
  }
  const int CG = (g_cta_group == 2 && (BN == 256 || narrow) && p.num_kb >= cg2_min_kb) ? 2 : 1;
  uint32_t wb[2] = {64, (uint32_t)(BN / CG)};
  rc = encode_map(&mb, L.w, 2, wd, ws, wb);
  if (rc) return rc;
  // output / residual maps: NHWC (conv) or [M][ld] (linear), one box = 128 pixels x 64 channels
  CUtensorMap mo, mr;
  {
    uint64_t od[5], os[4];
    uint32_t ob[5];
    const bool lin = (L.kind == LK_LINEAR);
    const int n_out = L.out_split > 0 ? (L.n_img - L.out_split) : L.n_img;
    FP_REQUIRE(n_out > 0, "out_split=%d leaves no output images (n_img=%d)", L.out_split, L.n_img);
    auto fill = [&](int ld, int nimg) {
      const uint64_t sw_ = (uint64_t)ld * E, sh_ = sw_ * Wo, sn_ = sh_ * Ho;
      od[0] = (uint64_t)ld;
      ob[0] = 64;
      od[4] = 1;
      ob[4] = 1;
      if (lin) {
        od[1] = (uint64_t)Wo; od[2] = 1; od[3] = 1;
        os[0] = sw_; os[1] = sh_; os[2] = sh_; os[3] = sh_;
        ob[1] = (uint32_t)p.bw; ob[2] = 1; ob[3] = 1;
      } else if (p.row_mode == 1) {  // tile rows ordered (h, n, w)
        od[1] = (uint64_t)Wo; od[2] = (uint64_t)nimg; od[3] = (uint64_t)Ho;
        os[0] = sw_; os[1] = sn_; os[2] = sh_; os[3] = sn_ * nimg;
        ob[1] = (uint32_t)p.bw; ob[2] = (uint32_t)p.bn; ob[3] = (uint32_t)(out_bh ? out_bh : p.bh);
      } else if (p.row_mode == 2) {  // tile rows ordered (h, w, n)
        od[1] = (uint64_t)nimg; od[2] = (uint64_t)Wo; od[3] = (uint64_t)Ho;
        os[0] = sn_; os[1] = sw_; os[2] = sh_; os[3] = sn_ * nimg;
        ob[1] = (uint32_t)p.bn; ob[2] = (uint32_t)p.bw; ob[3] = (uint32_t)p.bh;
      } else {  // (n, h, w)
        od[1] = (uint64_t)Wo; od[2] = (uint64_t)Ho; od[3] = (uint64_t)nimg;
        os[0] = sw_; os[1] = sh_; os[2] = sn_; os[3] = sn_ * nimg;
        ob[1] = (uint32_t)p.bw; ob[2] = (uint32_t)p.bh; ob[3] = (uint32_t)p.bn;
      }
    };
    p.odim_w = 1;
    p.odim_h = lin ? -1 : 2;
    p.odim_n = lin ? -1 : 3;
    if (p.row_mode == 1) { p.odim_n = 2; p.odim_h = 3; }
    if (p.row_mode == 2) { p.odim_n = 1; p.odim_w = 2; p.odim_h = 3; }
    fill(L.out_ld, n_out);
    rc = encode_map(&mo, L.out, 5, od, os, ob);
    if (rc) return rc;
    if (L.res) {
      fill(L.res_ld, L.n_img);
      rc = encode_map(&mr, L.res, 5, od, os, ob);
      if (rc) return rc;
    } else {
      mr = mo;
    }
  }

  if (swap_patch) return launch_swap_patch(ma, mb, mo, mr, p, stream);
  if (swap_ab) return launch_swap(ma, mb, mo, mr, p, stream);
  if (narrow) {
    if (CG == 2) return L.res ? launch_bn<128, 2, 4>(ma, mb, mo, mr, p, stream) : launch_bn<128, 2, 2>(ma, mb, mo, mr, p, stream);
    return launch_bn<128, 1, 2>(ma, mb, mo, mr, p, stream);
  }
  if (patch) {
    FP_REQUIRE(BN == 256, "patch mode is built for the 256-wide tile only");
    if (L.res) return CG == 2 ? launch_bn<256, 2, 4, true>(ma, mb, mo, mr, p, stream) : launch_bn<256, 1, 4, true>(ma, mb, mo, mr, p, stream);
    return CG == 2 ? launch_bn<256, 2, 2, true>(ma, mb, mo, mr, p, stream) : launch_bn<256, 1, 2, true>(ma, mb, mo, mr, p, stream);
  }
  if (BN == 256) {
    // residual layers: 4 staging slabs so the tile's residual is prefetched (one ring stage fewer)
    if (L.res) return CG == 2 ? launch_bn<256, 2, 4>(ma, mb, mo, mr, p, stream) : launch_bn<256, 1, 4>(ma, mb, mo, mr, p, stream);
    // K = 512 linears are bounded by their epilogue (8 k-blocks per tile): keep 4 output stores in flight
    if (CG == 1 && L.kind == LK_LINEAR) return launch_bn<256, 1, 8>(ma, mb, mo, mr, p, stream);
    return CG == 2 ? launch_bn<256, 2, 2>(ma, mb, mo, mr, p, stream) : launch_bn<256, 1, 2>(ma, mb, mo, mr, p, stream);
  }
  if (BN == 128) return launch_bn<128, 1, 2>(ma, mb, mo, mr, p, stream);
  return launch_bn<64, 1, 2>(ma, mb, mo, mr, p, stream);
}

}  // namespace fp
