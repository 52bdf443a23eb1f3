// fp_stem.cu — the 7x7 / stride-2 stem convolution (6 -> 64 channels, 160x160 -> 80x80) as a tcgen05
// implicit GEMM whose A operand is a *view* of one small shared-memory patch.
//
// Replaces (reference): learning/models/refine_network.py:34-35 and score_network.py:37-38, the first
// ConvBNReLU(C_in=6, C_out=64, kernel_size=7, stride=2) of encodeA / encoderA
// (network_modules.py:37-50), executed there by cuDNN under fp16 autocast.
//
// Why a dedicated kernel.  With 8 (6 + 2 zero) input channels the generic tile kernel (fp_gemm.cu) has to
// fetch, per output pixel and filter row, 8 input pixels = 128 B through a TMA box with overlapping
// strides: 7 x 16 KB per 128-pixel tile, 8.6x more bytes (and 128 B row requests) than the pixels the tile
// really touches.  Here the crop producer (fp_crop.cu) stores every padded image row as two half-rows,
// even columns then odd columns ("EO" layout: [n][166 rows][2][84 column pairs][8 ch] fp16), and the tile
// is 16 output rows x 8 output columns.  For filter row r and tap pair s (taps 2s, 2s+1) the K = 16 slice of
// A for output pixel (i, j) is  E[2i + r][j + s] ++ O[2i + r][j + s]  (16 B each), i.e. in shared memory
//     8 rows (j) at a 16 B pitch, 16 row groups (i) at a constant stride, two K chunks E / O at a constant offset
// which is exactly tcgen05's un-swizzled K-major canonical layout ((8,m),(8,2)) : ((16 B, SBO), (2 B, LBO)).
// So ONE 13 KB TMA box (37 rows x 2 x 11 pairs x 16 B) feeds all 7 x 4 = 28 MMAs (M = 128, N = 64, K = 16) of
// a tile through 28 descriptors that differ only in their start address; the 56 KB of packed weights stay
// resident in shared memory for the life of the (persistent) CTA.
//
// Roles per CTA (320 threads, one CTA per SM): warp 0 = TMA producer (patch ring), warp 1 = MMA issuer,
// warps 2..9 = two epilogue warpgroups, one per TMEM accumulator (TMEM -> +bias, ReLU -> fp16 -> 128B-swizzled
// slab -> TMA tensor store), fp32 accumulators double-buffered in TMEM (2 x 64 columns).
#include <stdlib.h>
#include <string.h>

#include "fp_common.cuh"
#include "fp_gemm.cuh"

namespace fp {

int encode_map_f16(CUtensorMap* map, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                   const uint32_t* box);
int encode_map_f16_linear(CUtensorMap* map, const void* base, int rank, const uint64_t* dims,
                          const uint64_t* strides_bytes, const uint32_t* box);
int num_sms();

namespace {

constexpr int kThreadsStem = 320;
constexpr int kTileH = 16, kTileW = 8;                   // output pixels per tile (M = 128)
constexpr int kPatchRows = 2 * (kTileH - 1) + 7;         // 37 padded input rows
constexpr int kPatchPairs = kTileW + 3;                  // 11 column pairs
constexpr int kParStride = kPatchPairs * 16;             // 176 B: E -> O half-row (LBO)
constexpr int kRowStride = 2 * kParStride;               // 352 B: padded input row
constexpr int kPatchBytes = kPatchRows * kRowStride;     // 13,024 B
constexpr int kPatchSlot = 13 * 1024;                    // ring slot (1024-aligned)
constexpr int kStagesStem = 6;
constexpr int kWTileBytes = 2 * 64 * 16;                 // one (r, s) weight tile: [E/O][64 ch][8 ci] fp16
constexpr int kWBytes = 28 * kWTileBytes;                // 57,344 B
constexpr int kSlab = 128 * 64 * 2;                      // 16 KB output slab
constexpr int kStemSmem = kWBytes + kStagesStem * kPatchSlot + 4 * kSlab + 1024 + 256;

struct StemParams {
  int tiles_w, tiles_h, n_img, total_tiles;
  const float* bias;
  int relu;
};

// un-swizzled K-major operand: 8 rows at 16 B, row groups `sbo` bytes apart, the two 8-element K chunks
// `lbo` bytes apart (cute::UMMA::make_umma_desc<Major::K>, LayoutType::INTERLEAVE)
__device__ __forceinline__ uint64_t umma_desc_linear(uint32_t smem_addr, uint32_t lbo, uint32_t sbo) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)(lbo >> 4) << 16;
  d |= (uint64_t)(sbo >> 4) << 32;
  d |= (uint64_t)1 << 46;  // descriptor version (sm_100); layout type 0 = no swizzle
  return d;
}

__device__ __forceinline__ void bulk_load_1d(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

__global__ void __launch_bounds__(kThreadsStem, 1)
    stem_conv_kernel(const __grid_constant__ CUtensorMap map_in, const __grid_constant__ CUtensorMap map_out,
                     const __half* __restrict__ wpack, const StemParams p) {
  constexpr int S = kStagesStem;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* wsm = smem;
  uint8_t* ring = smem + kWBytes;
  uint8_t* staging = ring + S * kPatchSlot;  // [2 groups][2][kSlab], 1024-aligned
  uint64_t* bars = reinterpret_cast<uint64_t*>(staging + 4 * kSlab);
  uint64_t* full = bars;                    // [S]
  uint64_t* empty = bars + S;               // [S]
  uint64_t* tmem_full = bars + 2 * S;       // [2]
  uint64_t* tmem_empty = bars + 2 * S + 2;  // [2]
  uint64_t* w_full = bars + 2 * S + 4;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * S + 6);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_in);
    tma_prefetch_desc(&map_out);
    for (int s = 0; s < S; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full[a], 1);
      mbar_init(&tmem_empty[a], 128);
    }
    mbar_init(w_full, 1);
    mbar_fence_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 128);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int tiles_per_img = p.tiles_w * p.tiles_h;
  pdl_trigger();

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (lane == 0) {
      mbar_expect_tx(w_full, kWBytes);
      bulk_load_1d(wsm, wpack, kWBytes, w_full);  // constant weights: fetched while the previous kernel drains
      pdl_wait();
      int stage = 0, phase = 0;
      for (int t = blockIdx.x; t < p.total_tiles; t += gridDim.x) {
        const int n = t / tiles_per_img, rem = t - n * tiles_per_img;
        const int th = rem / p.tiles_w, tw = rem - th * p.tiles_w;
        mbar_wait(&empty[stage], phase ^ 1);
        mbar_expect_tx(&full[stage], kPatchBytes);
        // box (11 pairs x 8 ch, E/O, 37 rows, 1 image) at (64 tw, 0, 32 th, n)
        tma_load_5d(&map_in, &full[stage], ring + stage * kPatchSlot, tw * kTileW * 8, 0, th * 2 * kTileH, n, 0);
        if (++stage == S) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc_f16(64, 128);
      mbar_wait(w_full, 0);
      const uint32_t w_addr = smem_u32(wsm);
      int stage = 0, phase = 0, it = 0;
      for (int t = blockIdx.x; t < p.total_tiles; t += gridDim.x, ++it) {
        const int acc = it & 1;
        mbar_wait(&tmem_empty[acc], ((it >> 1) & 1) ^ 1);
        mbar_wait(&full[stage], phase);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * 64;
        const uint32_t patch = smem_u32(ring + stage * kPatchSlot);
#pragma unroll
        for (int r = 0; r < 7; ++r) {
#pragma unroll
          for (int s = 0; s < 4; ++s) {
            // A: rows j at 16 B from pair j + s of padded row 2i + r; row groups i two padded rows apart
            const uint64_t da = umma_desc_linear(patch + r * kRowStride + s * 16, kParStride, 2 * kRowStride);
            // B: [E/O][64 ch][8]: rows (channels) at 16 B, groups of 8 channels 128 B apart, K chunks 1 KB apart
            const uint64_t db = umma_desc_linear(w_addr + (r * 4 + s) * kWTileBytes, 1024, 128);
            umma_f16(d_tmem, da, db, idesc, (r | s) ? 1u : 0u);
          }
        }
        umma_commit(&empty[stage]);
        umma_commit(&tmem_full[acc]);
        if (++stage == S) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue (warps 2..9)
    // Two independent warpgroups: group g drains the tiles with (it & 1) == g, i.e. TMEM accumulator g, through its
    // own pair of staging slabs and its own named barrier, so the per-tile chain (TMEM load -> smem -> TMA store)
    // of one tile overlaps the next tile's.
    const int quarter = warp & 3;     // TMEM lanes [32*quarter, +32)
    const int grp = (warp - 2) >> 2;  // which accumulator / tile parity
    const int row = quarter * 32 + lane;
    const bool leader = (quarter == 2 && lane == 0);  // warps 2 and 6
    const uint32_t row_off = (uint32_t)row * 128u;
    const uint32_t sw = (uint32_t)(row & 7);
    const float4* bias4 = reinterpret_cast<const float4*>(p.bias);
    pdl_wait();  // the output buffer may still be read by an earlier kernel
    int use = 0;
    for (int t = blockIdx.x + grp * gridDim.x; t < p.total_tiles; t += 2 * gridDim.x, ++use) {
      const int n = t / tiles_per_img, rem = t - n * tiles_per_img;
      const int th = rem / p.tiles_w, tw = rem - th * p.tiles_w;
      uint8_t* slab = staging + (grp * 2 + (use & 1)) * kSlab;
      // the TMA store that last used this slab (two of this group's tiles ago) must have finished reading it
      if (leader) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
      asm volatile("bar.sync %0, 128;" ::"r"(1 + grp) : "memory");
      mbar_wait(&tmem_full[grp], use & 1);
      tc_fence_after();
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        uint32_t v[32];
        tmem_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + grp * 64 + h * 32, v);
        tmem_ld_wait();
        if (h == 1) {
          tc_fence_before();
          mbar_arrive(&tmem_empty[grp]);
        }
#pragma unroll
        for (int q4 = 0; q4 < 4; ++q4) {
          const int q = h * 4 + q4;
          const float4 b0 = __ldg(bias4 + q * 2), b1 = __ldg(bias4 + q * 2 + 1);
          const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
          float a[8];
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            a[k] = __uint_as_float(v[q4 * 8 + k]) + bb[k];
            if (p.relu) a[k] = fmaxf(a[k], 0.f);
          }
          *reinterpret_cast<uint4*>(slab + row_off + (((uint32_t)q ^ sw) << 4)) =
              make_uint4(pack_half2(a[0], a[1]), pack_half2(a[2], a[3]), pack_half2(a[4], a[5]), pack_half2(a[6], a[7]));
        }
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      asm volatile("bar.sync %0, 128;" ::"r"(1 + grp) : "memory");
      if (leader) {
        tma_store_5d(&map_out, slab, 0, tw * kTileW, th * kTileH, n, 0);
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      }
    }
    if (leader) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 128);
  }
}

}  // namespace

// in: EO-layout padded image [n][Hin+6][2][(Win+8)/2][8] fp16; w: packed [7][4][2][64][8] fp16 (packing.pack_conv7)
int stem_conv_launch(const GemmLayer& L, cudaStream_t stream) {
  FP_REQUIRE(L.Cin == 8 && L.Cout == 64, "CONV7_S2: the stem kernel is 8 (6 + 2 zero) -> 64 channels");
  FP_REQUIRE(L.Hin % (2 * kTileH) == 0 && L.Win % (2 * kTileW) == 0, "CONV7_S2: unsupported size %dx%d", L.Hin, L.Win);
  FP_REQUIRE(!L.res && !L.post_add && L.out_split == 0, "CONV7_S2: residual / post-add / split are not supported");
  FP_REQUIRE(L.out_ld % 8 == 0 && L.out_ld >= 64, "CONV7_S2: bad out_ld %d", L.out_ld);
  FP_REQUIRE((reinterpret_cast<uintptr_t>(L.w) & 15) == 0, "CONV7_S2: weights must be 16-byte aligned");
  if (L.n_img == 0) return 0;
  const int Ho = L.Hin / 2, Wo = L.Win / 2;
  const uint64_t E = 2;
  const uint64_t rows = L.Hin + 6, pairs = (L.Win + 8) / 2;
  CUtensorMap mi, mo;
  {
    // (channel, pair) are contiguous in memory and are merged into one dimension, so that a box row is the
    // 176 contiguous bytes of 11 pairs: the TMA unit's cost is per box row, not per byte
    uint64_t d[5] = {8 * pairs, 2, rows, (uint64_t)L.n_img, 1};
    uint64_t s[4] = {pairs * 8 * E, 2 * pairs * 8 * E, rows * 2 * pairs * 8 * E, rows * 2 * pairs * 8 * E * L.n_img};
    uint32_t b[5] = {8 * (uint32_t)kPatchPairs, 2, (uint32_t)kPatchRows, 1, 1};
    int rc = encode_map_f16_linear(&mi, L.in, 5, d, s, b);
    if (rc) return rc;
  }
  {
    uint64_t d[5] = {(uint64_t)L.out_ld, (uint64_t)Wo, (uint64_t)Ho, (uint64_t)L.n_img, 1};
    uint64_t s[4] = {(uint64_t)L.out_ld * E, (uint64_t)L.out_ld * E * Wo, (uint64_t)L.out_ld * E * Wo * Ho,
                     (uint64_t)L.out_ld * E * Wo * Ho * L.n_img};
    uint32_t b[5] = {64, (uint32_t)kTileW, (uint32_t)kTileH, 1, 1};
    int rc = encode_map_f16(&mo, L.out, 5, d, s, b);
    if (rc) return rc;
  }
  StemParams p;
  p.tiles_w = Wo / kTileW;
  p.tiles_h = Ho / kTileH;
  p.n_img = L.n_img;
  p.total_tiles = p.tiles_w * p.tiles_h * L.n_img;
  p.bias = L.bias;
  p.relu = L.relu;
  static std::atomic<unsigned long long> attr_mask{0};  // per device: the attribute is device state
  if (!device_bit_test(attr_mask)) {
    FP_CUDA_OK(cudaFuncSetAttribute(stem_conv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kStemSmem));
    device_bit_set(attr_mask);
  }
  const int sms = num_sms();
  FP_REQUIRE(sms > 0, "no CUDA device");
  const int grid = p.total_tiles < sms ? p.total_tiles : sms;
  note_plan({PK_STEM, 64, 1, 0, 0, grid, p.total_tiles, kTileW, kTileH, 1, p.total_tiles, 1});
  prof_mark_begin(0, 2.0 * (double)L.n_img * Ho * Wo * 64.0 * (7.0 * 7.0 * 6.0), stream);
  FP_CUDA_OK(launch_pdl(stem_conv_kernel, dim3(grid), dim3(kThreadsStem), kStemSmem, stream, 1, mi, mo,
                        reinterpret_cast<const __half*>(L.w), p));
  prof_mark_end(stream);
  note_launches(1);
  FP_CUDA_OK(cudaGetLastError());
  return 0;
}

}  // namespace fp
