// fp_api_ops.cu — C-ABI entry points that expose single operators (used by the parity tests to
// bisect the pipeline layer by layer; the product entry points live in fp_api.cu).
#include "../../include/fpose.h"
#include "fp_common.cuh"
#include "fp_attn.cuh"
#include "fp_crop.cuh"
#include "fp_gemm.cuh"

#include <vector>

namespace fp {
const char* get_last_error();
int prof_collect(int kind, double* total_ms, double* total_work, int* launches);
}

extern "C" {

const char* fp_last_error(void) { return fp::get_last_error(); }

unsigned long long fp_launch_count(void) { return fp::launch_count(); }

int fp_prof_enable(int on) {
  fp::g_prof_on = on != 0;
  return 0;
}

int fp_prof_collect(int kind, double* total_ms, double* total_work, int* launches) {
  if (!total_ms || !total_work || !launches) {
    fp::set_last_error("fp_prof_collect: null output");
    return -1;
  }
  return fp::prof_collect(kind, total_ms, total_work, launches);
}

int fp_op_build_meshlets(int V, int F, const float* pos, const int* faces, int* info, int* face_of_tri_out,
                         float* meshlets_out) {
  try {
    if (!pos || !faces || !info || V <= 0 || F <= 0) {
      fp::set_last_error("fp_op_build_meshlets: bad argument");
      return -1;
    }
    for (int i = 0; i < 3 * F; ++i)
      if (faces[i] < 0 || faces[i] >= V) {
        fp::set_last_error("fp_op_build_meshlets: face index out of range");
        return -1;
      }
    std::vector<float> nrm((size_t)V * 3, 0.f), att((size_t)V * 3, 0.f);
    fp::MeshHost mh;
    int rc = fp::build_mesh_host(V, F, pos, nrm.data(), att.data(), 3, faces, mh);
    if (rc) return rc;
    int max_t = 0, max_v = 0, total = 0;
    for (const fp::Meshlet& m : mh.meshlets) {
      max_t = m.n_tris > max_t ? m.n_tris : max_t;
      max_v = m.n_verts > max_v ? m.n_verts : max_v;
      total += m.n_tris;
      for (int t = 0; t < m.n_tris; ++t) {
        const uint2 tr = mh.ml_tris[m.tri_off + t];
        for (int k = 0; k < 3; ++k) {
          const int slot = (tr.x >> (8 * k)) & 255;
          if (slot >= m.n_verts || mh.ml_verts[m.vert_off + slot] != faces[3 * tr.y + k]) {
            fp::set_last_error("fp_op_build_meshlets: meshlet triangle does not map back to its face");
            return -4;
          }
          // every vertex of the meshlet lies inside its bounding sphere
          const float* q = pos + 3 * faces[3 * tr.y + k];
          const float dx = q[0] - m.cx, dy = q[1] - m.cy, dz = q[2] - m.cz;
          if (dx * dx + dy * dy + dz * dz > m.r * m.r * 1.0001f + 1e-12f) {
            fp::set_last_error("fp_op_build_meshlets: vertex outside the meshlet's bounding sphere");
            return -4;
          }
        }
        if (face_of_tri_out) face_of_tri_out[m.tri_off + t] = (int)tr.y;
      }
    }
    if (meshlets_out)
      for (size_t i = 0; i < mh.meshlets.size(); ++i) {
        const fp::Meshlet& m = mh.meshlets[i];
        const float rec[8] = {m.cx, m.cy, m.cz, m.r, m.ax, m.ay, m.az, m.cutoff};
        for (int k = 0; k < 8; ++k) meshlets_out[8 * i + k] = rec[k];
      }
    info[0] = (int)mh.meshlets.size();
    info[1] = mh.closed;
    info[2] = mh.front_sign;
    info[3] = max_t;
    info[4] = max_v;
    info[5] = total;
    return 0;
  } catch (...) {
    fp::set_last_error("fp_op_build_meshlets: exception");
    return -3;
  }
}

int fp_op_attention(const void* qkv, void* out, int B, int impl, void* stream) {
  if (!qkv || !out) {
    fp::set_last_error("fp_op_attention: null argument");
    return -1;
  }
  fp::AttnParams ap;
  ap.qkv = reinterpret_cast<const __half*>(qkv);
  ap.ld = 1536;
  ap.q_off = 0;
  ap.k_off = 512;
  ap.v_off = 1024;
  ap.group_col_stride = 0;
  ap.n_groups = 1;
  ap.out = reinterpret_cast<__half*>(out);
  ap.ld_out = 512;
  ap.out_group_stride = 0;
  ap.B = B;
  ap.T = 400;
  ap.n_heads = 4;
  ap.scale = 0.08838834764831845f;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  (void)impl;  // one implementation: the tcgen05 kernel
  return fp::attn_tc_launch(ap, st);
}

int fp_op_attention_grouped(const void* qkv, void* out, int B, int n_groups, void* stream) {
  if (!qkv || !out || B < 0 || (n_groups != 1 && n_groups != 2)) {
    fp::set_last_error("fp_op_attention_grouped: null argument, B < 0 or n_groups not 1 / 2");
    return -1;
  }
  // the AttnParams of run_score_feats (n_groups = 1) and run_refine_heads (n_groups = 2) in fp_api.cu
  fp::AttnParams ap;
  ap.qkv = reinterpret_cast<const __half*>(qkv);
  ap.ld = 1536 * n_groups;
  ap.q_off = 0;
  ap.k_off = 512;
  ap.v_off = 1024;
  ap.group_col_stride = n_groups == 2 ? 1536 : 0;
  ap.n_groups = n_groups;
  ap.out = reinterpret_cast<__half*>(out);
  ap.ld_out = 512;
  ap.out_group_stride = n_groups == 2 ? (size_t)B * 400 * 512 : 0;
  ap.B = B;
  ap.T = 400;
  ap.n_heads = 4;
  ap.scale = 0.08838834764831845f;
  return fp::attn_core_launch(ap, reinterpret_cast<cudaStream_t>(stream));
}

int fp_op_gemm_last_plan(int* out, int n) {
  if (!out || n < 0) {
    fp::set_last_error("fp_op_gemm_last_plan: null output");
    return -1;
  }
  fp::GemmPlan pl;
  if (!fp::last_plan(&pl)) {
    fp::set_last_error("fp_op_gemm_last_plan: no GEMM launch on this thread yet");
    return -1;
  }
  const int v[FP_GEMM_PLAN_FIELDS] = {pl.kernel, pl.bn,   pl.cg, pl.slabs, pl.patch,   pl.grid,
                                      pl.work_tiles, pl.bw, pl.bh, pl.bimg, pl.m_tiles, pl.n_tiles};
  for (int i = 0; i < n && i < FP_GEMM_PLAN_FIELDS; ++i) out[i] = v[i];
  return 0;
}

int fp_op_gemm_layer(const fp_gemm_layer_t* l, void* stream) {
  if (!l) {
    fp::set_last_error("fp_op_gemm_layer: null layer");
    return -1;
  }
  fp::GemmLayer L;
  L.kind = l->kind;
  L.n_img = l->n_img;
  L.Hin = l->Hin;
  L.Win = l->Win;
  L.Cin = l->Cin;
  L.Cout = l->Cout;
  L.in = l->in;
  L.w = l->w;
  L.bias = l->bias;
  L.res = l->res;
  L.res_ld = l->res_ld;
  L.out = l->out;
  L.out_ld = l->out_ld;
  L.out_split = l->out_split;
  L.post_add = l->post_add;
  L.relu = l->relu;
  return fp::gemm_layer_launch(L, reinterpret_cast<cudaStream_t>(stream));
}

}  // extern "C"
