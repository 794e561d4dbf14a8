// Open-vocabulary matching: voxel->point gather, optional L2 normalisation, fp16 product with the
// CLIP text embeddings, row max / argmax -- one pass over the features, nothing materialised at
// [N_pts, C].  Replaces the torch ops at run/evaluate.py:288-323.
//
// HBM-bound: 4*C bytes read per point (3 KB at C = 768) against 2*C*K flops; one warp owns one
// point, the text matrix (K*C*2 bytes, <= 245 KB) stays in L1/L2.
#include "common.cuh"
#include <algorithm>
#include <stdlib.h>

namespace osb {

template <int NP>  // half2 pairs per lane: C = 64 * NP
struct RowRegs {
  float v[2 * NP];
};

// load a feature row into registers as the fp16-rounded values the reference multiplies
template <int NP, bool F16, bool NORMALIZE>
__device__ __forceinline__ void load_row(const void *__restrict__ feat, int64_t row, int lane, RowRegs<NP> &r) {
  constexpr int C = 64 * NP;
  float ss = 0.f;
  if (F16) {
    const __half2 *p = reinterpret_cast<const __half2 *>(feat) + row * (C / 2);
#pragma unroll
    for (int j = 0; j < NP; ++j) {
      const float2 f = __half22float2(__ldg(p + lane + 32 * j));
      r.v[2 * j] = f.x; r.v[2 * j + 1] = f.y;
      ss += f.x * f.x + f.y * f.y;
    }
  } else {
    const float2 *p = reinterpret_cast<const float2 *>(feat) + row * (C / 2);
#pragma unroll
    for (int j = 0; j < NP; ++j) {
      const float2 f = __ldg(p + lane + 32 * j);
      r.v[2 * j] = f.x; r.v[2 * j + 1] = f.y;
      ss += f.x * f.x + f.y * f.y;
    }
  }
  if (NORMALIZE) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    float nrm = sqrtf(ss);
    if (F16) {
      // the reference takes norm / +1e-5 / division on an fp16 tensor (evaluate.py:303-305)
      nrm = __half2float(__float2half_rn(nrm));
      const float d = __half2float(__float2half_rn(nrm + 1e-5f));
#pragma unroll
      for (int j = 0; j < 2 * NP; ++j) r.v[j] = __half2float(__float2half_rn(r.v[j] / d));
    } else {
      const float d = nrm + 1e-5f;
#pragma unroll
      for (int j = 0; j < 2 * NP; ++j) r.v[j] = __half2float(__float2half_rn(r.v[j] / d));
    }
  } else if (!F16) {
#pragma unroll
    for (int j = 0; j < 2 * NP; ++j) r.v[j] = __half2float(__float2half_rn(r.v[j]));   // .half()
  }
}

template <int NP>
__device__ __forceinline__ void score_row(const RowRegs<NP> &r, const __half2 *__restrict__ text, int k_text, int lane,
                                          __half *__restrict__ scores_row, float &best, int &best_k) {
  constexpr int C = 64 * NP;
  best = -INFINITY;
  best_k = 0;
  for (int k = 0; k < k_text; ++k) {
    const __half2 *t = text + (int64_t)k * (C / 2);
    float acc = 0.f;
#pragma unroll
    for (int j = 0; j < NP; ++j) {
      const float2 f = __half22float2(__ldg(t + lane + 32 * j));
      acc = fmaf(r.v[2 * j], f.x, acc);
      acc = fmaf(r.v[2 * j + 1], f.y, acc);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    const __half h = __float2half_rn(acc);
    const float s = __half2float(h);
    if (scores_row != nullptr && lane == 0) scores_row[k] = h;
    if (s > best) { best = s; best_k = k; }
  }
}

template <int NP, bool F16, bool NORMALIZE>
__global__ void __launch_bounds__(256)
k_match_scores(const void *__restrict__ feat, const int64_t *__restrict__ inds_reverse, int64_t n_pts,
               const __half2 *__restrict__ text, int k_text, __half *__restrict__ scores, int64_t *__restrict__ label,
               float *__restrict__ smax) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t p = warp; p < n_pts; p += nwarps) {
    const int64_t v = inds_reverse ? inds_reverse[p] : p;
    RowRegs<NP> r;
    load_row<NP, F16, NORMALIZE>(feat, v, lane, r);
    float best; int best_k;
    score_row<NP>(r, text, k_text, lane, scores ? scores + p * k_text : nullptr, best, best_k);
    if (lane == 0) {
      if (label) label[p] = best_k;
      if (smax) smax[p] = best;
    }
  }
}

template <int NP>
__global__ void __launch_bounds__(256)
k_match_ensemble(const float *__restrict__ feat3d, const __half *__restrict__ feat2d, const int64_t *__restrict__ inds_reverse,
                 int64_t n_pts, const float *__restrict__ smax3d, const float *__restrict__ smax2d,
                 const __half2 *__restrict__ text, int k_text, __half *__restrict__ scores, int64_t *__restrict__ label,
                 __half *__restrict__ feat_out) {
  constexpr int C = 64 * NP;
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t p = warp; p < n_pts; p += nwarps) {
    const int64_t v = inds_reverse ? inds_reverse[p] : p;
    const bool use2d = smax3d[p] < smax2d[p];
    RowRegs<NP> r;
    if (use2d) load_row<NP, true, false>(feat2d, v, lane, r);
    else       load_row<NP, false, false>(feat3d, v, lane, r);
    if (feat_out) {
      __half2 *o = reinterpret_cast<__half2 *>(feat_out) + p * (C / 2);
#pragma unroll
      for (int j = 0; j < NP; ++j) o[lane + 32 * j] = __floats2half2_rn(r.v[2 * j], r.v[2 * j + 1]);
    }
    float best; int best_k;
    score_row<NP>(r, text, k_text, lane, scores ? scores + p * k_text : nullptr, best, best_k);
    if (lane == 0 && label) label[p] = best_k;
  }
}

// tensor-core implementation (match_tc.cu)
int match_tc_run(const void *feat, int feat_is_f16, const void *feat2_f16, const float *sel_a, const float *sel_b, int c,
                 const int64_t *inds_reverse, int64_t n_pts, const void *text_f16, int k_text, int normalize,
                 void *scores_f16, int64_t *label, float *smax, void *feat_out_f16, void *store_f16, int first,
                 cudaStream_t stream);

static bool use_simt() {   // OSB_MATCH_SIMT=1 selects the CUDA-core kernels below (cross-check path)
  static int v = -1;
  if (v < 0) { const char *e = getenv("OSB_MATCH_SIMT"); v = (e && e[0] == '1') ? 1 : 0; }
  return v == 1;
}

static unsigned match_grid(int64_t n_pts) {
  return (unsigned)std::min<int64_t>(ceil_div(n_pts, 8), 148 * 8);
}

}  // namespace osb

using namespace osb;

extern "C" {

int osb_match_scores(const void *feat, int32_t feat_is_f16, int64_t n_vox, int32_t c, const int64_t *inds_reverse,
                     int64_t n_pts, const void *text_f16, int32_t k_text, int32_t normalize, void *scores_f16,
                     int64_t *label, float *smax, void *stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  OSB_CHECK(c == 512 || c == 768, "osb_match_scores: feature width %d unsupported (OpenScene uses 512 / 768)", c);
  OSB_CHECK(k_text >= 1 && n_vox > 0, "osb_match_scores: bad shape");
  if (n_pts == 0) return 0;
  if (!use_simt())
    return match_tc_run(feat, feat_is_f16, nullptr, nullptr, nullptr, c, inds_reverse, n_pts, text_f16, k_text, normalize,
                        scores_f16, label, smax, nullptr, nullptr, 0, stream);
  const unsigned grid = match_grid(n_pts);
  const __half2 *text = (const __half2 *)text_f16;
  __half *scores = (__half *)scores_f16;
#define OSB_MS(NP, F16, NRM) \
  k_match_scores<NP, F16, NRM><<<grid, 256, 0, stream>>>(feat, inds_reverse, n_pts, text, k_text, scores, label, smax)
  if (c == 768) {
    if (feat_is_f16) { if (normalize) OSB_MS(12, true, true); else OSB_MS(12, true, false); }
    else             { if (normalize) OSB_MS(12, false, true); else OSB_MS(12, false, false); }
  } else {
    if (feat_is_f16) { if (normalize) OSB_MS(8, true, true); else OSB_MS(8, true, false); }
    else             { if (normalize) OSB_MS(8, false, true); else OSB_MS(8, false, false); }
  }
#undef OSB_MS
  OSB_LAUNCH_CHECK();
  return 0;
}

int osb_match_ensemble(const float *feat3d, const void *feat2d_f16, int64_t n_vox, int32_t c, const int64_t *inds_reverse,
                       int64_t n_pts, const float *smax3d, const float *smax2d, const void *text_f16, int32_t k_text,
                       void *scores_f16, int64_t *label, void *feat_out_f16, void *stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  OSB_CHECK(c == 512 || c == 768, "osb_match_ensemble: feature width %d unsupported", c);
  OSB_CHECK(k_text >= 1 && n_vox > 0, "osb_match_ensemble: bad shape");
  if (n_pts == 0) return 0;
  if (!use_simt())
    return match_tc_run(feat3d, 0, feat2d_f16, smax3d, smax2d, c, inds_reverse, n_pts, text_f16, k_text, 0, scores_f16, label,
                        nullptr, feat_out_f16, nullptr, 0, stream);
  const unsigned grid = match_grid(n_pts);
  if (c == 768)
    k_match_ensemble<12><<<grid, 256, 0, stream>>>(feat3d, (const __half *)feat2d_f16, inds_reverse, n_pts, smax3d, smax2d,
                                                   (const __half2 *)text_f16, k_text, (__half *)scores_f16, label,
                                                   (__half *)feat_out_f16);
  else
    k_match_ensemble<8><<<grid, 256, 0, stream>>>(feat3d, (const __half *)feat2d_f16, inds_reverse, n_pts, smax3d, smax2d,
                                                  (const __half2 *)text_f16, k_text, (__half *)scores_f16, label,
                                                  (__half *)feat_out_f16);
  OSB_LAUNCH_CHECK();
  return 0;
}

int osb_match_accumulate(const void *feat, int32_t feat_is_f16, const void *feat2_f16, const float *sel_a, const float *sel_b,
                         int64_t n_vox, int32_t c, const int64_t *inds_reverse, int64_t n_pts, const void *text_f16,
                         int32_t k_text, int32_t normalize, void *store_f16, int32_t first, int64_t *label, void *stream_) {
  OSB_CHECK(c == 512 || c == 768, "osb_match_accumulate: feature width %d unsupported (OpenScene uses 512 / 768)", c);
  OSB_CHECK(k_text >= 1 && k_text <= 5 * 96, "osb_match_accumulate: K_text=%d outside 1..480 (one TMEM allocation)", k_text);
  OSB_CHECK(n_vox > 0 && n_pts >= 0, "osb_match_accumulate: bad shape (n_vox=%lld, n_pts=%lld)", (long long)n_vox,
            (long long)n_pts);
  OSB_CHECK(inds_reverse != nullptr || n_pts == n_vox,
            "osb_match_accumulate: without inds_reverse n_pts (%lld) must equal n_vox (%lld)", (long long)n_pts, (long long)n_vox);
  OSB_CHECK(feat != nullptr && text_f16 != nullptr, "osb_match_accumulate: feat and text must not be NULL");
  OSB_CHECK(store_f16 != nullptr, "osb_match_accumulate: store (fp16 [n_pts, K], read and written in place) is NULL");
  OSB_CHECK(feat2_f16 == nullptr || (sel_a != nullptr && sel_b != nullptr),
            "osb_match_accumulate: a second source needs both select arrays");
  OSB_CHECK(!use_simt(), "osb_match_accumulate: no CUDA-core variant; OSB_MATCH_SIMT=1 cannot serve the accumulate epilogue");
  if (n_pts == 0) return 0;
  return match_tc_run(feat, feat_is_f16, feat2_f16, sel_a, sel_b, c, inds_reverse, n_pts, text_f16, k_text, normalize, nullptr,
                      label, nullptr, nullptr, store_f16, first ? 1 : 0, (cudaStream_t)stream_);
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------
// Repeat accumulation of class logits (run/eval_mink.py:168-216): one warp per point gathers the voxel's fp32 logits row
// through inds_reverse, folds it into the running fp32 sum (store = pred + 0.0 on the first repeat, pred + store after it)
// and writes the first-maximum argmax of this repeat alone and of the accumulated row.  One pass instead of torch's
// gather + add + two argmaxes over [N_pts, C].
namespace osb {
__device__ __forceinline__ void warp_argmax(float &best, int &best_k) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int ok = __shfl_xor_sync(0xffffffffu, best_k, o);
    if (ob > best || (ob == best && ok < best_k)) { best = ob; best_k = ok; }
  }
}

__global__ void __launch_bounds__(256)
k_logits_accumulate(const float *__restrict__ logits, int c, const int64_t *__restrict__ inds_reverse, int64_t n_pts,
                    float *__restrict__ store, int first, int64_t *__restrict__ label_cur, int64_t *__restrict__ label_acc) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t p = warp; p < n_pts; p += nwarps) {
    const float *src = logits + (inds_reverse ? __ldg(inds_reverse + p) : p) * c;
    float *st = store + p * c;
    float bc = -INFINITY, ba = -INFINITY;
    int kc = 0x7fffffff, ka = 0x7fffffff;
    for (int k = lane; k < c; k += 32) {
      const float v = __ldg(src + k);
      const float s = __fadd_rn(v, first ? 0.f : st[k]);
      st[k] = s;
      if (k == lane || v > bc) { bc = v; kc = k; }       // a lane's first column seeds its candidate (rows of -inf)
      if (k == lane || s > ba) { ba = s; ka = k; }
    }
    warp_argmax(bc, kc);
    warp_argmax(ba, ka);
    if (lane == 0) {
      if (label_cur) label_cur[p] = kc;
      if (label_acc) label_acc[p] = ka;
    }
  }
}
}  // namespace osb

extern "C" int osb_logits_accumulate(const float *logits, int64_t n_vox, int32_t c, const int64_t *inds_reverse, int64_t n_pts,
                                     float *store, int32_t first, int64_t *label_cur, int64_t *label_acc, void *stream_) {
  OSB_CHECK(c >= 1 && n_vox > 0 && n_pts >= 0, "osb_logits_accumulate: bad shape (n_vox=%lld, C=%d, n_pts=%lld)",
            (long long)n_vox, c, (long long)n_pts);
  OSB_CHECK(inds_reverse != nullptr || n_pts == n_vox,
            "osb_logits_accumulate: without inds_reverse n_pts (%lld) must equal n_vox (%lld)", (long long)n_pts, (long long)n_vox);
  OSB_CHECK(logits != nullptr, "osb_logits_accumulate: logits is NULL");
  OSB_CHECK(store != nullptr, "osb_logits_accumulate: store (fp32 [n_pts, C], read and written in place) is NULL");
  if (n_pts == 0) return 0;
  const unsigned grid = (unsigned)std::min<int64_t>(osb::ceil_div(n_pts, 8), 148 * 16);
  osb::k_logits_accumulate<<<grid, 256, 0, (cudaStream_t)stream_>>>(logits, c, inds_reverse, n_pts, store, first ? 1 : 0,
                                                                     label_cur, label_acc);
  OSB_LAUNCH_CHECK();
  return 0;
}

// ---------------------------------------------------------------------------------------------------
// Folded head (optional fast path, openscene_b200/engine.py: forward_scores): the final 1x1x1 convolution
// f = x W (96 -> 768) and the cosine product with the text matrix T are re-associated,
//     f . t_k = x . (W t_k) = x . U_k,      |f|^2 = x (W W^T) x^T = |x L|^2   (W W^T = L L^T, Cholesky),
// so one 96 -> (96 + K) convolution produces z = [x L | x U] and this kernel finishes a row:
//     score_k = fp16( (x.U_k) / (|x L| + 1e-5) ),  label = argmax_k.
namespace osb {
__global__ void k_folded_head_finish(const float *__restrict__ z, int64_t n, int ld, int c_norm, int k_text,
                                     __half *__restrict__ scores, int64_t *__restrict__ label, float *__restrict__ smax) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t p = warp; p < n; p += nwarps) {
    const float *row = z + p * ld;
    float ss = 0.f;
    for (int c = lane; c < c_norm; c += 32) { const float v = __ldg(row + c); ss = fmaf(v, v, ss); }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    const float d = sqrtf(ss) + 1e-5f;
    float best = -INFINITY;
    int best_k = 0x7fffffff;
    for (int k = lane; k < k_text; k += 32) {
      const __half h = __float2half_rn(__ldg(row + c_norm + k) / d);
      if (scores) scores[p * k_text + k] = h;
      const float s = __half2float(h);
      if (s > best) { best = s; best_k = k; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ob = __shfl_xor_sync(0xffffffffu, best, o);
      const int ok = __shfl_xor_sync(0xffffffffu, best_k, o);
      if (ob > best || (ob == best && ok < best_k)) { best = ob; best_k = ok; }
    }
    if (lane == 0) {
      if (label) label[p] = best_k;
      if (smax) smax[p] = best;
    }
  }
}
}  // namespace osb

extern "C" int osb_folded_head_finish(const float *z, int64_t n, int32_t ld, int32_t c_norm, int32_t k_text, void *scores_f16,
                                      int64_t *label, float *smax, void *stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  OSB_CHECK(n > 0 && c_norm > 0 && k_text > 0 && ld >= c_norm + k_text, "osb_folded_head_finish: bad shape");
  const unsigned grid = (unsigned)std::min<int64_t>(osb::ceil_div(n, 8), 148 * 8);
  osb::k_folded_head_finish<<<grid, 256, 0, stream>>>(z, n, ld, c_norm, k_text, (__half *)scores_f16, label, smax);
  OSB_LAUNCH_CHECK();
  return 0;
}
