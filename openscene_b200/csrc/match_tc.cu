// Open-vocabulary matching on 5th-gen tensor cores (run/evaluate.py:288-323).
//
//   scores[p, k] = fp16( sum_c a[p, c] * text[k, c] ),  a[p,:] = fp16( prep(feat[v(p), :]) ),  fp32 accumulation
//
// with prep = identity (`.half()`), or x / (|x| + 1e-5) (the normalised products of the ensemble branch), v(p) =
// inds_reverse[p] (voxel -> point expansion without materialising predictions[inds_reverse]), or a per-point choice
// between the 3-D and the fused 2-D feature (ensemble select).  The operands are rounded to fp16 exactly where the
// reference rounds them, so the [N_pts, C] x [C, K] product is the reference's own fp16 GEMM.
//
// One CTA = 128 points.  Warps 0-15 build the A operand: one warp per row at a time, the row lives in registers
// (coalesced 256-byte loads), is reduced for the norm, rounded to fp16 and written into the K-major 128B-swizzled
// shared-memory tile of all C/64 depth chunks (192 KB for C = 768).  Warp 16 streams the text matrix chunk by chunk with
// TMA (rows >= K_text are out of bounds -> zero fill), warp 17 issues `tcgen05.mma kind::f16` (M=128, N<=96 per pass,
// K=16), warps 0-3 read the accumulators from TMEM, round to fp16, take the first-maximum argmax and write
// scores / labels / row maxima.  HBM-bound: 4*C (or 2*C) bytes per point against 2*C*K flops.
//
// Accumulate epilogue (osb_match_accumulate, the test_repeats loop of run/evaluate.py:385-425): with `store` set, each
// fp16 score h is folded into the caller's running fp16 sum instead of being written out -- store = h + 0.0 on the first
// repeat (turns -0 into +0 like the reference's `pred + 0.0`), store = __hadd(h, store) after it (one fp16 rounding,
// bit-identical to torch's fp32 add rounded to fp16) -- and the label is the first maximum of the ACCUMULATED row.
#include "tc_ptx.cuh"
#include <algorithm>

namespace osb {

constexpr int MT_M = 128;
constexpr int MT_NW = 96;            // text rows per MMA pass (N of the instruction)
constexpr int MT_PW = 16;             // A-producer warps (8 rows each)
constexpr int MT_THREADS = (MT_PW + 2) * 32;   // + TMA warp + MMA warp
constexpr int MT_BSTAGES = 2;

struct MatchTcParams {
  const void *feat;                  // [n_vox, C] fp32 or fp16
  const __half *feat2;               // optional second source (fp16) for the ensemble select
  const float *sel_a, *sel_b;        // ensemble: use feat2 where sel_a[p] < sel_b[p]
  const int64_t *inds_reverse;       // [n_pts] or NULL
  int64_t n_pts;
  int C, k_text, n_pass, tmem_cols;
  int feat_is_f16, normalize;
  __half *scores;                    // [n_pts, k_text] or NULL
  int64_t *label;                    // [n_pts] or NULL
  float *smax;                       // [n_pts] or NULL
  __half *feat_out;                  // [n_pts, C] or NULL: the fp16 operand actually multiplied (ensemble feature)
  __half *store;                     // [n_pts, k_text] or NULL: running fp16 sum over repeats (accumulate epilogue)
  int first;                         // store: 1 = first repeat (store is write-only)
};

__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t acc) {
  umma_bf16(tmem_d, desc_a, desc_b, idesc, acc);      // same instruction; operand format comes from the descriptor
}

template <int NP>   // half2 pairs per lane: C = 64 * NP
__global__ void __launch_bounds__(MT_THREADS, 1)
k_match_tc(const __grid_constant__ CUtensorMap tmT, const MatchTcParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  constexpr int C = 64 * NP;
  constexpr int A_BYTES = NP * MT_M * 128;                      // NP chunks of [128 rows x 128 B]
  constexpr int B_BYTES = MT_NW * 128;
  uint8_t *sA = smem, *sB = smem + A_BYTES;
  uint64_t *bars = reinterpret_cast<uint64_t *>(sB + MT_BSTAGES * B_BYTES);   // b_full[2], b_empty[2], a_full, accum
  uint32_t *s_misc = reinterpret_cast<uint32_t *>(bars + 8);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int64_t row0 = (int64_t)blockIdx.x * MT_M;
  const uint32_t b_full = smem_u32(bars), b_empty = smem_u32(bars + 2), a_full = smem_u32(bars + 4), accum = smem_u32(bars + 5);

  if (tid == 0) {
    for (int s = 0; s < MT_BSTAGES; ++s) { mbar_init(b_full + 8 * s, 1); mbar_init(b_empty + 8 * s, 1); }
    mbar_init(a_full, MT_PW * 32);
    mbar_init(accum, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == MT_PW + 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s_misc[0])), "r"((uint32_t)p.tmem_cols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  if (tid == MT_PW * 32) asm volatile("prefetch.tensormap [%0];" ::"l"(&tmT) : "memory");
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = s_misc[0];
  const int n_stage = p.n_pass * NP;

  if (warp < MT_PW) {
    // ============================ A producers: 8 rows per warp ==============================
    // RB rows are in flight per warp (their loads are issued before any is consumed): 16 warps x RB x 3 KB of
    // outstanding loads per SM keeps HBM busy from the single resident CTA; 16 warps also spread the
    // convert / normalise instruction stream over all four schedulers.
    constexpr int RB = 2, ROWS_PW = MT_M / MT_PW;
    for (int rr0 = 0; rr0 < ROWS_PW; rr0 += RB) {
      float v[RB][2 * NP];
      bool f16[RB], live[RB];
      float ss[RB];
#pragma unroll
      for (int u = 0; u < RB; ++u) {
        const int64_t pt = row0 + warp * ROWS_PW + rr0 + u;
        live[u] = pt < p.n_pts;
        f16[u] = false;
        ss[u] = 0.f;
        if (live[u]) {
          const int64_t vox = p.inds_reverse ? __ldg(p.inds_reverse + pt) : pt;
          bool second = false;
          if (p.feat2 != nullptr) second = (p.sel_a == nullptr) ? true : (__ldg(p.sel_a + pt) < __ldg(p.sel_b + pt));
          f16[u] = second || p.feat_is_f16;
          const void *src = second ? (const void *)p.feat2 : p.feat;
          if (f16[u]) {
            const __half2 *q = reinterpret_cast<const __half2 *>(src) + vox * (C / 2);
#pragma unroll
            for (int j = 0; j < NP; ++j) {
              const float2 f = __half22float2(__ldg(q + lane + 32 * j));
              v[u][2 * j] = f.x; v[u][2 * j + 1] = f.y;
            }
          } else {
            const float2 *q = reinterpret_cast<const float2 *>(src) + vox * (C / 2);
#pragma unroll
            for (int j = 0; j < NP; ++j) {
              const float2 f = __ldg(q + lane + 32 * j);
              v[u][2 * j] = f.x; v[u][2 * j + 1] = f.y;
            }
          }
        } else {
#pragma unroll
          for (int j = 0; j < 2 * NP; ++j) v[u][j] = 0.f;
        }
      }
#pragma unroll
      for (int u = 0; u < RB; ++u) {
        const int r = warp * ROWS_PW + rr0 + u;
        const int64_t pt = row0 + r;
        if (p.normalize) {
#pragma unroll
          for (int j = 0; j < 2 * NP; ++j) ss[u] = fmaf(v[u][j], v[u][j], ss[u]);
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) ss[u] += __shfl_xor_sync(0xffffffffu, ss[u], o);
          float nrm = sqrtf(ss[u]);
          float d;
          if (f16[u]) {   // the reference takes norm, +1e-5 and the division on an fp16 tensor (evaluate.py:303-305)
            nrm = __half2float(__float2half_rn(nrm));
            d = __half2float(__float2half_rn(nrm + 1e-5f));
          } else {
            d = nrm + 1e-5f;
          }
          // x / d evaluated as x * (1/d) (one rounding more than the reference's division; the following fp16
          // rounding absorbs it except for values within 2^-24 of an fp16 rounding boundary)
          const float rd = __frcp_rn(d);
#pragma unroll
          for (int j = 0; j < 2 * NP; ++j) v[u][j] = v[u][j] * rd;
        }
        // chunk j of this row: lane holds elements 2*lane, 2*lane+1 -> bytes [4*lane, 4*lane+4) of the 128-byte line
        const uint32_t line = smem_u32(sA) + r * 128 + ((((4 * lane) >> 4) ^ (r & 7)) << 4) + ((4 * lane) & 15);
#pragma unroll
        for (int j = 0; j < NP; ++j) {
          const __half2 h = __floats2half2_rn(v[u][2 * j], v[u][2 * j + 1]);       // the reference's `.half()`
          asm volatile("st.shared.b32 [%0], %1;" ::"r"(line + j * (MT_M * 128)), "r"(*reinterpret_cast<const uint32_t *>(&h)) : "memory");
          if (p.feat_out != nullptr && live[u])
            reinterpret_cast<__half2 *>(p.feat_out)[pt * (C / 2) + lane + 32 * j] = h;
        }
      }
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");           // generic-proxy writes -> UMMA reads
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(a_full) : "memory");
  } else if (warp == MT_PW) {
    // ============================ TMA producer: text chunks ==================================
    int s = 0; uint32_t phase = 0;
    for (int t = 0; t < n_stage; ++t) {
      const int pass = t / NP, c = t % NP;
      mbar_wait(b_empty + 8 * s, phase ^ 1);
      if (elect_one()) {
        mbar_expect_tx(b_full + 8 * s, (uint32_t)B_BYTES);
        tma_load_2d(smem_u32(sB + s * B_BYTES), &tmT, b_full + 8 * s, c * 64, pass * MT_NW);
      }
      __syncwarp();
      if (++s == MT_BSTAGES) { s = 0; phase ^= 1; }
    }
  } else {
    // ============================ MMA issuer ==================================================
    // instruction descriptor: D=f32, A=B=f16 (format 0), K-major both, N = 96, M = 128
    const uint32_t idesc = (1u << 4) | ((uint32_t)(MT_NW >> 3) << 17) | ((uint32_t)(MT_M >> 4) << 24);
    mbar_wait(a_full, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    int s = 0; uint32_t phase = 0;
    for (int t = 0; t < n_stage; ++t) {
      const int pass = t / NP, c = t % NP;
      mbar_wait(b_full + 8 * s, phase);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      if (elect_one()) {
        const uint64_t da = umma_desc(smem_u32(sA + c * (MT_M * 128))), db = umma_desc(smem_u32(sB + s * B_BYTES));
#pragma unroll
        for (int h = 0; h < 4; ++h)      // 64 fp16 per chunk = 4 K-steps of 16 (32 bytes each)
          umma_f16(tmem_base + pass * MT_NW, da + 2 * h, db + 2 * h, idesc, (c > 0 || h > 0) ? 1u : 0u);
        umma_commit(b_empty + 8 * s);
      }
      __syncwarp();
      if (++s == MT_BSTAGES) { s = 0; phase ^= 1; }
    }
    if (elect_one()) umma_commit(accum);
    __syncwarp();
  }

  if (warp < 4) {
    // ============================ epilogue: fp16 rounding, argmax =============================
    mbar_wait(accum, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const int64_t pt = row0 + warp * 32 + lane;
    float best = -INFINITY;
    int best_k = 0;
    for (int col = 0; col < p.n_pass * MT_NW; col += 16) {
      if (col >= p.k_text) break;                                   // warp-uniform
      uint32_t a[16];
      tmem_ld16(tmem_base + ((uint32_t)(warp * 32) << 16) + col, a);
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const int k = col + j;
        if (k < p.k_text) {
          __half h = __float2half_rn(__uint_as_float(a[j]));
          if (p.store != nullptr && pt < p.n_pts) {
            __half *st = p.store + pt * p.k_text + k;
            h = __hadd(h, p.first ? __float2half_rn(0.f) : *st);
            *st = h;
          }
          const float sc = __half2float(h);
          if (p.scores != nullptr && pt < p.n_pts) p.scores[pt * p.k_text + k] = h;
          if (sc > best) { best = sc; best_k = k; }
        }
      }
    }
    if (pt < p.n_pts) {
      if (p.label) p.label[pt] = best_k;
      if (p.smax) p.smax[pt] = best;
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == MT_PW + 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)p.tmem_cols));
}

static int launch_match_tc(const MatchTcParams &p, const void *text_f16, cudaStream_t stream) {
  CUtensorMap tmT;
  if (make_tmap_2b(&tmT, text_f16, (uint64_t)p.C, (uint64_t)p.k_text, MT_NW, 1)) return 1;
  const int NP = p.C / 64;
  const size_t smem = (size_t)NP * MT_M * 128 + MT_BSTAGES * MT_NW * 128 + 128 + 1024;
  const unsigned grid = (unsigned)ceil_div(p.n_pts, MT_M);
  if (NP == 12) {
    OSB_SMEM_ATTR_ONCE(k_match_tc<12>, 227 * 1024);
    k_match_tc<12><<<grid, MT_THREADS, smem, stream>>>(tmT, p);
  } else {
    OSB_SMEM_ATTR_ONCE(k_match_tc<8>, 227 * 1024);
    k_match_tc<8><<<grid, MT_THREADS, smem, stream>>>(tmT, p);
  }
  OSB_LAUNCH_CHECK();
  return 0;
}

int match_tc_run(const void *feat, int feat_is_f16, const void *feat2_f16, const float *sel_a, const float *sel_b, int c,
                 const int64_t *inds_reverse, int64_t n_pts, const void *text_f16, int k_text, int normalize,
                 void *scores_f16, int64_t *label, float *smax, void *feat_out_f16, void *store_f16, int first,
                 cudaStream_t stream) {
  MatchTcParams p{};
  p.feat = feat; p.feat2 = (const __half *)feat2_f16; p.sel_a = sel_a; p.sel_b = sel_b;
  p.inds_reverse = inds_reverse; p.n_pts = n_pts; p.C = c; p.k_text = k_text;
  p.n_pass = (k_text + MT_NW - 1) / MT_NW;
  OSB_CHECK(p.n_pass * MT_NW <= 512, "match: K_text=%d too large for one TMEM allocation", k_text);
  p.tmem_cols = 32;
  while (p.tmem_cols < p.n_pass * MT_NW) p.tmem_cols <<= 1;
  p.feat_is_f16 = feat_is_f16; p.normalize = normalize;
  p.scores = (__half *)scores_f16; p.label = label; p.smax = smax; p.feat_out = (__half *)feat_out_f16;
  p.store = (__half *)store_f16; p.first = first;
  return launch_match_tc(p, text_f16, stream);
}

}  // namespace osb
