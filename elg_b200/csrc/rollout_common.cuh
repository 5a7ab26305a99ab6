// Pieces shared by the rollout kernels (rollout.cu: fp32-pipe attention, resident + streaming; rollout_tc.cu:
// tensor-core attention, resident; rollout_stc.cu: tensor-core attention over streamed tiles).  The two tensor-core
// kernels also share their TMEM column plan, the split-precision MMA issue and the local policy (section below).
#pragma once
#include <string.h>
#include "common.cuh"
#include "umma.cuh"

namespace elg {

constexpr int RW = 16;              // warps per CTA
constexpr int RT = RW * 32;         // threads per CTA
constexpr int MT_MAX = 64;          // rows per CTA
constexpr int N_RES_MAX = 112;      // nodes the resident variant supports
constexpr int N_STREAM_MAX = 8192;  // nodes the streaming variant supports (uint16 ids, sort kernel)
constexpr int DS = 128;             // stride of the per-row dense penalty+local scratch (one node chunk)
constexpr int TS = 36;              // padded row stride of the VPE / PE tables in smem
constexpr int SS = 116;             // resident: row stride of the staged scores (112 scores + 4 neighbour-mask words)
constexpr int A_HALF = 16384;       // resident: bytes of one fp16 A operand (64 rows x 128 k, K-major core matrices)
constexpr unsigned FULL = 0xffffffffu;

struct RolloutArgs {
  elg_tables t;
  const float* derived;
  int problem, B, M, N1, MT, tiles, k_local;
  int ns_stride;      // n_steps is indexed [aug-instance * ns_stride + tile] (ns_stride = elg_rollout_tiles())
  float xi, clip;
  const int32_t* start_nodes;
  int mode;
  unsigned long long seed;
  int t_max;
  int16_t* tours;
  float* reward;
  int32_t* n_steps;
  float* logp;
  int32_t* work_counter;
  // single decode step from caller-provided state (model.one_step_rollout)
  int single_step;
  unsigned long long step_id;
  const int32_t* st_cur;
  const float* st_load;
  const int32_t* st_first;
  const uint32_t* st_mask;
  int32_t* out_selected;
  float* out_prob;
  float* out_logits;
};

// ---- streamed tensor-core rollout (rollout_stc.cu): tiles of elg_tables.et and the scratch elg_tables.ws ------------
constexpr int STC_TILE = ELG_TILE_NODES;       // nodes per tile
__host__ __device__ inline int stc_tiles(int N1) { return (N1 + STC_TILE - 1) / STC_TILE; }
struct StcWs {
  size_t mask, vis, nb, total;          // byte offsets: three bit masks [rows][Wp] uint32
  int Wp, NP;                           // mask words per row (4 per tile), padded node count
};
__host__ __device__ inline StcWs stc_ws_layout(long long rows, int N1) {
  StcWs w;
  w.Wp = stc_tiles(N1) * 4;
  w.NP = stc_tiles(N1) * STC_TILE;
  const size_t mb = (size_t)rows * w.Wp * 4;
  w.mask = 0; w.vis = mb; w.nb = 2 * mb;
  w.total = 3 * mb;
  return w;
}

// ---- small PTX helpers --------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// TMA bulk copy global -> shared (1D), completion signalled on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// Philox4x32-10 (counter-based RNG for the sampling mode)
__device__ __forceinline__ uint4 philox4x32(uint4 ctr, uint2 key) {
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    uint32_t hi0 = __umulhi(0xD2511F53u, ctr.x), lo0 = 0xD2511F53u * ctr.x;
    uint32_t hi1 = __umulhi(0xCD9E8D57u, ctr.z), lo1 = 0xCD9E8D57u * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += 0x9E3779B9u;
    key.y += 0xBB67AE85u;
  }
  return ctr;
}

__device__ __forceinline__ float octet_max(float v) {
  v = fmaxf(v, __shfl_xor_sync(FULL, v, 1));
  v = fmaxf(v, __shfl_xor_sync(FULL, v, 2));
  return fmaxf(v, __shfl_xor_sync(FULL, v, 4));
}
__device__ __forceinline__ float octet_sum(float v) {
  v += __shfl_xor_sync(FULL, v, 1);
  v += __shfl_xor_sync(FULL, v, 2);
  return v + __shfl_xor_sync(FULL, v, 4);
}

// ---- the two tensor-core kernels (rollout_tc.cu, rollout_stc.cu) ------------------------------------------------
// TMEM columns: [0,128) Q hi|lo, later O hi|lo   [128,256) O accumulators (8 heads x 16)   [256,512) S / P buffers,
// later the score accumulators.  The local policy runs before the first Q K^T and borrows columns: [128,192) partial
// (sum, g) of the four sequence quarters, later [pem | z]   [192,224) ol hi|lo   [256,256+4*KT) local softmax weights
// hi|lo per head   [448,512) vps accumulators
constexpr uint32_t TC_COL_Q = 0, TC_COL_O = 128, TC_COL_S = 256;
constexpr uint32_t TC_COL_PX = 128, TC_COL_D2 = 128, TC_COL_A2 = 192, TC_COL_A1 = 256, TC_COL_D1 = 448;
constexpr float TC_P_SCALE_LOG2 = 10.f;      // softmax weights are 2^(s - m + 10): keeps small weights out of fp16 subnormals

__host__ __device__ constexpr int tc_n2(int K1) { return (K1 + 4 + 15) & ~15; }      // columns of [pem | z]

// i-th word of w; 0 for i >= 4 (rollout_tc's key windows read one word past the last)
__device__ __forceinline__ uint32_t pick4(const uint32_t (&w)[4], int i) {
  return i == 0 ? w[0] : (i == 1 ? w[1] : (i == 2 ? w[2] : (i == 3 ? w[3] : 0u)));
}
// named barriers: the two key halves of a row (64 threads), one softmax group (256), one lane quadrant (128)
__device__ __forceinline__ void pair_sync(int id) { asm volatile("bar.sync %0, 64;" ::"r"(id) : "memory"); }
__device__ __forceinline__ void group_sync(int id) { asm volatile("bar.sync %0, 256;" ::"r"(id) : "memory"); }
__device__ __forceinline__ void quad_sync(int id) { asm volatile("bar.sync %0, 128;" ::"r"(id) : "memory"); }

// position (0..127) of the n-th (0-based) set bit of the 128-bit value r[3]:r[2]:r[1]:r[0]; n < popc(r)
__device__ __forceinline__ int select128(const uint32_t (&r)[4], int n) {
  const int c0 = __popc(r[0]), c1 = c0 + __popc(r[1]), c2 = c1 + __popc(r[2]);
  const int w = (n >= c0 ? 1 : 0) + (n >= c1 ? 1 : 0) + (n >= c2 ? 1 : 0);
  int m = n - (w == 0 ? 0 : (w == 1 ? c0 : (w == 2 ? c1 : c2)));
  uint32_t x = pick4(r, w);
  int pos = 0, t;
  t = __popc(x & 0xffffu); if (m >= t) { m -= t; pos = 16; x >>= 16; }
  t = __popc(x & 0xffu);   if (m >= t) { m -= t; pos += 8; x >>= 8; }
  t = __popc(x & 0xfu);    if (m >= t) { m -= t; pos += 4; x >>= 4; }
  t = __popc(x & 0x3u);    if (m >= t) { m -= t; pos += 2; x >>= 2; }
  t = (int)(x & 1u);       if (m >= t) pos += 1;
  return w * 32 + pos;
}

// D (+)= A B in split precision (x = hi + lo, fp16 each) over nks k-steps: lo*hi, hi*lo, then hi*hi into the one fp32
// accumulator.  The two small cross terms go first so that they are not lost against hi*hi (tests/test_umma_selftest.py).
// A in TMEM (k-step aStep columns), B in shared memory (k-step bStep bytes, leading byte offset lbo).
__device__ __forceinline__ void mma_split3(uint32_t d, uint32_t aHi, uint32_t aLo, uint32_t aStep, uint32_t bHi, uint32_t bLo,
                                           uint32_t bStep, uint32_t lbo, uint32_t idesc, int nks, bool acc) {
#pragma unroll
  for (int ks = 0; ks < nks; ++ks) umma::mma_f16_ts(d, aLo + aStep * ks, umma::make_desc(bHi + ks * bStep, lbo, 128), idesc, acc || ks > 0);
#pragma unroll
  for (int ks = 0; ks < nks; ++ks) umma::mma_f16_ts(d, aHi + aStep * ks, umma::make_desc(bLo + ks * bStep, lbo, 128), idesc, true);
#pragma unroll
  for (int ks = 0; ks < nks; ++ks) umma::mma_f16_ts(d, aHi + aStep * ks, umma::make_desc(bHi + ks * bStep, lbo, 128), idesc, true);
}

// Model constants of the local policy -> shared memory (layout L: TcL<KT> or StcL).  B operands in the tcgen05 layout
// written by elg_prepare_model: per head [hi | lo] of the first KT sequence positions out of KT_MAX; [PW | ZW] as built
// for this model's K1 (N2 = tc_n2(K1) columns).
template <class L, int KT>
__device__ __forceinline__ void stage_local_consts(float* w, const float* derived, int N2, int tid) {
  const float* loc = derived + DER_LOC;
  for (int i = tid; i < E; i += RT) w[L::wl + i] = derived[DER_WL + i];
  for (int i = tid; i < LH * 4; i += RT) w[L::u + i] = loc[LOC_U + i];
  for (int i = tid; i < LH * KT_MAX; i += RT) w[L::tt + i] = loc[LOC_T + i];
  for (int i = tid; i < LE * 4; i += RT) w[L::a + i] = (i & 3) == 3 ? loc[LOC_CV + (i >> 2)] : loc[LOC_A + i];
  for (int i = tid; i < KT_MAX; i += RT) w[L::pb + i] = loc[LOC_PB + i];
  for (int i = tid; i < 4; i += RT) w[L::zb + i] = loc[LOC_ZB + i];
  for (int i = tid; i < LH * KT * 16; i += RT) {            // 32-bit words: per head 2 x KT * 8
    const int h = i / (KT * 16), r = i % (KT * 16), part = r / (KT * 8), x = r % (KT * 8);
    w[L::op1 + i] = loc[LOC_OP1 + h * (KT_MAX * 16) + part * (KT_MAX * 8) + x];
  }
  for (int i = tid; i < N2 * LE; i += RT) w[L::op2 + i] = loc[LOC_OP2 + i];
}

// ---- local policy, steps (3)-(6) (CVRP/models.py:51-175, TSP/models.py:48-110), folded tables of elg_prepare_model ----
// Thread (row, wsub) owns the PT sequence positions [p0, p0 + PT) of its row's local sequence (KT positions, PT = KT / 4).
// The kernels find the neighbourhood and fill the features; the code below scores the positions, forms the softmax
// weights, runs both contractions on the tensor core and returns `penalty + local` per position.
template <int PT>
struct LocalSeq {
  float f0[PT], f1[PT], f2[PT];   // features: distance (scaled by the largest), polar angle, demand / load (cvrp)
  float cpen;                     // distance penalty = -f0 * cpen
  int p0, nv;                     // first position; positions s < nv exist
  bool dep_off;                   // position 0 is the depot, which is masked (the row stands on it)

  // head h's (u0, u1, u2) and table entries t[p0 + s]; a masked depot scores -inf
  __device__ __forceinline__ void load_head(const float* sU, const float* sT, int h, float4& u, float (&tq)[PT]) const {
    u = *reinterpret_cast<const float4*>(sU + h * 4);
#pragma unroll
    for (int i = 0; i < PT / 4; ++i) {
      const float4 t4 = *reinterpret_cast<const float4*>(sT + h * KT_MAX + p0 + 4 * i);
      tq[4 * i] = t4.x; tq[4 * i + 1] = t4.y; tq[4 * i + 2] = t4.z; tq[4 * i + 3] = t4.w;
    }
    if (dep_off) tq[0] = -INFINITY;
  }
  // score of position s (log2 domain, the constant query folded into u and t); -inf past the sequence
  __device__ __forceinline__ float score(const float4& u, const float (&tq)[PT], int s) const {
    const float v = fmaf(u.z, f2[s], fmaf(u.y, f1[s], fmaf(u.x, f0[s], tq[s])));
    return s < nv ? v : -INFINITY;
  }
};

// (3) this thread's maximum score per head; the kernel combines the four quarters of the row
template <int PT>
__device__ __forceinline__ void lp_head_max(const LocalSeq<PT>& ls, const float* sU, const float* sT, float (&m4)[LH]) {
#pragma unroll
  for (int h = 0; h < LH; ++h) {
    float4 u;
    float tq[PT];
    ls.load_head(sU, sT, h, u, tq);
    float m = -INFINITY;
#pragma unroll
    for (int s = 0; s < PT; ++s) m = fmaxf(m, ls.score(u, tq, s));
    m4[h] = m;
  }
}

// (4) weights 2^(s - max + 10) -> A operand of head h (TMEM, fp16 hi/lo, slot = sequence position); partial
//     (sum, sum w f) of my positions -> TMEM exchange columns
template <int PT, int KT>
__device__ __forceinline__ void lp_weights(const LocalSeq<PT>& ls, const float* sU, const float* sT, const float (&mh)[LH],
                                           uint32_t tl, int wsub) {
#pragma unroll
  for (int h = 0; h < LH; ++h) {
    const float moff = mh[h] == -INFINITY ? 0.f : mh[h] - TC_P_SCALE_LOG2;
    float sum = 0.f, g0 = 0.f, g1 = 0.f, g2 = 0.f;
    uint32_t hw[PT / 2], lw[PT / 2];
    float4 u;
    float tq[PT];
    ls.load_head(sU, sT, h, u, tq);
#pragma unroll
    for (int i = 0; i < PT / 2; ++i) {
      const float w0 = umma::ex2_raw(ls.score(u, tq, 2 * i) - moff);    // -inf (masked / beyond np) -> 0
      const float w1 = umma::ex2_raw(ls.score(u, tq, 2 * i + 1) - moff);
      sum += w0;
      g0 = fmaf(w0, ls.f0[2 * i], g0); g1 = fmaf(w0, ls.f1[2 * i], g1); g2 = fmaf(w0, ls.f2[2 * i], g2);
      sum += w1;
      g0 = fmaf(w1, ls.f0[2 * i + 1], g0); g1 = fmaf(w1, ls.f1[2 * i + 1], g1); g2 = fmaf(w1, ls.f2[2 * i + 1], g2);
      umma::split2_f16(w0, w1, hw[i], lw[i]);
    }
    const uint32_t ca = tl + TC_COL_A1 + h * KT + wsub * (PT / 2);
    static_assert(PT == 8 || PT == 12, "4 or 6 words of weights per thread and head");
    if constexpr (PT == 8) {
      umma::st4(ca, hw);
      umma::st4(ca + KT / 2, lw);
    } else {
      umma::st4(ca, hw); umma::st2(ca + 4, hw + 4);
      umma::st4(ca + KT / 2, lw); umma::st2(ca + KT / 2 + 4, lw + 4);
    }
    const uint32_t px[4] = {__float_as_uint(sum), __float_as_uint(g0), __float_as_uint(g1), __float_as_uint(g2)};
    umma::st4(tl + TC_COL_PX + 16 * wsub + 4 * h, px);
  }
}

// vps_h = W_h (Wv PE)_h, per head KT/16 k-steps (one thread issues)
template <int KT>
__device__ __forceinline__ void lp_issue_vps(uint32_t tm, uint32_t op1, uint32_t idescO) {
#pragma unroll
  for (int h = 0; h < LH; ++h) {
    const uint32_t aHi = tm + TC_COL_A1 + h * KT, bHi = op1 + h * (KT * 64);
    mma_split3(tm + TC_COL_D1 + 16 * h, aHi, aHi + KT / 2, 8, bHi, bHi + KT * 32, 512, 256, idescO, KT / 16, false);
  }
}

// (5) thread = (row, local head wsub): ol = (Wv We) g + Wv be + vps, normalised -> A operand of the second contraction
__device__ __forceinline__ void lp_ol(uint32_t tl, int wsub, const float* sA) {
  uint32_t dv[8], pq[16];
  umma::ld8_nw(tl + TC_COL_D1 + 16 * wsub, dv);
  umma::ld4_nw(tl + TC_COL_PX + 4 * wsub, pq);
  umma::ld4_nw(tl + TC_COL_PX + 16 + 4 * wsub, pq + 4);
  umma::ld4_nw(tl + TC_COL_PX + 32 + 4 * wsub, pq + 8);
  umma::ld4_nw(tl + TC_COL_PX + 48 + 4 * wsub, pq + 12);
  umma::wait_ld();
  const float sum = (umma::after_wait(pq[0]) + umma::after_wait(pq[4])) + (umma::after_wait(pq[8]) + umma::after_wait(pq[12]));
  const float inv_s = sum > 0.f ? 1.f / sum : 0.f;
  const float g0 = ((umma::after_wait(pq[1]) + umma::after_wait(pq[5])) + (umma::after_wait(pq[9]) + umma::after_wait(pq[13]))) * inv_s;
  const float g1 = ((umma::after_wait(pq[2]) + umma::after_wait(pq[6])) + (umma::after_wait(pq[10]) + umma::after_wait(pq[14]))) * inv_s;
  const float g2 = ((umma::after_wait(pq[3]) + umma::after_wait(pq[7])) + (umma::after_wait(pq[11]) + umma::after_wait(pq[15]))) * inv_s;
  float ol[LD];
#pragma unroll
  for (int c = 0; c < LD; ++c) {
    const float4 a4 = *reinterpret_cast<const float4*>(sA + (wsub * LD + c) * 4);
    ol[c] = fmaf(a4.z, g2, fmaf(a4.y, g1, a4.x * g0)) + a4.w + umma::after_wait(dv[c]) * inv_s;
  }
  uint32_t hw[4], lw[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) umma::split2_f16(ol[2 * i], ol[2 * i + 1], hw[i], lw[i]);
  umma::st4(tl + TC_COL_A2 + 4 * wsub, hw);
  umma::st4(tl + TC_COL_A2 + 16 + 4 * wsub, lw);
}

// [pem | z] = ol [PW | ZW], 2 k-steps (one thread issues); the accumulator takes over the exchange columns
__device__ __forceinline__ void lp_issue_pemz(uint32_t tm, uint32_t op2, int N2, uint32_t idescL2) {
  const uint32_t lbo2 = (uint32_t)N2 * 16u;
  mma_split3(tm + TC_COL_D2, tm + TC_COL_A2, tm + TC_COL_A2 + 16, 8, op2, op2 + (uint32_t)N2 * 64u, 2 * lbo2, lbo2, idescL2, 2, false);
}

// (6) penalty + local score of my positions: pen + f . z + z3 + pem[p] (tables carry the 1/sqrt(32));
//     store(s, p, value) for every position p = p0 + s < np of an active row
template <int PT, class Store>
__device__ __forceinline__ void lp_pen_local(const LocalSeq<PT>& ls, uint32_t tl, int K1, int np, bool act, const float* sZB,
                                             const float* sPB, Store store) {
  uint32_t dp[PT], dz[4];
  umma::ld8_nw(tl + TC_COL_D2 + ls.p0, dp);
  if constexpr (PT > 8) umma::ld4_nw(tl + TC_COL_D2 + ls.p0 + 8, dp + 8);
  umma::ld4_nw(tl + TC_COL_D2 + K1, dz);
  umma::wait_ld();
  if (act) {
    const float z0 = umma::after_wait(dz[0]) + sZB[0], z1 = umma::after_wait(dz[1]) + sZB[1];
    const float z2 = umma::after_wait(dz[2]) + sZB[2], c0 = umma::after_wait(dz[3]) + sZB[3];
#pragma unroll
    for (int s = 0; s < PT; ++s) {
      const int p = ls.p0 + s;
      if (p < np) {
        const float pem = umma::after_wait(dp[s]) + sPB[p];
        store(s, p, (fmaf(ls.f2[s], z2, fmaf(ls.f1[s], z1, ls.f0[s] * z0)) + c0 + pem) - ls.f0[s] * ls.cpen);
      }
    }
  }
}

// O (accumulated P V of heads 4 grp + 2 kh, + 1) / their denominators la, lb -> fp16 hi/lo O operand over the dead Q operand
__device__ __forceinline__ void store_o_operand(uint32_t tl, int grp, int kh, float la, float lb, bool act) {
  uint32_t orr[32], hw[16], lw[16];            // 32 consecutive accumulator columns
  umma::ld32_nw(tl + TC_COL_O + 16 * (4 * grp + 2 * kh), orr);
  umma::wait_ld();
#pragma unroll
  for (int i2 = 0; i2 < 2; ++i2) {
    const float inv_l = act ? 1.f / (i2 ? lb : la) : 0.f;
#pragma unroll
    for (int d2 = 0; d2 < 8; ++d2)
      umma::split2_f16(act ? umma::after_wait(orr[i2 * 16 + 2 * d2]) * inv_l : 0.f,
                       act ? umma::after_wait(orr[i2 * 16 + 2 * d2 + 1]) * inv_l : 0.f, hw[i2 * 8 + d2], lw[i2 * 8 + d2]);
  }
  umma::st16s<1>(tl + TC_COL_Q + 8 * (4 * grp + 2 * kh), hw);
  umma::st16s<1>(tl + TC_COL_Q + 64 + 8 * (4 * grp + 2 * kh), lw);
}

// Length of the tour segment i -> j: from the instance's unscaled coordinates rounded to an integer when the table has
// them (TSPLIB / CVRPLIB metric), else from the unit-square coordinates xy of the instance
__device__ __forceinline__ float seg_cost(const elg_tables& t, int b, int N1, const float* xy, int i, int j) {
  if (t.unscaled) {
    const float* ux = t.unscaled + (size_t)b * N1 * 2;
    return rintf(seglen(ux[2 * i] - ux[2 * j], ux[2 * i + 1] - ux[2 * j + 1]));
  }
  return seglen(xy[2 * i] - xy[2 * j], xy[2 * i + 1] - xy[2 * j + 1]);
}

// Optional per-phase cycle accounting (tools/phase_timing.py builds with -DELG_PHASE_TIMING; never in the shipped library)
#ifdef ELG_PHASE_TIMING
static __device__ unsigned long long g_phase_clk[16];   // one copy per translation unit
#define PHASE_T0() long long pt_ = clock64()
#define PHASE_MARK(i) do { if (threadIdx.x == 0) { const long long n_ = clock64(); pclk[i] += (unsigned long long)(n_ - pt_); pt_ = n_; } } while (0)
#else
#define PHASE_T0()
#define PHASE_MARK(i)
#endif


}  // namespace elg
