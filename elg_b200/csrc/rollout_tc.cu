// Tensor-core rollout kernel (resident instances, greedy decoding): the same per-step path as rollout.cu
// (reference file:line list there), with every dense contraction of the step on tcgen05 and every operand that
// changes per step living in TENSOR MEMORY (lane = POMO row):
//
//   global policy (CVRP/models.py:330-352, TSP/models.py:252-272)
//   S_h = Q_h K_h'^T        A = Q   (TMEM, written by tcgen05.st)      B = K' fp16 hi/lo (smem, resident)
//   O_h = P_h V_h           A = P_h (TMEM, written in place of S_h)    B = V^T fp16 hi/lo (smem, resident)
//   score = O E'^T          A = O   (TMEM)                             B = E' fp16 hi/lo (smem, resident)
//   local policy (CVRP/models.py:51-175, TSP/models.py:48-110), folded tables of elg_prepare_model
//   vps_h = W_h VPE_h       A = softmax weights of local head h over the <= 48 sequence positions (TMEM)
//                           B = (Wv PE(p)) of head h, 16 x KT (smem, model constant)
//   [pem | z] = ol [PW | ZW]  A = local attention output ol, 32 wide (TMEM)   B = (K1 + 4) x 32 (smem, model constant)
//
// Split precision (x = hi + lo, fp16 each) with the two small cross terms issued BEFORE hi*hi into the same fp32
// accumulator keeps every contraction fp32-grade (mma_split3 in rollout_common.cuh, tests/test_umma_selftest.py).
//
// CTA = one (aug-instance, tile of <= 112 POMO rows); TMEM lane = row.  16 warps: warp w owns TMEM lane quadrant
// q = w % 4 (rows 32q..32q+31) and sub-slot wsub = w / 4, so a row is served by four threads in four warps that
// exchange data through the row's TMEM lane or through shared memory + a 128-thread named barrier:
//   L        local policy, thread = (row, quarter wsub of the local sequence): rank-space validity bits of the
//            distance-presorted neighbour list, first-k walk by bit scans, features from the pair table; then the
//            local policy shared with rollout_stc.cu (rollout_common.cuh): 4-head scores + softmax weights -> TMEM A
//            operand, the two contractions on the tensor core, thread = (row, local head wsub) in between; results to
//            shared memory ordered by node id
//   softmax  two independent groups of 8 warps (grp = wsub / 2): group g walks heads 4g..4g+3 one at a time through
//            its own S/P buffer, its own mbarrier and a 256-thread named barrier, so one group's tensor-core / TMEM
//            latency is covered by the other group's arithmetic.  thread = (row, key half kh = wsub & 1); the two
//            halves of a row exchange (max, sum) through shared memory + a 64-thread named barrier
//   B3       thread = (row, quarter wsub of the node columns): clip*tanh(score + eb + {penalty+local | xi}) + mask,
//            first-max argmax combined across the 4 quarters through shared memory
//   C        env step: every thread of a row recomputes the scalar state, owns mask word wsub
//
// TMEM columns: the plan in rollout_common.cuh, with S / P buffers of 2 * N1p columns at [256, 256 + 2 * N1p)
#include <cstdlib>
#include "rollout_common.cuh"

namespace elg {

constexpr int TC_MT_MAX = 112;
constexpr int TC_XCH_FLOATS = 2 * 4 * 128 * 4;      // local-policy exchanges (validity words, neighbour bits), alias `add`

// Shared-memory layout in floats.  Every offset is a compile-time constant (sized for the largest resident instance:
// 112 node slots, 112 rows, KT local positions), so that shared-memory addresses are immediates instead of registers.
constexpr int TC_NP = 112;                  // node slots (N1 rounded up to 16, at most)
template <int KT>
struct TcL {
  static constexpr int MT = TC_MT_MAX;
  static constexpr int ops = 0;                                  // E' | K' | V^T slots, each fp16 hi + lo (TC_NP x 128 x 2 x 2 bytes)
  static constexpr int op1 = ops + 3 * TC_NP * 128;              // per local head: (Wv PE)_h^T, 16 x KT, fp16 hi + lo
  static constexpr int op2 = op1 + LH * KT * 16;                 // [PW | ZW], (K1 + 4 -> N2) x 32, fp16 hi + lo
  static constexpr int eb = op2 + tc_n2(KT) * LE;
  static constexpr int xy = eb + TC_NP;
  static constexpr int dem = xy + 2 * TC_NP;
  static constexpr int wl = dem + TC_NP;
  static constexpr int u = wl + E;
  static constexpr int tt = u + LH * 4;
  static constexpr int a = tt + LH * KT_MAX;                     // (Wv We)[c][0..2], (Wv be)[c]
  static constexpr int pb = a + LE * 4;
  static constexpr int zb = pb + KT_MAX;
  static constexpr int cur = zb + 4;
  static constexpr int first = cur + MT;
  static constexpr int load = first + MT;
  static constexpr int tlen = load + MT;
  static constexpr int fin = tlen + MT;
  static constexpr int mask = fin + MT;                           // word-major [4][128]: bank = row % 32 whatever the word
  static constexpr int vis = mask + 4 * 128;                     // two copies: a step reads one and writes the other
  static constexpr int add = vis + 2 * MT * 4;                       // penalty + local of each row's neighbours (stride KT), ordered by node id
  static constexpr int nb = add + (MT * KT > TC_XCH_FLOATS ? MT * KT : TC_XCH_FLOATS);   // neighbour bit mask per row
  static constexpr int xch = nb + MT * 4;                        // softmax (max, sum) exchange; later the 4 argmax candidates per row
  static constexpr int ctrl = xch + 2 * 4 * 128;
  static constexpr int bar = ctrl + 4;                           // 5 mbarriers + TMEM base address
  static constexpr int total = bar + 12;
};
static_assert(TcL<48>::total * 4 <= 227 * 1024 && TcL<32>::total * 4 <= 227 * 1024, "layout exceeds one SM's shared memory");

#ifdef ELG_PHASE_TIMING
// The softmax rounds split per group: each group's leader accumulates five sub-phases of its own rounds and counts them
// (slot 5), so the two groups' waits can be told apart from their arithmetic (tools/phase_timing.py)
static __device__ unsigned long long g_sm_clk[2][8];
__device__ __forceinline__ unsigned int sm_clock() {
  unsigned int c;
  asm volatile("mov.u32 %0, %%clock;" : "=r"(c)::"memory");
  return c;
}
#define SM_T0() unsigned int sclk_ = sm_clock()
#define SM_MARK(i) do { if (leader) { const unsigned int n_ = sm_clock(); smclk[i] += n_ - sclk_; sclk_ = n_; } } while (0)
#else
#define SM_T0()
#define SM_MARK(i)
#endif

// =================================================================================================
// NP = 112: the node count rounded up to 16 is known at compile time (the 100-node benchmark shapes); NP = 0: run time
template <int PROBLEM, int MAXE, int NP>
__global__ void __launch_bounds__(RT, 1) rollout_tc_kernel(const RolloutArgs A) {
  constexpr bool CVRP = PROBLEM == ELG_CVRP;
  constexpr int DEP = CVRP ? 1 : 0;
  extern __shared__ __align__(128) float sm[];
  const int N1 = A.N1;
  const int N1p = NP ? NP : ((N1 + 15) & ~15);
  const int W = (N1 + 31) >> 5;
  constexpr int KT = MAXE * 8;
  const int K1 = A.k_local + DEP;
  using L = TcL<MAXE * 8>;
  const float* sEb = sm + L::eb;
  const float* sXY = sm + L::xy;
  const float* sDem = sm + L::dem;
  const float* sWL = sm + L::wl;
  const float* sU = sm + L::u;
  const float* sT = sm + L::tt;
  const float* sA = sm + L::a;
  const float* sPB = sm + L::pb;
  const float* sZB = sm + L::zb;
  int* sCur = reinterpret_cast<int*>(sm + L::cur);
  int* sFirst = reinterpret_cast<int*>(sm + L::first);
  float* sLoad = sm + L::load;
  float* sTlen = sm + L::tlen;
  int* sFin = reinterpret_cast<int*>(sm + L::fin);
  uint32_t* sMask = reinterpret_cast<uint32_t*>(sm + L::mask);
  uint32_t* sVis = reinterpret_cast<uint32_t*>(sm + L::vis);
  float* sAdd = sm + L::add;
  uint32_t* sNb = reinterpret_cast<uint32_t*>(sm + L::nb);
  float* sXm = sm + L::xch;              // [4][128]
  float* sXl = sm + L::xch + 512;        // [4][128]
  int* sCtrl = reinterpret_cast<int*>(sm + L::ctrl);
  uint64_t* bar = reinterpret_cast<uint64_t*>(sm + L::bar);      // TMA completion
  uint64_t* bar_sc = bar + 1;                                     // tcgen05.commit of the score MMA
  uint64_t* bar_loc = bar + 4;                                    // tcgen05.commit of the local-policy MMAs
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bar + 5);

  // the warp index through a shuffle: the compiler then knows it is warp-uniform and keeps everything derived from it
  // (softmax group, TMEM addresses, MMA operands) in uniform registers, so the leader issues each tcgen05.mma without
  // first moving its operands into uniform registers (R2UR) on the chain of every decode step
  const int tid = threadIdx.x, warp = __shfl_sync(FULL, tid >> 5, 0), lane = tid & 31;
  const int q = warp & 3, wsub = warp >> 2, grp = wsub >> 1, kh = wsub & 1;     // softmax group (heads 4*grp..), key half
  uint64_t* bar_grp = bar + 2 + grp;                              // tcgen05.commit of this softmax group's MMAs
  const int row = q * 32 + lane;                   // TMEM lane = row of the tile
  const int rc = row < A.MT ? row : 0;             // clamped index into the per-row state arrays
  const int KH = N1p >> 1, CQ = N1p >> 2;          // keys per softmax thread, node columns per B3 thread

  {
    stage_local_consts<L, KT>(sm, A.derived, tc_n2(K1), tid);
    if (tid == 0) {
      mbar_init(bar, 1);
      mbar_init(bar + 1, 1);
      mbar_init(bar + 2, 1);
      mbar_init(bar + 3, 1);
      mbar_init(bar + 4, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) umma::tmem_alloc(tmem_ptr, 512);
    umma::fence_async_smem();
    umma::fence_before_sync();
  }
  __syncthreads();
  umma::fence_after_sync();
  const uint32_t tm = *tmem_ptr;
  const uint32_t tl = tm + ((uint32_t)(q * 32) << 16);          // this warp's lane quadrant

  // tensor-core operand addresses (shared memory) and instruction descriptors
  const uint32_t seg = (uint32_t)N1p * 512u;                    // bytes of one operand (hi + lo)
  const uint32_t half = (uint32_t)N1p * 256u;
  constexpr uint32_t slot = TC_NP * 512u;                      // bytes of one operand slot
  const uint32_t opE = umma::smem_addr(sm + L::ops), opK = opE + slot, opV = opK + slot;
  const uint32_t lboN = (uint32_t)N1p * 16u;                    // K' / E': N1p rows per 8-column chunk
  const uint32_t idescS = umma::make_idesc_f16(128, N1p), idescO = umma::make_idesc_f16(128, 16);
  const int nks = N1p >> 4;
  // local policy: thread (row, wsub) owns sequence positions [wsub * PT, wsub * PT + PT)
  constexpr int PT = MAXE * 2;
  const int N2 = tc_n2(K1);
  const uint32_t op1 = umma::smem_addr(sm + L::op1), op2 = umma::smem_addr(sm + L::op2);
  const uint32_t idescL2 = umma::make_idesc_f16(128, N2);

  const int total_work = A.B * A.tiles;
  // mbarrier parities: bar_loc completes twice per decode step (always 0, then 1), bar_sc once and each bar_grp five
  // times (four rounds + the accumulated O), so both follow the parity of the number of decode steps done so far
  uint32_t bar_phase = 0, step_par = 0;
  const bool leader = tid == grp * 256;                           // issues this group's MMAs
#ifdef ELG_PHASE_TIMING
  unsigned long long pclk[16] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
  unsigned int smclk[6] = {0, 0, 0, 0, 0, 0};
#endif

  for (int iter = 0;; ++iter) {
    int work;
    if (A.work_counter) {
      if (tid == 0) sCtrl[0] = atomicAdd(A.work_counter, 1);
      __syncthreads();
      work = sCtrl[0];
    } else {
      work = blockIdx.x + iter * gridDim.x;
    }
    if (work >= total_work) break;
    const int b = work / A.tiles, tile = work % A.tiles;
    const int row0 = tile * A.MT;
    const int nrows = min(A.MT, A.M - row0);

    // ---- the instance's operands: one TMA bulk copy per operand, resident for the whole rollout ----------
    if (tid == 0) {
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      mbar_expect_tx(bar, 3 * seg);
      const uint8_t* src = reinterpret_cast<const uint8_t*>(A.t.e) + (size_t)b * 3 * seg;
      uint8_t* dst = reinterpret_cast<uint8_t*>(sm + L::ops);
      bulk_g2s(dst, src, seg, bar);
      bulk_g2s(dst + slot, src + seg, seg, bar);
      bulk_g2s(dst + 2 * slot, src + 2 * seg, seg, bar);
    }
    for (int i = tid; i < N1p; i += RT) {
      const bool ok = i < N1;
      (sm + L::eb)[i] = ok ? A.t.eb[(size_t)b * N1 + i] : 0.f;
      (sm + L::xy)[2 * i] = ok ? A.t.xy[((size_t)b * N1 + i) * 2] : 0.f;
      (sm + L::xy)[2 * i + 1] = ok ? A.t.xy[((size_t)b * N1 + i) * 2 + 1] : 0.f;
      (sm + L::dem)[i] = (CVRP && ok) ? A.t.demand[(size_t)b * N1 + i] : 0.f;
    }
    for (int r = tid; r < A.MT; r += RT) {
      const size_t g = (size_t)b * A.M + row0 + r;
      const bool ok = r < nrows;
      if (A.single_step && ok) {
        sCur[r] = A.st_cur[g];
        sFirst[r] = CVRP ? 0 : A.st_first[g];
        sLoad[r] = CVRP ? A.st_load[g] : 1.f;
        sFin[r] = 0;
      } else {
        sCur[r] = 0; sFirst[r] = 0; sLoad[r] = 1.f;
        sFin[r] = ok ? 0 : 1;
      }
      sTlen[r] = 0.f;
    }
    for (int i = tid; i < A.MT * 4; i += RT) {
      const int r = i >> 2, w = i & 3;
      sVis[i] = 0u;
      sVis[TC_MT_MAX * 4 + i] = 0u;
      sMask[w * 128 + r] = (A.single_step && r < nrows && w < W) ? A.st_mask[((size_t)b * A.M + row0 + r) * W + w] : 0u;
    }
    mbar_wait(bar, bar_phase);
    bar_phase ^= 1;
    __syncthreads();

    const bool in_tile = row < nrows;
    // Start of a decode step: the row's two 16-byte chunks of the neighbour list of `cur` and its query row are fetched
    // together; the Q operand  q = Wq_last [enc[cur]; load] (cvrp) / q_first + Wq_last enc[cur] (tsp), fp16 hi/lo -> TMEM,
    // is finished after the list has been tested (tcgen05.st is warp-collective: every lane stores, dead rows zeros)
    uint4 preLa = make_uint4(0, 0, 0, 0), preLb = make_uint4(0, 0, 0, 0);
    auto prefetch_step = [&](float4 (&qv)[2 * D / 4], int cur, int first, bool live) {
      preLa = preLb = make_uint4(0, 0, 0, 0);
#pragma unroll
      for (int d4 = 0; d4 < 2 * D / 4; ++d4) qv[d4] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (live) {
        const uint4* lp = reinterpret_cast<const uint4*>(reinterpret_cast<const uint8_t*>(A.t.nbr) + ((size_t)b * N1 + cur) * ELG_NBR_NODE_BYTES(N1));
        preLa = __ldg(lp + 2 * wsub);
        preLb = __ldg(lp + 2 * wsub + 1);
        const float4* qp = reinterpret_cast<const float4*>(A.t.qtab + ((size_t)b * N1 + cur) * E + 2 * wsub * D);
#pragma unroll
        for (int d4 = 0; d4 < 2 * D / 4; ++d4) qv[d4] = __ldg(qp + d4);
        if (!CVRP) {
          const float4* fp = reinterpret_cast<const float4*>(A.t.qfirst + ((size_t)b * N1 + first) * E + 2 * wsub * D);
#pragma unroll
          for (int d4 = 0; d4 < 2 * D / 4; ++d4) {
            const float4 f4 = __ldg(fp + d4);
            qv[d4].x = f4.x + qv[d4].x; qv[d4].y = f4.y + qv[d4].y; qv[d4].z = f4.z + qv[d4].z; qv[d4].w = f4.w + qv[d4].w;
          }
        }
      }
    };
    auto finish_step = [&](const float4 (&qv)[2 * D / 4], float ld, bool live) {
      uint32_t hw[16], lw[16];
      if (live) {
#pragma unroll
        for (int d4 = 0; d4 < 2 * D / 4; ++d4) {
          float4 v4 = qv[d4];
          if (CVRP) {
            const float4 wl = *reinterpret_cast<const float4*>(sWL + 2 * wsub * D + d4 * 4);
            v4.x = fmaf(ld, wl.x, v4.x); v4.y = fmaf(ld, wl.y, v4.y);
            v4.z = fmaf(ld, wl.z, v4.z); v4.w = fmaf(ld, wl.w, v4.w);
          }
          umma::split2_f16(v4.x, v4.y, hw[d4 * 2], lw[d4 * 2]);
          umma::split2_f16(v4.z, v4.w, hw[d4 * 2 + 1], lw[d4 * 2 + 1]);
        }
      } else {
#pragma unroll
        for (int i = 0; i < 16; ++i) hw[i] = lw[i] = 0u;
      }
      umma::st16s<1>(tl + TC_COL_Q + 16 * wsub, hw);
      umma::st16s<1>(tl + TC_COL_Q + 64 + 16 * wsub, lw);
    };
    int t = 0;
    for (;; ++t) {
      const bool forced = !A.single_step && (t < 1 + DEP);
      PHASE_T0();
      // row state at the start of the step (registers: phase C of this step overwrites the shared copies)
      const int cur0 = sCur[rc];
      const float ld0 = sLoad[rc];
      const bool act = in_tile && !sFin[rc];

      if (!forced) {
        uint32_t mw[4];
        {
          mw[0] = sMask[rc]; mw[1] = sMask[128 + rc]; mw[2] = sMask[256 + rc]; mw[3] = sMask[384 + rc];
        }
        float4 qv[2 * D / 4];                        // heads 2*wsub, 2*wsub + 1 of the query row: 32 consecutive k
        prefetch_step(qv, cur0, CVRP ? 0 : sFirst[rc], act);       // global loads in flight while the list is tested
        // =================== L: local policy (CVRP/models.py:51-175, TSP/models.py:48-110) ======================
        // (1) validity of the distance-presorted neighbour list of `cur` in RANK space: this thread tests the 32
        //     list entries of its two 16-byte chunks (entry e = s + 8 i sits at byte i of chunk s, nbr_pos()); the
        //     four quarters are OR-ed through shared memory
        const uint8_t* nrow = reinterpret_cast<const uint8_t*>(A.t.nbr) + ((size_t)b * N1 + cur0) * ELG_NBR_NODE_BYTES(N1);
        uint32_t R[4];
        {
          uint32_t rp[4] = {0u, 0u, 0u, 0u};
          if (act) {
            const uint32_t lw2[2][4] = {{preLa.x, preLa.y, preLa.z, preLa.w}, {preLb.x, preLb.y, preLb.z, preLb.w}};
#pragma unroll
            for (int c = 0; c < 2; ++c)
#pragma unroll
              for (int i = 0; i < 16; ++i) {
                const uint32_t id = (lw2[c][i >> 2] >> ((i & 3) * 8)) & 0xffu;
                const uint32_t free1 = ~__funnelshift_r(sMask[(id >> 5) * 128 + rc], 0u, id) & 1u;      // conflict-free: bank = row % 32
                rp[i >> 2] |= free1 << ((i & 3) * 8 + c);
              }
          }
          uint4* xr = reinterpret_cast<uint4*>(sAdd);                     // [4][128] exchange (aliases the dead `add` rows)
          xr[wsub * 128 + row] = make_uint4(rp[0] << (2 * wsub), rp[1] << (2 * wsub), rp[2] << (2 * wsub), rp[3] << (2 * wsub));
          quad_sync(11 + q);
          const uint4 x0 = xr[row], x1 = xr[128 + row], x2 = xr[256 + row], x3 = xr[384 + row];
          R[0] = x0.x | x1.x | x2.x | x3.x; R[1] = x0.y | x1.y | x2.y | x3.y;
          R[2] = x0.z | x1.z | x2.z | x3.z; R[3] = x0.w | x1.w | x2.w | x3.w;
          const int NLs = N1 - DEP;                                        // list entries; the padding holds id 0
#pragma unroll
          for (int w = 0; w < 4; ++w) {
            const int nb = NLs - w * 32;
            R[w] &= nb >= 32 ? FULL : (nb > 0 ? ((1u << nb) - 1u) : 0u);
          }
        }
        finish_step(qv, ld0, act);
        PHASE_MARK(0);
        const bool depot_masked = (mw[0] & 1u) != 0u;
        // (2) the first kk = min(k, #valid) set bits are the local neighbourhood, in rank order; with the depot in
        //     front (cvrp) they are sequence positions p = 0 .. np-1; this thread owns p in [wsub PT, wsub PT + PT)
        const int kk = min(__popc(R[0]) + __popc(R[1]) + __popc(R[2]) + __popc(R[3]), A.k_local);
        const int np = act ? kk + DEP : 0;
        const int p0 = wsub * PT;
        const float4* rec = reinterpret_cast<const float4*>(nrow + ELG_NBR_STRIDE + ELG_NBR_PAIR_BYTES(N1));   // by list rank
        LocalSeq<PT> ls;
        ls.p0 = p0;
        ls.cpen = 1.f;
        uint32_t idw[PT / 4];                                             // this thread's node ids, 4 per word
        uint32_t nbp[4] = {0u, 0u, 0u, 0u};                               // their bits in node space
        {
          // list positions of my neighbours: skip to the first one with a rank select, then walk the set bits
          int epos[PT];
          unsigned long long ra = 0ull, rb = 0ull;
          const int cfirst = max(p0 - DEP, 0);                            // rank of my first neighbour among the valid ones
          if (cfirst < kk) {
            const int e0 = select128(R, cfirst);
            ra = ((unsigned long long)R[1] << 32) | R[0];
            rb = ((unsigned long long)R[3] << 32) | R[2];
            if (e0 < 64) { ra &= ~0ull << e0; } else { ra = 0ull; rb &= ~0ull << (e0 - 64); }
          }
#pragma unroll
          for (int s = 0; s < PT; ++s) {
            epos[s] = 0;
            if (DEP && s == 0 && wsub == 0) continue;                     // the depot: features (0, 0, 0), node 0
            const bool in_a = ra != 0ull;
            const unsigned long long x = in_a ? ra : rb;
            epos[s] = max(__ffsll((long long)x) - 1, 0) + (in_a ? 0 : 64);
            const unsigned long long y = x & (x - 1ull);
            ra = in_a ? y : ra;
            rb = in_a ? rb : y;
          }
          // one 16-byte record per neighbour: (distance, angle, demand, node id); the largest distance is the last one's
          float4 rv[PT];
          float4 rlast = make_float4(0.f, 0.f, 0.f, 0.f);
          if (kk > 0) rlast = __ldg(rec + select128(R, kk - 1));
#pragma unroll
          for (int s = 0; s < PT; ++s) {
            const bool mine = (p0 + s) < np && !(DEP && s == 0 && wsub == 0);
            rv[s] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (mine) rv[s] = __ldg(rec + epos[s]);
          }
          const float dmax = rlast.x;
          const float r0d = dmax != 0.f ? 1.f / (dmax + 1e-6f) : 1.f;      // cvrp: cur_dist / (max + 1e-6); dmax == 0 -> dd itself
          // penalty -d / dmax (no eps, CVRP/models.py:380,403) = -f0 (dmax + 1e-6) / dmax; tsp: -d / (dmax + 1e-6) = -f0
          if (CVRP && dmax != 0.f) ls.cpen = (dmax + 1e-6f) / dmax;
          const float rtsp = 1.f / (dmax + 1e-6f);
          const float rld = 1.f / ld0;
#pragma unroll
          for (int i = 0; i < PT / 4; ++i) idw[i] = 0u;
          unsigned long long na = 0ull, nb2 = 0ull;
#pragma unroll
          for (int s = 0; s < PT; ++s) {
            const bool mine = (p0 + s) < np && !(DEP && s == 0 && wsub == 0);
            ls.f0[s] = ls.f1[s] = ls.f2[s] = 0.f;
            if (mine) {
              const int nd = __float_as_int(rv[s].w);
              idw[s >> 2] |= (uint32_t)nd << ((s & 3) * 8);
              if (CVRP) {
                ls.f0[s] = rv[s].x * r0d;
                ls.f2[s] = rv[s].z * rld;
              } else {
                ls.f0[s] = rv[s].x * rtsp;
              }
              ls.f1[s] = rv[s].y;
              const unsigned long long bit = 1ull << (nd & 63);
              na |= (nd & 64) ? 0ull : bit;
              nb2 |= (nd & 64) ? bit : 0ull;
            }
          }
          if (DEP && wsub == 0 && np > 0) na |= 1ull;                     // the depot heads the local sequence
          nbp[0] = (uint32_t)na; nbp[1] = (uint32_t)(na >> 32); nbp[2] = (uint32_t)nb2; nbp[3] = (uint32_t)(nb2 >> 32);
        }
        PHASE_MARK(1);
        // (3) scores of the constant local query, all four heads for my positions (log2 domain); the row's maximum
        //     per head and the neighbour bits of the row come from the four quarters through shared memory
        ls.nv = np - p0;
        ls.dep_off = DEP && wsub == 0 && depot_masked;
        float mh[LH];
        {
          uint32_t nbw[4];                                                // neighbour bit mask of the row (node space)
          // the maxima only serve as a common offset: rounded UP to fp16 they fit 8 bytes per thread (softmax exchange area)
          uint32_t mp[2];
          {
            float m4[LH];
            lp_head_max(ls, sU, sT, m4);
            mp[0] = umma::pack_h2(__float2half_ru(m4[0]), __float2half_ru(m4[1]));
            mp[1] = umma::pack_h2(__float2half_ru(m4[2]), __float2half_ru(m4[3]));
          }
          uint2* xm = reinterpret_cast<uint2*>(sXm);                      // [4][128]
          uint4* xn = reinterpret_cast<uint4*>(sAdd) + 512;               // [4][128], behind the validity exchange
          xm[wsub * 128 + row] = make_uint2(mp[0], mp[1]);
          xn[wsub * 128 + row] = make_uint4(nbp[0], nbp[1], nbp[2], nbp[3]);
          quad_sync(11 + q);
          {
            const uint2 a0 = xm[row], a1 = xm[128 + row], a2 = xm[256 + row], a3 = xm[384 + row];
            const __half2 h01 = __hmax2(__hmax2(*reinterpret_cast<const __half2*>(&a0.x), *reinterpret_cast<const __half2*>(&a1.x)),
                                        __hmax2(*reinterpret_cast<const __half2*>(&a2.x), *reinterpret_cast<const __half2*>(&a3.x)));
            const __half2 h23 = __hmax2(__hmax2(*reinterpret_cast<const __half2*>(&a0.y), *reinterpret_cast<const __half2*>(&a1.y)),
                                        __hmax2(*reinterpret_cast<const __half2*>(&a2.y), *reinterpret_cast<const __half2*>(&a3.y)));
            const float2 f01 = __half22float2(h01), f23 = __half22float2(h23);
            mh[0] = f01.x; mh[1] = f01.y; mh[2] = f23.x; mh[3] = f23.y;
            const uint4 n0 = xn[row], n1 = xn[128 + row], n2 = xn[256 + row], n3 = xn[384 + row];
            nbw[0] = (n0.x | n1.x) | (n2.x | n3.x); nbw[1] = (n0.y | n1.y) | (n2.y | n3.y);
            nbw[2] = (n0.z | n1.z) | (n2.z | n3.z); nbw[3] = (n0.w | n1.w) | (n2.w | n3.w);
          }
          if (wsub == 0 && act) *reinterpret_cast<uint4*>(sNb + rc * 4) = make_uint4(nbw[0], nbw[1], nbw[2], nbw[3]);   // read back in (6) and B3
        }
        PHASE_MARK(2);
        // (4) softmax weights -> TMEM, then the vps contraction
        lp_weights<PT, KT>(ls, sU, sT, mh, tl, wsub);
        umma::wait_st();                                                   // also the Q operand
        umma::fence_before_sync();
        __syncthreads();
        if (tid == 0) {
          umma::fence_after_sync();
          lp_issue_vps<KT>(tm, op1, idescO);
          umma::commit(bar_loc);
        }
        PHASE_MARK(3);
        // (5) ol -> A operand of the second contraction
        mbar_wait(bar_loc, 0u);
        umma::fence_after_sync();
        lp_ol(tl, wsub, sA);
        umma::wait_st();
        umma::fence_before_sync();
        __syncthreads();

        // MMA issue helpers (leaders only)
        auto issue_qk = [&](int head) {
          const uint32_t aHi = tm + TC_COL_Q + 8 * head, bHi = opK + head * 2 * lboN;
          mma_split3(tm + TC_COL_S + grp * N1p, aHi, aHi + 64, 0, bHi, bHi + half, 0, lboN, idescS, 1, false);
        };
        auto issue_pv = [&](int head) {
          const uint32_t pHi = tm + TC_COL_S + grp * N1p, vHi = opV + head * (N1p * 32);
          mma_split3(tm + TC_COL_O + 16 * head, pHi, pHi + (N1p >> 1), 8, vHi, vHi + half, 512, 256, idescO, nks, false);
        };
        if (leader) {
          umma::fence_after_sync();
          if (tid == 0) {
            lp_issue_pemz(tm, op2, N2, idescL2);
            umma::commit(bar_loc);
          }
          issue_qk(4 * grp);
          umma::commit(bar_grp);
        }
        PHASE_MARK(4);
        // (6) penalty + local score of my positions, stored ordered by node id for phase B3 (runs while the tensor core
        //     works on the first Q K^T)
        mbar_wait(bar_loc, 1u);
        umma::fence_after_sync();
        {
          const uint4 n4 = *reinterpret_cast<const uint4*>(sNb + rc * 4);
          const uint32_t nbw[4] = {n4.x, n4.y, n4.z, n4.w};
          const int pc1 = __popc(nbw[0]), pc2 = pc1 + __popc(nbw[1]), pc3 = pc2 + __popc(nbw[2]);
          lp_pen_local(ls, tl, K1, np, act, sZB, sPB, [&](int s, int, float v) {
            const int nd = (idw[s >> 2] >> ((s & 3) * 8)) & 0xff, wd = nd >> 5;
            const uint32_t below = pick4(nbw, wd) & ((1u << (nd & 31)) - 1u);
            const int rank = (wd == 0 ? 0 : (wd == 1 ? pc1 : (wd == 2 ? pc2 : pc3))) + __popc(below);
            sAdd[rc * KT + rank] = v;
          });
        }
        PHASE_MARK(5);

        // ---- valid-key bits of this row (unmasked and < N1); this thread's window: keys [kh*KH, kh*KH + KH) ----
        uint32_t inv[4];
        {
          const uint32_t mq[4] = {sMask[rc], sMask[128 + rc], sMask[256 + rc], sMask[384 + rc]};
#pragma unroll
          for (int w = 0; w < 4; ++w) {
            const int nb = N1 - w * 32;
            const uint32_t lim = nb >= 32 ? FULL : (nb > 0 ? ((1u << nb) - 1u) : 0u);
            inv[w] = act ? (~mq[w] & lim) : 0u;
          }
        }
        uint32_t v0, v1;
        {
          const int s0 = kh * KH, wd = s0 >> 5, sh = s0 & 31;
          v0 = __funnelshift_r(pick4(inv, wd), pick4(inv, wd + 1), sh);
          v1 = __funnelshift_r(pick4(inv, wd + 1), pick4(inv, wd + 2), sh);
        }
        float lt0 = 0.f, lt1 = 0.f, lt2 = 0.f, lt3 = 0.f;       // softmax denominators of heads 4*grp + rho

        SM_T0();
#pragma unroll 1
        for (int rho = 0; rho < 4; ++rho) {
          mbar_wait(bar_grp, (step_par + rho) & 1u);
          umma::fence_after_sync();
          SM_MARK(0);
          const uint32_t sb = tl + TC_COL_S + grp * N1p;
          uint32_t sr[56];
          // KH = 8..56 columns in at most three loads (32 + 16 + 8, register i <-> column i); columns past KH that the
          // fixed shapes drag along lie inside the allocation and are never used
          {
            const uint32_t s0 = sb + kh * KH;
            umma::ld32_nw(s0, sr);
            if (KH > 32) umma::ld16_nw(s0 + 32, sr + 32);
            if (KH > 48) umma::ld8_nw(s0 + 48, sr + 48);
          }
          umma::wait_ld();
          float mloc = -INFINITY;
#pragma unroll
          for (int c8 = 0; c8 < 7; ++c8)
            if (c8 * 8 < KH) {
#pragma unroll
              for (int i = c8 * 8; i < c8 * 8 + 8; ++i) {
                const bool valid = ((i < 32 ? (v0 >> i) : (v1 >> (i - 32))) & 1u) != 0u;
                const float s = valid ? umma::after_wait(sr[i]) : -INFINITY;
                sr[i] = __float_as_uint(s);
                mloc = fmaxf(mloc, s);
              }
            }
          // the row's maximum over both key halves first (shared memory + 64-thread barrier): both halves then use the same
          // offset, no rescaling of the weights; the two partial denominators meet at the normalisation of O
          sXm[wsub * 128 + row] = mloc;
          SM_MARK(1);
          pair_sync(1 + grp * 4 + q);
          const float mm = fmaxf(mloc, sXm[(wsub ^ 1) * 128 + row]);
          const float moff = mm == -INFINITY ? 0.f : mm - TC_P_SCALE_LOG2;
          SM_MARK(2);
          float lloc = 0.f;
          // P (fp16 hi/lo, two keys per 32-bit column) in place of S: hi at [sb, sb + N1p/2), lo behind it
#pragma unroll
          for (int c8 = 0; c8 < 7; ++c8)
            if (c8 * 8 < KH) {
#pragma unroll
              for (int i = c8 * 4; i < c8 * 4 + 4; ++i) {       // keys (2i, 2i+1) -> hi word in sr[2i], lo word in sr[2i+1]
                const float pa = umma::ex2_raw(__uint_as_float(sr[2 * i]) - moff);
                const float pb = umma::ex2_raw(__uint_as_float(sr[2 * i + 1]) - moff);
                lloc += pa + pb;
                uint32_t hwd, lwd;
                umma::split2_f16(pa, pb, hwd, lwd);
                sr[2 * i] = hwd;
                sr[2 * i + 1] = lwd;
              }
            }
          if (rho == 0) lt0 = lloc; else if (rho == 1) lt1 = lloc; else if (rho == 2) lt2 = lloc; else lt3 = lloc;
          umma::st_words<2>(sb + kh * (KH >> 1), sr, KH >> 1);
          umma::st_words<2>(sb + (N1p >> 1) + kh * (KH >> 1), sr + 1, KH >> 1);
          umma::wait_st();
          umma::fence_before_sync();
          SM_MARK(3);
          // round 0 is CTA-wide: the first P V overwrites accumulator columns that held [pem | z], which the other
          // group's threads may still be reading in (6)
          if (rho == 0) __syncthreads(); else group_sync(9 + grp);
          if (leader) {
            umma::fence_after_sync();
            issue_pv(4 * grp + rho);
            if (rho < 3) issue_qk(4 * grp + rho + 1);
            umma::commit(bar_grp);
          }
          SM_MARK(4);
#ifdef ELG_PHASE_TIMING
          smclk[5] += 1;
#endif
          PHASE_MARK(6);

        }

        // ---- O = P V accumulated: normalise, fp16 hi/lo -> O operand (TMEM, over the dead Q operand) ------------
        mbar_wait(bar_grp, step_par);
        umma::fence_after_sync();
        {
          // this thread normalises heads 4*grp + 2*kh, + 1 and needs the other key half's denominators of those two heads;
          // it publishes its own partial denominators of the two heads the partner normalises
          sXm[wsub * 128 + row] = kh ? lt0 : lt2;
          sXl[wsub * 128 + row] = kh ? lt1 : lt3;
          pair_sync(1 + grp * 4 + q);
          const float la = (kh ? lt2 : lt0) + sXm[(wsub ^ 1) * 128 + row];
          const float lb = (kh ? lt3 : lt1) + sXl[(wsub ^ 1) * 128 + row];
          store_o_operand(tl, grp, kh, la, lb, act);
          umma::wait_st();
          umma::fence_before_sync();
        }
        __syncthreads();
        if (tid == 0) {
          // scores = O E'^T (the reference's single-head matmul(mh_atten_out, single_head_key), Wo folded into E')
          umma::fence_after_sync();
          mma_split3(tm + TC_COL_S, tm + TC_COL_Q, tm + TC_COL_Q + 64, 8, opE, opE + half, 2 * lboN, lboN, idescS, 8, false);
          umma::commit(bar_sc);
        }
        PHASE_MARK(7);

        // ---- B3: logits of this thread's node columns [wsub*CQ, wsub*CQ + CQ) -----------------------------------
        mbar_wait(bar_sc, step_par);
        step_par ^= 1u;
        umma::fence_after_sync();
        PHASE_MARK(8);
        {
          uint32_t xr[28];
          const int c0n = wsub * CQ;
          {
            const uint32_t s0 = tl + TC_COL_S + c0n;
            umma::ld16_nw(s0, xr);
            if (CQ > 16) umma::ld8_nw(s0 + 16, xr + 16);
            if (CQ > 24) umma::ld4_nw(s0 + 24, xr + 24);
          }
          umma::wait_ld();
          float best = -INFINITY;
          int bidx = 0x7fffffff;
          bool need_all = false;
          if (act) {
            const uint4 n4 = *reinterpret_cast<const uint4*>(sNb + rc * 4);
            const uint32_t nbw[4] = {n4.x, n4.y, n4.z, n4.w};
            const int wd = c0n >> 5, sh = c0n & 31;
            const uint32_t vwin = __funnelshift_r(pick4(inv, wd), pick4(inv, wd + 1), sh);      // unmasked & < N1
            const uint32_t nwin = __funnelshift_r(pick4(nbw, wd), pick4(nbw, wd + 1), sh);      // neighbour (or depot)
            int rbase = __popc(pick4(nbw, wd) & ((1u << sh) - 1u));
            rbase += wd > 0 ? __popc(nbw[0]) : 0;
            rbase += wd > 1 ? __popc(nbw[1]) : 0;
            rbase += wd > 2 ? __popc(nbw[2]) : 0;
            const float* arow = sAdd + rc * KT + rbase;
            float* lo = A.out_logits ? A.out_logits + ((size_t)b * A.M + row0 + row) * N1 : nullptr;
            // pass 1: pre-activation x = score + eb + {penalty + local | xi}; -inf where masked; first maximum
            float xmax = -INFINITY;
            int xidx = 0x7fffffff;
#pragma unroll
            for (int c4 = 0; c4 < 7; ++c4)
              if (c4 * 4 < CQ) {
#pragma unroll
                for (int i = c4 * 4; i < c4 * 4 + 4; ++i) {
                  float x = -INFINITY;
                  if ((vwin >> i) & 1u) {
                    const bool isnb = (nwin >> i) & 1u;
                    const float add = isnb ? arow[__popc(nwin & ((1u << i) - 1u))] : A.xi;
                    x = (umma::after_wait(xr[i]) + sEb[c0n + i]) + add;
                    if (x > xmax) { xmax = x; xidx = c0n + i; }
                  }
                  xr[i] = __float_as_uint(x);
                }
              }
            // tanh is monotone, so the arg-max of clip*tanh(x) is the arg-max of x unless fp32 tanh maps a smaller x to
            // the same (or, by a 1-2 ulp wobble, larger) logit.  |d tanh| >= 4 e^(-2|x|) |dx| near the maximum, so only
            // pre-activations within w = max(1e-4, 5e-7 e^(2|xmax|)) of it can tie (w covers ~4 ulp of tanh); in the
            // saturated range that is a wide window, otherwise just the maximum -> a single tanh per row.
            const float thr = xmax - fmaxf(1e-4f, 5e-7f * __expf(2.f * fabsf(xmax)));
            int ncand = 0;
#pragma unroll
            for (int c4 = 0; c4 < 7; ++c4)
              if (c4 * 4 < CQ) {
#pragma unroll
                for (int i = c4 * 4; i < c4 * 4 + 4; ++i) ncand += (__uint_as_float(xr[i]) >= thr && __uint_as_float(xr[i]) != -INFINITY) ? 1 : 0;
              }
            need_all = ncand > 1 || lo != nullptr;
            if (ncand == 1) { best = A.clip * tanhf(xmax); bidx = xidx; }
          }
          const bool slow = __any_sync(FULL, need_all);
          if (slow) {        // rare (ties / saturation) or diagnostic (logits requested): every logit
            float* lo = (act && A.out_logits) ? A.out_logits + ((size_t)b * A.M + row0 + row) * N1 : nullptr;
            if (need_all) { best = -INFINITY; bidx = 0x7fffffff; }
#pragma unroll
            for (int c4 = 0; c4 < 7; ++c4)
              if (c4 * 4 < CQ) {
#pragma unroll
                for (int i = c4 * 4; i < c4 * 4 + 4; ++i) {
                  const int j = c0n + i;
                  const float x = __uint_as_float(xr[i]);
                  const float v = (need_all && x != -INFINITY) ? A.clip * tanhf(x) : -INFINITY;
                  if (need_all && v > best) { best = v; bidx = j; }
                  if (lo && j < N1) lo[j] = v;
                }
              }
          }
          umma::fence_before_sync();
          sXm[wsub * 128 + row] = best;
          reinterpret_cast<int*>(sXl)[wsub * 128 + row] = bidx;
        }
        PHASE_MARK(9);
      }
      quad_sync(11 + q);       // the four candidates of a row come from the four warps of its lane quadrant: no CTA-wide wait

      // ---- selection: first-max over the 4 column quarters (ties -> lowest index, as torch.argmax) ----------------
      int sl;
      if (forced) {
        sl = (CVRP && t == 0) ? 0 : A.start_nodes[min(row0 + row, A.M - 1)];
      } else {
        float bv = -INFINITY;
        int bi = 0x7fffffff;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const float ov = sXm[c * 128 + row];
          const int oi = reinterpret_cast<const int*>(sXl)[c * 128 + row];
          if (ov > bv) { bv = ov; bi = oi; }
        }
        sl = act ? bi : 0;
      }
      bool live_after = false;
      if (A.single_step) {
        if (wsub == 0 && in_tile) {
          const size_t g = (size_t)b * A.M + row0 + row;
          A.out_selected[g] = sl;
          if (A.out_prob) A.out_prob[g] = 1.f;
        }
      } else if (in_tile) {
        // ================= phase C: environment step; this thread owns mask word `wsub` of its row =============
        const bool was_fin = !act;
        bool fin = was_fin;
        float ld = 1.f;
        // visited words: every thread of the row reads all four, then rewrites its own -- into the other copy, so that no
        // thread can see a word of this step before it has read the previous step's
        const uint32_t* visR = sVis + (t & 1) * (TC_MT_MAX * 4);
        uint32_t* visW = sVis + ((t + 1) & 1) * (TC_MT_MAX * 4);
        const uint4 v4 = *reinterpret_cast<const uint4*>(visR + rc * 4);
        uint32_t vw[4] = {v4.x, v4.y, v4.z, v4.w};
        const uint32_t sbit = 1u << (sl & 31);
        vw[0] |= (sl >> 5) == 0 ? sbit : 0u; vw[1] |= (sl >> 5) == 1 ? sbit : 0u;
        vw[2] |= (sl >> 5) == 2 ? sbit : 0u; vw[3] |= (sl >> 5) == 3 ? sbit : 0u;
        if (CVRP) {
          const bool at_depot = sl == 0;
          ld = at_depot ? 1.f : ld0 - sDem[sl];
          vw[0] = at_depot ? (vw[0] | 1u) : (vw[0] & ~1u);
          bool allv = true;
#pragma unroll
          for (int w = 0; w < 4; ++w) {
            const int nb = N1 - w * 32;
            if (nb > 0) {
              const uint32_t fullw = nb >= 32 ? FULL : ((1u << nb) - 1u);
              allv = allv && ((vw[w] & fullw) == fullw);
            }
          }
          fin = was_fin || allv;
          if (wsub < W) {
            uint32_t big = 0u;
            const float lde = __fadd_rn(ld, 1e-6f);
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              const int j = wsub * 32 + i;
              if (j < N1 && lde < sDem[j]) big |= 1u << i;
            }
            const uint32_t mine = pick4(vw, wsub);
            uint32_t mk = mine | big;
            if (wsub == 0 && fin) mk &= ~1u;               // finished rows may stay at the depot
            visW[rc * 4 + wsub] = mine;
            sMask[wsub * 128 + rc] = mk;
          }
        } else {
          if (wsub < W) {
            const uint32_t mine = pick4(vw, wsub);
            visW[rc * 4 + wsub] = mine;
            sMask[wsub * 128 + rc] = mine;
          }
        }
        live_after = !fin;
        if (wsub == 0) {
          if (t > 0) {
            sTlen[rc] += seg_cost(A.t, b, N1, sXY, cur0, sl);
          }
          if (!CVRP && t == 0) sFirst[rc] = sl;
          sCur[rc] = sl;
          sLoad[rc] = ld;
          sFin[rc] = fin ? 1 : 0;
          if (t < A.t_max) A.tours[((size_t)b * A.M + row0 + row) * A.t_max + t] = (int16_t)sl;
        }
      }
      PHASE_MARK(10);
      if (A.single_step) break;
      bool more = __syncthreads_or(live_after ? 1 : 0) != 0;
      PHASE_MARK(11);
      if (!CVRP) more = (t + 1) < N1;
      if (!more || t + 1 >= A.t_max) { ++t; break; }
    }

    // ---- epilogue: rewards ---------------------------------------------------------------------
    if (!A.single_step) {
      for (int r = tid; r < nrows; r += RT) {
        float len = sTlen[r];
        if (!CVRP) {
          len += seg_cost(A.t, b, N1, sXY, sCur[r], sFirst[r]);
        }
        const size_t g = (size_t)b * A.M + row0 + r;
        A.reward[g] = -len;
        if (A.logp) A.logp[g] = 0.f;                 // greedy decoding: no log-likelihood
      }
      if (tid == 0) A.n_steps[b * A.ns_stride + tile] = t;
    }
    __syncthreads();
  }
  umma::fence_before_sync();
  __syncthreads();
  if (warp == 0) umma::tmem_dealloc(tm, 512);
#ifdef ELG_PHASE_TIMING
  if (tid == 0)
    for (int i = 0; i < 16; ++i) atomicAdd(&g_phase_clk[i], pclk[i]);
  if (leader)
    for (int i = 0; i < 6; ++i) atomicAdd(&g_sm_clk[grp][i], (unsigned long long)smclk[i]);
#endif
}

// ---- host side ----------------------------------------------------------------------------------
// local sequence length / 8: 4 (<= 32 positions) or 6 (<= 48); longer local sequences do not fit the tensor-memory plan
static int tc_maxe(const elg_model_desc* d) {
  const int KT = d->local_k + (d->problem == ELG_CVRP ? 1 : 0);
  return KT <= 32 ? 4 : (KT <= 48 ? 6 : 0);
}

// Largest row tile (multiple of 4, <= 112) whose layout fits the 227 KB of one SM; 0 = none
int rollout_tc_max_rows(const elg_model_desc* d, int N1) {
  if (N1 > N_RES_MAX || tc_maxe(d) == 0) return 0;
  return TC_MT_MAX;
}

// Tiles per aug-instance the tensor-core kernel would use for (B, M, N1); 0 = the shape is not eligible
int rollout_tc_tiles(const elg_model_desc* d, int B, int M, int N1, int* mt_out) {
  const int cap = rollout_tc_max_rows(d, N1);
  if (cap == 0) return 0;
  int tiles = (M + cap - 1) / cap;
  // Splitting the rows of an instance over several CTAs does not pay: a step of a 52-row tile takes 97 % of the time of a
  // 100-row tile (latency-bound phases; tools/small_batch_timing.py: 64 aug-instances 5.30 ms as one tile, 5.15 ms as two).
  if (const char* e = getenv("ELG_TC_TILES")) {        // diagnostic override (tools/small_batch_timing.py)
    const int v = atoi(e);
    if (v >= 1 && v <= 8 && v * cap >= M) tiles = v;
  }
  int mt = (((M + tiles - 1) / tiles) + 3) & ~3;
  if (mt > cap) { mt = cap; tiles = (M + mt - 1) / mt; }
  if (mt_out) *mt_out = mt;
  return tiles;
}

int launch_rollout_tc(const elg_model_desc* d, RolloutArgs& a, cudaStream_t st) {
  int mt = 0;
  const int tiles = rollout_tc_tiles(d, a.B, a.M, a.N1, &mt);
  ELG_REQUIRE(tiles > 0, ELG_EUNSUPPORTED, "tensor-core rollout does not fit (N1=%d)", a.N1);
  ELG_REQUIRE(a.mode == ELG_GREEDY, ELG_EUNSUPPORTED, "tensor-core rollout is greedy-only");
  a.tiles = tiles;
  a.MT = mt;
  const int maxe = tc_maxe(d);
  const size_t smem = (size_t)(maxe == 4 ? TcL<32>::total : TcL<48>::total) * sizeof(float);
  int dev = 0, sms = 148;
  ELG_CUDA_OK(cudaGetDevice(&dev));
  ELG_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int work = a.B * a.tiles;
  const int grid = work < sms ? work : sms;
  const bool np112 = ((a.N1 + 15) & ~15) == 112;
#define ELG_TK(P, ME)                                                                                              \
  do {                                                                                                             \
    if (np112) {                                                                                                   \
      ELG_CUDA_OK(cudaFuncSetAttribute(rollout_tc_kernel<P, ME, 112>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
      rollout_tc_kernel<P, ME, 112><<<grid, RT, smem, st>>>(a);                                                    \
    } else {                                                                                                       \
      ELG_CUDA_OK(cudaFuncSetAttribute(rollout_tc_kernel<P, ME, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
      rollout_tc_kernel<P, ME, 0><<<grid, RT, smem, st>>>(a);                                                      \
    }                                                                                                              \
  } while (0)
  if (d->problem == ELG_CVRP) {
    if (maxe == 4) ELG_TK(ELG_CVRP, 4); else ELG_TK(ELG_CVRP, 6);
  } else {
    if (maxe == 4) ELG_TK(ELG_TSP, 4); else ELG_TK(ELG_TSP, 6);
  }
#undef ELG_TK
  ELG_LAUNCH_OK();
  return ELG_OK;
}

}  // namespace elg

#ifdef ELG_PHASE_TIMING
// out32: [0, 16) the phases of a decode step (thread 0), [16, 32) the softmax rounds of group 0 and group 1 (8 each)
extern "C" int elg_debug_phase_clocks_tc(unsigned long long* out32, int reset) {
  ELG_CUDA_OK(cudaMemcpyFromSymbol(out32, elg::g_phase_clk, sizeof(unsigned long long) * 16));
  ELG_CUDA_OK(cudaMemcpyFromSymbol(out32 + 16, elg::g_sm_clk, sizeof(unsigned long long) * 16));
  if (reset) {
    unsigned long long z[16] = {0};
    ELG_CUDA_OK(cudaMemcpyToSymbol(elg::g_phase_clk, z, sizeof(z)));
    ELG_CUDA_OK(cudaMemcpyToSymbol(elg::g_sm_clk, z, sizeof(z)));
  }
  return ELG_OK;
}
#endif
