// Streamed tensor-core rollout kernel: greedy decoding of LARGE instances (112 < N+1 <= 8192, POMO width up to the
// reference's min(N, 1000); CVRP/test_vrplib.py:116) -- the same per-step path as rollout_tc.cu (reference file:line
// list in rollout.cu), but the node axis no longer fits on chip, so the three contractions of the global policy
// (CVRP/models.py:330-352, TSP/models.py:252-272) stream their B operands tile by tile:
//
//   for every tile of 128 keys:   TMA bulk copies of the K' and V^T tiles (fp16 hi/lo tcgen05 operands, 2 x 64 KB,
//       written once per batch by split_tiles_kernel into elg_tables.et)            -> shared memory
//     S_h = Q_h K'_h^T (N = 128)  A = Q (TMEM)    online softmax over the tiles in the log2 domain: running maximum and
//     O_h += P_h V_h   (N = 16)   A = P (TMEM)    denominator per (row, head) in registers; when a tile raises the maximum
//                                                 the head's 16 accumulator columns are rescaled in tensor memory first
//   for every tile of 128 nodes:  TMA bulk copy of the E' tile (64 KB; the next one streams in while this one's scores are read)
//     score = O E'^T  (N = 128)   A = O (TMEM)    running first-max arg-max of clip * tanh(score + eb + xi) over the tiles
//
// CTA = one (aug-instance, tile of 128 POMO rows); TMEM lane = row; 16 warps as in rollout_tc.cu (lane quadrant q =
// warp % 4, sub-slot wsub = warp / 4; two softmax groups of 8 warps with their own S/P buffer and mbarrier).
// The local policy (CVRP/models.py:51-175) is rollout_tc.cu's, steps (3)-(6) shared through rollout_common.cuh (12
// sequence positions per thread); its neighbourhood comes from the uint16 rank-ordered neighbour lists, tested 128
// entries at a time until k valid ones are found, and its features (distance, polar angle, demand / load) are computed
// in the kernel.  The ~k
// neighbour nodes of a row get their exact logit per tile: the scores of flagged nodes are parked in an on-chip
// [128 rows][128 nodes] scratch (the second 64 KB buffer), left out of the running arg-max, and compared with their
// penalty + local score by the threads that own the local sequence.
// Per-row bit masks (masked / visited / neighbour, one 32-bit word per 32 nodes) live in global scratch (L2-resident).
//
// TMEM columns: the plan in rollout_common.cuh, with S / P buffers [256,384) / [384,512) of the two groups, later the two
// score-tile accumulators
#include "rollout_common.cuh"

namespace elg {

constexpr int SKT = 48, SPT = 12;             // local sequence slots (k + depot <= 48), slots per thread

struct StcL {      // shared-memory layout in floats (compile-time)
  static constexpr int buf = 0;                                  // 2 x 64 KB: K' | V^T tile, later two E' tiles
  static constexpr int op1 = buf + 2 * 16384;                    // local policy B operands (see rollout_tc.cu)
  static constexpr int op2 = op1 + LH * SKT * 16;
  static constexpr int wl = op2 + 64 * LE;
  static constexpr int u = wl + E;
  static constexpr int tt = u + LH * 4;
  static constexpr int a = tt + LH * KT_MAX;
  static constexpr int pb = a + LE * 4;
  static constexpr int zb = pb + KT_MAX;
  static constexpr int cur = zb + 4;
  static constexpr int first = cur + 128;
  static constexpr int load = first + 128;
  static constexpr int tlen = load + 128;
  static constexpr int fin = tlen + 128;
  static constexpr int cnt = fin + 128;                          // visited customers per row
  static constexpr int np = cnt + 128;                           // local sequence length per row
  static constexpr int add = np + 128;                           // [128][SKT] penalty + local per sequence position
  static constexpr int addid = add + 128 * SKT;                  // [128][SKT] uint16 node ids
  static constexpr int xch = addid + 128 * SKT / 2;              // [4][128] float4: validity words / denominators
  static constexpr int xm = xch + 4 * 128 * 4;                   // [4][128] float2: maxima / arg-max candidates
  static constexpr int eb = xm + 4 * 128 * 2;                    // [2][128] score bias of the current node tiles
  static constexpr int dem = eb + 256;                           // demands of the instance when N+1 <= 4096 (phase C)
  static constexpr int ctrl = dem + 4096;
  static constexpr int bar = ctrl + 4;                           // 9 mbarriers + TMEM base address
  static constexpr int total = bar + 20;
};
static_assert(StcL::total * 4 <= 227 * 1024, "layout exceeds one SM's shared memory");

__device__ __forceinline__ float scr_at(const float* sSc, int row, int jl, int lane) { return sSc[row * 128 + (jl ^ lane)]; }

// =================================================================================================
template <int PROBLEM>
__global__ void __launch_bounds__(RT, 1) rollout_stc_kernel(const RolloutArgs A) {
  constexpr bool CVRP = PROBLEM == ELG_CVRP;
  constexpr int DEP = CVRP ? 1 : 0;
  using L = StcL;
  extern __shared__ __align__(128) float sm[];
  const int N1 = A.N1;
  const int NT = stc_tiles(N1);
  const int K1 = A.k_local + DEP;
  const int N2 = tc_n2(K1);
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
  int* sCnt = reinterpret_cast<int*>(sm + L::cnt);
  int* sNp = reinterpret_cast<int*>(sm + L::np);
  float* sAdd = sm + L::add;
  uint16_t* sAddId = reinterpret_cast<uint16_t*>(sm + L::addid);
  float4* sX4 = reinterpret_cast<float4*>(sm + L::xch);
  float2* sX2 = reinterpret_cast<float2*>(sm + L::xm);
  float* sEb = sm + L::eb;
  int* sCtrl = reinterpret_cast<int*>(sm + L::ctrl);
  uint64_t* bar_kv = reinterpret_cast<uint64_t*>(sm + L::bar);   // TMA: K' tile
  uint64_t* bar_e = bar_kv + 1;                                   // [2] TMA: E' tiles
  uint64_t* bar_scm = bar_kv + 3;                                 // [2] tcgen05.commit of the score tiles
  uint64_t* bar_g = bar_kv + 5;                                   // [2] tcgen05.commit of the softmax groups
  uint64_t* bar_loc = bar_kv + 7;                                 // tcgen05.commit of the local-policy MMAs
  uint64_t* bar_v = bar_kv + 8;                                   // TMA: V^T tile
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bar_kv + 9);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int q = warp & 3, wsub = warp >> 2, grp = wsub >> 1, kh = wsub & 1;
  uint64_t* bar_grp = bar_g + grp;
  const int row = q * 32 + lane;
  const StcWs WS = stc_ws_layout((long long)A.B * A.M, N1);
  const int Wp = WS.Wp;
  uint8_t* wsb = reinterpret_cast<uint8_t*>(A.t.ws);

  {
    stage_local_consts<L, SKT>(sm, A.derived, N2, tid);
    if (tid == 0) {
      for (int i = 0; i < 9; ++i) mbar_init(bar_kv + i, 1);
      sCtrl[1] = 0;
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) umma::tmem_alloc(tmem_ptr, 512);
    umma::fence_async_smem();
    umma::fence_before_sync();
  }
  __syncthreads();
  umma::fence_after_sync();
  const uint32_t tm = *tmem_ptr;
  const uint32_t tl = tm + ((uint32_t)(q * 32) << 16);
  const uint32_t bufA = umma::smem_addr(sm + L::buf), bufB = bufA + 65536u;       // K' | V^T, or E' slot 0 | E' slot 1
  const uint32_t op1 = umma::smem_addr(sm + L::op1), op2 = umma::smem_addr(sm + L::op2);
  const uint32_t idescS = umma::make_idesc_f16(128, 128), idescO = umma::make_idesc_f16(128, 16);
  const uint32_t idescL2 = umma::make_idesc_f16(128, N2);
  constexpr uint32_t lboN = 128u * 16u;                  // K' / E' tiles: 128 rows per 8-column chunk

  const int tiles_m = (A.M + 127) >> 7;
  const int total_work = A.B * tiles_m;
  uint32_t ph_kv = 0, ph_v = 0, ph_e[2] = {0, 0}, ph_sc[2] = {0, 0}, ph_grp = 0;      // mbarrier parities
  const bool leader = tid == grp * 256;
#ifdef ELG_PHASE_TIMING
  unsigned long long pclk[16] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
#endif

  for (;;) {
    if (tid == 0) sCtrl[0] = atomicAdd(A.work_counter, 1);
    __syncthreads();
    const int work = sCtrl[0];
    if (work >= total_work) break;
    const int b = work / tiles_m, tile = work % tiles_m;
    const int row0 = tile * 128;
    const int nrows = min(128, A.M - row0);
    const bool in_tile = row < nrows;
    const size_t g = (size_t)b * A.M + row0 + (in_tile ? row : 0);        // global row (clamped for idle lanes)
    uint32_t* gmask = reinterpret_cast<uint32_t*>(wsb + WS.mask) + g * Wp;
    uint32_t* gvis = reinterpret_cast<uint32_t*>(wsb + WS.vis) + g * Wp;
    uint32_t* gnb = reinterpret_cast<uint32_t*>(wsb + WS.nb) + g * Wp;
    const uint8_t* et = reinterpret_cast<const uint8_t*>(A.t.et) + (size_t)b * NT * ELG_TILE_BYTES;
    const float* pXY = A.t.xy + (size_t)b * N1 * 2;
    const float* pDem = CVRP ? A.t.demand + (size_t)b * N1 : nullptr;
    const float* pEb = A.t.eb + (size_t)b * N1;

    if (CVRP && N1 <= 4096)
      for (int i = tid; i < N1; i += RT) (sm + L::dem)[i] = pDem[i];
    const float* cDem = (CVRP && N1 <= 4096) ? sm + L::dem : pDem;       // phase C compares every demand with the load
    if (tid < 128) {
      sCur[tid] = 0; sFirst[tid] = 0; sLoad[tid] = 1.f; sTlen[tid] = 0.f; sCnt[tid] = 0; sNp[tid] = 0;
      sFin[tid] = tid < nrows ? 0 : 1;
    }
    if (in_tile)
      for (int w = wsub; w < Wp; w += 4) { gmask[w] = 0u; gvis[w] = 0u; gnb[w] = 0u; }
    __syncthreads();

    int t = 0;
    for (;; ++t) {
      const bool forced = t < 1 + DEP;
      const int cur0 = sCur[row];
      const float ld0 = sLoad[row];
      const bool act = in_tile && !sFin[row];
      const int cnt0 = sCnt[row];
      int sl = 0;
      PHASE_T0();

      if (!forced) {
        // ---- K' / V^T of key tile 0 on their way while the local policy runs ---------------------------------------
        if (tid == 0) {
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          mbar_expect_tx(bar_kv, 65536u);
          bulk_g2s(sm + L::buf, et + 65536, 65536u, bar_kv);
          mbar_expect_tx(bar_v, 65536u);
          bulk_g2s(sm + L::buf + 16384, et + 131072, 65536u, bar_v);
        }
        // ---- Q operand ----------------------------------------------------------------------------------------------
        {
          uint32_t hw[16], lw[16];
          if (act) {
            const float4* qp = reinterpret_cast<const float4*>(A.t.qtab + ((size_t)b * N1 + cur0) * E + 2 * wsub * D);
            const float4* fp = CVRP ? nullptr : reinterpret_cast<const float4*>(A.t.qfirst + ((size_t)b * N1 + sFirst[row]) * E + 2 * wsub * D);
#pragma unroll
            for (int d4 = 0; d4 < 2 * D / 4; ++d4) {
              float4 v4 = __ldg(qp + d4);
              if (CVRP) {
                const float4 wl = *reinterpret_cast<const float4*>(sWL + 2 * wsub * D + d4 * 4);
                v4.x = fmaf(ld0, wl.x, v4.x); v4.y = fmaf(ld0, wl.y, v4.y);
                v4.z = fmaf(ld0, wl.z, v4.z); v4.w = fmaf(ld0, wl.w, v4.w);
              } else {
                const float4 f4 = __ldg(fp + d4);
                v4.x = f4.x + v4.x; v4.y = f4.y + v4.y; v4.z = f4.z + v4.z; v4.w = f4.w + v4.w;
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
        }
        PHASE_MARK(0);

        // =================== L: local policy ===========================================================================
        // (1) the first k valid entries of the rank-ordered neighbour list of `cur`, 128 entries at a time: this thread
        //     tests entries [128 c + 32 wsub, + 32) of chunk c, the four quarters are OR-ed through shared memory
        const int NL = N1 - DEP, kloc = A.k_local;
        const uint16_t* nlist = reinterpret_cast<const uint16_t*>(A.t.nbr) + ((size_t)b * N1 + cur0) * ELG_NBR16_STRIDE(NL);
        const int p0 = wsub * SPT;
        const int ps = max(p0 - DEP, 0), pe = min(p0 + SPT - DEP, kloc);      // my neighbour ranks [ps, pe)
        int epos[SPT];
#pragma unroll
        for (int s = 0; s < SPT; ++s) epos[s] = 0;
        int c0 = 0, elast = -1;
        const int nchunks = (NL + 127) >> 7;
        for (int c = 0; c < nchunks; ++c) {
          const bool want = act && c0 < kloc;
          uint32_t rp = 0u;
          if (want) {
            const int e0 = c * 128 + wsub * 32;
            const uint4* lp = reinterpret_cast<const uint4*>(nlist + e0);
            uint4 lv[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) lv[i] = (e0 + 8 * i < NL) ? __ldg(lp + i) : make_uint4(0, 0, 0, 0);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const uint32_t wd[4] = {lv[i].x, lv[i].y, lv[i].z, lv[i].w};
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                const uint32_t id = (wd[j >> 1] >> ((j & 1) * 16)) & 0xffffu;
                const bool ok = (e0 + 8 * i + j) < NL;
                const uint32_t mwd = ok ? gmask[id >> 5] : FULL;
                rp |= (~__funnelshift_r(mwd, 0u, id) & 1u) << (8 * i + j);
              }
            }
          }
          uint32_t* xr = reinterpret_cast<uint32_t*>(sX4);                 // [4][128] words
          xr[wsub * 128 + row] = rp;
          quad_sync(11 + q);
          const uint32_t R[4] = {xr[row], xr[128 + row], xr[256 + row], xr[384 + row]};
          const int cc = __popc(R[0]) + __popc(R[1]) + __popc(R[2]) + __popc(R[3]);
          if (want && cc > 0) {
            const int take = min(cc, kloc - c0);
            elast = c * 128 + select128(R, take - 1);
            // my ranks inside this chunk: [max(ps, c0), min(pe, c0 + cc))
            const int lo = max(ps, c0), hi = min(pe, c0 + cc);
            if (lo < hi) {
              const int e1 = select128(R, lo - c0);
              unsigned long long ra = ((unsigned long long)R[1] << 32) | R[0], rb = ((unsigned long long)R[3] << 32) | R[2];
              if (e1 < 64) { ra &= ~0ull << e1; } else { ra = 0ull; rb &= ~0ull << (e1 - 64); }
#pragma unroll
              for (int s = 0; s < SPT; ++s) {
                const int r = ps + s;
                if (r >= lo && r < hi) {
                  const bool in_a = ra != 0ull;
                  const unsigned long long x = in_a ? ra : rb;
                  epos[s] = c * 128 + max(__ffsll((long long)x) - 1, 0) + (in_a ? 0 : 64);
                  const unsigned long long y = x & (x - 1ull);
                  ra = in_a ? y : ra;
                  rb = in_a ? rb : y;
                }
              }
            }
          }
          c0 += want ? cc : 0;
          const int more = __syncthreads_or((act && c0 < kloc && c + 1 < nchunks) ? 1 : 0);   // also fences the exchange buffer
          if (!more) break;
        }
        const int kk = min(c0, kloc);
        PHASE_MARK(1);
        const int np = act ? kk + DEP : 0;
        // slot s of this thread is sequence position p0 + s; neighbour rank p0 + s - DEP (the depot heads the cvrp sequence)
        LocalSeq<SPT> ls;
        ls.p0 = p0;
        ls.cpen = 1.f;
        uint32_t idw[SPT / 2];
        {
          const float xc = pXY[2 * cur0], yc = pXY[2 * cur0 + 1];
          float dmax = 0.f;
          if (kk > 0) {
            const int nl = nlist[elast];
            dmax = dist2(xc - pXY[2 * nl], yc - pXY[2 * nl + 1]);
          }
          const float r0d = CVRP ? (dmax != 0.f ? 1.f / (dmax + 1e-6f) : 1.f) : 1.f / (dmax + 1e-6f);
          if (CVRP && dmax != 0.f) ls.cpen = (dmax + 1e-6f) / dmax;       // penalty -d / dmax = -f0 (dmax + 1e-6) / dmax
          const float rld = 1.f / ld0;
#pragma unroll
          for (int i = 0; i < SPT / 2; ++i) idw[i] = 0u;
#pragma unroll
          for (int s = 0; s < SPT; ++s) {
            ls.f0[s] = ls.f1[s] = ls.f2[s] = 0.f;
            const int p = p0 + s;
            // the rank of slot s among my ranks: slots of wsub 0 are shifted by the depot
            const int sr = (DEP && wsub == 0) ? s - 1 : s;
            const bool mine = p < np && !(DEP && p == 0);
            if (mine) {
              const int nd = nlist[epos[sr < 0 ? 0 : sr]];
              idw[s >> 1] |= (uint32_t)nd << ((s & 1) * 16);
              const float xn = pXY[2 * nd], yn = pXY[2 * nd + 1];
              const float dd = dist2(xc - xn, yc - yn);
              ls.f0[s] = dd * r0d;
              ls.f1[s] = atan2f(yn - yc, xn - xc);
              if (CVRP) ls.f2[s] = pDem[nd] * rld;
              atomicOr(gnb + (nd >> 5), 1u << (nd & 31));               // flagged: left out of the streamed arg-max
            }
          }
          if (DEP && wsub == 0 && np > 0) atomicOr(gnb, 1u);
        }
        const bool depot_masked = CVRP && act && (gmask[0] & 1u);
        PHASE_MARK(2);
        // (3) per-head maxima of the row: fp32, combined over the four quarters through shared memory
        ls.nv = np - p0;
        ls.dep_off = DEP && wsub == 0 && depot_masked;
        float mh[LH];
        {
          lp_head_max(ls, sU, sT, mh);
          sX4[wsub * 128 + row] = make_float4(mh[0], mh[1], mh[2], mh[3]);
          quad_sync(11 + q);
          const float4 a0 = sX4[row], a1 = sX4[128 + row], a2 = sX4[256 + row], a3 = sX4[384 + row];
          mh[0] = fmaxf(fmaxf(a0.x, a1.x), fmaxf(a2.x, a3.x)); mh[1] = fmaxf(fmaxf(a0.y, a1.y), fmaxf(a2.y, a3.y));
          mh[2] = fmaxf(fmaxf(a0.z, a1.z), fmaxf(a2.z, a3.z)); mh[3] = fmaxf(fmaxf(a0.w, a1.w), fmaxf(a2.w, a3.w));
        }
        // (4) softmax weights -> TMEM, then the vps contraction
        lp_weights<SPT, SKT>(ls, sU, sT, mh, tl, wsub);
        umma::wait_st();
        umma::fence_before_sync();
        __syncthreads();
        if (tid == 0) {
          umma::fence_after_sync();
          lp_issue_vps<SKT>(tm, op1, idescO);
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

        // MMA issue helpers (leaders only): operands of the current key tile sit in the two 64 KB buffers
        auto issue_qk = [&](int head) {
          const uint32_t aHi = tm + TC_COL_Q + 8 * head, bHi = bufA + head * 2 * lboN;
          mma_split3(tm + TC_COL_S + grp * 128, aHi, aHi + 64, 0, bHi, bHi + 32768u, 0, lboN, idescS, 1, false);
        };
        auto issue_pv = [&](int head, bool accumulate) {
          const uint32_t pHi = tm + TC_COL_S + grp * 128, vHi = bufB + head * (128 * 32);
          mma_split3(tm + TC_COL_O + 16 * head, pHi, pHi + 64, 8, vHi, vHi + 32768u, 512, 256, idescO, 8, accumulate);
        };
        if (tid == 0) {
          umma::fence_after_sync();
          lp_issue_pemz(tm, op2, N2, idescL2);
          umma::commit(bar_loc);
        }
        PHASE_MARK(4);
        // (6) penalty + local score per sequence position -> shared memory (with the node ids), read back after the score tiles
        mbar_wait(bar_loc, 1u);
        umma::fence_after_sync();
        lp_pen_local(ls, tl, K1, np, act, sZB, sPB, [&](int s, int p, float v) {
          sAdd[row * SKT + p] = v;
          sAddId[row * SKT + p] = (uint16_t)((idw[s >> 1] >> ((s & 1) * 16)) & 0xffffu);
        });
        if (wsub == 0) sNp[row] = np;          // 0 for an idle row
        umma::fence_before_sync();
        __syncthreads();                       // [pem | z] read by everybody before the first P V reuses the columns

        PHASE_MARK(5);
        // =================== global policy: online softmax over the key tiles ==========================================
        float mr0 = -INFINITY, mr1 = -INFINITY, mr2 = -INFINITY, mr3 = -INFINITY;      // running maxima of heads 4 grp + rho
        float lt0 = 0.f, lt1 = 0.f, lt2 = 0.f, lt3 = 0.f;                               // running denominators (my key half)
        for (int kt = 0; kt < NT; ++kt) {
          // valid-key bits of my 64 keys of this tile
          uint32_t v0 = 0u, v1 = 0u;
          if (act) {
            const uint2 mw = *reinterpret_cast<const uint2*>(gmask + 4 * kt + 2 * kh);
            const int base = kt * 128 + kh * 64;
            const int n0 = N1 - base, n1 = N1 - base - 32;
            v0 = ~mw.x & (n0 >= 32 ? FULL : (n0 > 0 ? ((1u << n0) - 1u) : 0u));
            v1 = ~mw.y & (n1 >= 32 ? FULL : (n1 > 0 ? ((1u << n1) - 1u) : 0u));
          }
          if (leader) {
            mbar_wait(bar_kv, ph_kv);
            umma::fence_after_sync();
            issue_qk(4 * grp);
            umma::commit(bar_grp);
          }
          ph_kv ^= 1;
#pragma unroll 1
          for (int rho = 0; rho < 4; ++rho) {
            mbar_wait(bar_grp, ph_grp);
            ph_grp ^= 1;
            umma::fence_after_sync();
            if (rho == 3 && leader && kt + 1 < NT) {
              // the K' tile has been read for the last time by this group; the second leader to get here refills it
              if (atomicAdd(&sCtrl[1], 1) == 1) {
                sCtrl[1] = 0;
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                mbar_expect_tx(bar_kv, 65536u);
                bulk_g2s(sm + L::buf, et + (size_t)(kt + 1) * ELG_TILE_BYTES + 65536, 65536u, bar_kv);
              }
            }
            const uint32_t sb = tl + TC_COL_S + grp * 128;
            uint32_t sr[64];
            umma::ld32_nw(sb + kh * 64, sr);
            umma::ld32_nw(sb + kh * 64 + 32, sr + 32);
            umma::wait_ld();
            float mloc = -INFINITY;
#pragma unroll
            for (int i = 0; i < 64; ++i) {
              const bool valid = ((i < 32 ? (v0 >> i) : (v1 >> (i - 32))) & 1u) != 0u;
              const float s = valid ? umma::after_wait(sr[i]) : -INFINITY;
              sr[i] = __float_as_uint(s);
              mloc = fmaxf(mloc, s);
            }
            // the row's maximum over this tile: both key halves (shared memory + 64-thread barrier)
            float* xmx = reinterpret_cast<float*>(sX2);
            xmx[wsub * 128 + row] = mloc;
            pair_sync(1 + grp * 4 + q);
            const float mt = fmaxf(mloc, xmx[(wsub ^ 1) * 128 + row]);
            const float mold = rho == 0 ? mr0 : (rho == 1 ? mr1 : (rho == 2 ? mr2 : mr3));
            const float mnew = fmaxf(mold, mt);
            const float fsc = mold == mnew ? 1.f : umma::ex2_raw(mold - mnew);      // mold = -inf -> 0 (nothing accumulated yet)
            if (rho == 0) mr0 = mnew; else if (rho == 1) mr1 = mnew; else if (rho == 2) mr2 = mnew; else mr3 = mnew;
            // a higher maximum: rescale the head's accumulator columns (my half of the 16) before P V adds to them
            if (kt > 0 && __any_sync(FULL, fsc != 1.f)) {
              uint32_t oc[8];
              const uint32_t oa = tl + TC_COL_O + 16 * (4 * grp + rho) + 8 * kh;
              umma::ld8_nw(oa, oc);
              umma::wait_ld();
#pragma unroll
              for (int i = 0; i < 8; ++i) oc[i] = __float_as_uint(umma::after_wait(oc[i]) * fsc);
              umma::st8(oa, oc);
            }
            const float moff = mnew == -INFINITY ? 0.f : mnew - TC_P_SCALE_LOG2;
            float lloc = 0.f;
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              const float pa = umma::ex2_raw(__uint_as_float(sr[2 * i]) - moff);
              const float pb2 = umma::ex2_raw(__uint_as_float(sr[2 * i + 1]) - moff);
              lloc += pa + pb2;
              uint32_t hwd, lwd;
              umma::split2_f16(pa, pb2, hwd, lwd);
              sr[2 * i] = hwd;
              sr[2 * i + 1] = lwd;
            }
            {
              const float lold = rho == 0 ? lt0 : (rho == 1 ? lt1 : (rho == 2 ? lt2 : lt3));
              const float lnew = fmaf(lold, fsc, lloc);
              if (rho == 0) lt0 = lnew; else if (rho == 1) lt1 = lnew; else if (rho == 2) lt2 = lnew; else lt3 = lnew;
            }
            // P (fp16 hi/lo, two keys per column) in place of S: hi at [sb, sb + 64), lo behind it
            umma::st16s<2>(sb + kh * 32, sr);
            umma::st16s<2>(sb + kh * 32 + 16, sr + 32);
            umma::st16s<2>(sb + 64 + kh * 32, sr + 1);
            umma::st16s<2>(sb + 64 + kh * 32 + 16, sr + 33);
            umma::wait_st();
            umma::fence_before_sync();
            group_sync(9 + grp);
            if (leader) {
              if (rho == 0) mbar_wait(bar_v, ph_v);                   // the tile's V^T (in flight since the end of the previous tile)
              umma::fence_after_sync();
              issue_pv(4 * grp + rho, kt > 0);
              if (rho < 3) issue_qk(4 * grp + rho + 1);
              umma::commit(bar_grp);
            }
          }
          // every MMA of this tile done (both groups) before the buffers are refilled / the accumulators are read
          mbar_wait(bar_grp, ph_grp);
          ph_grp ^= 1;
          ph_v ^= 1;
          umma::fence_after_sync();
          umma::fence_before_sync();
          __syncthreads();
          if (tid == 0 && kt + 1 < NT) {          // V^T of the next tile; its K' has been on its way since round 3
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            mbar_expect_tx(bar_v, 65536u);
            bulk_g2s(sm + L::buf + 16384, et + (size_t)(kt + 1) * ELG_TILE_BYTES + 131072, 65536u, bar_v);
          }
        }
        PHASE_MARK(6);
        // ---- E' tile 0 on its way; O = accumulators / denominators -> O operand -----------------------------------------
        if (tid == 0) {
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          mbar_expect_tx(bar_e, 65536u);
          bulk_g2s(sm + L::buf, et, 65536u, bar_e);
        }
        sX4[wsub * 128 + row] = make_float4(lt0, lt1, lt2, lt3);
        if (tid < 128) sEb[tid] = tid < N1 ? pEb[tid] : 0.f;
        pair_sync(1 + grp * 4 + q);
        {
          const float4 lo4 = sX4[(wsub ^ 1) * 128 + row];
          const float la = kh ? (lt2 + lo4.z) : (lt0 + lo4.x), lb = kh ? (lt3 + lo4.w) : (lt1 + lo4.y);
          umma::fence_after_sync();
          store_o_operand(tl, grp, kh, la, lb, act);
          umma::wait_st();
          umma::fence_before_sync();
        }
        __syncthreads();

        PHASE_MARK(7);
        // =================== score tiles: running arg-max of clip * tanh(score + eb + xi) ================================
        // E' tiles come through the first 64 KB buffer (the next one is requested as soon as the tile's MMAs are done, i.e.
        // while its scores are being read); the second buffer is a [128 rows][128 nodes] scratch for the scores of the
        // tile's NEIGHBOUR nodes, which get `penalty + local` instead of xi from the threads that own the local sequence
        auto issue_score = [&](int nt) {
          mma_split3(tm + TC_COL_S + (nt & 1) * 128, tm + TC_COL_Q, tm + TC_COL_Q + 64, 8, bufA, bufA + 32768u, 2 * lboN, lboN, idescS, 8, false);
          umma::commit(bar_scm);
        };
        float* sSc = sm + L::buf + 16384;                 // scratch: score of node jl of this tile at [row][jl ^ (row & 31)]
        float xbest = -INFINITY, vbest = -INFINITY, win = 0.f;
        int ibest = 0x7fffffff;
        auto consider = [&](float x, int j) {
          // tanh is monotone: only pre-activations within `win` of the running maximum can reach its logit (rollout_tc.cu)
          if (x > xbest - win) {
            const float v = A.clip * tanhf(x);
            if (v > vbest || (v == vbest && j < ibest)) { vbest = v; ibest = j; }
            if (x > xbest) { xbest = x; win = fmaxf(1e-4f, 5e-7f * __expf(2.f * fabsf(x))); }
          }
        };
        const int npr = act ? sNp[row] : 0;
        for (int nt = 0; nt < NT; ++nt) {
          const int sl2 = nt & 1;
          if (tid == 0) {
            mbar_wait(bar_e, ph_e[0]);
            umma::fence_after_sync();
            issue_score(nt);
          }
          ph_e[0] ^= 1;
          mbar_wait(bar_scm, ph_sc[0]);
          ph_sc[0] ^= 1;
          umma::fence_after_sync();
          if (tid == 0 && nt + 1 < NT) {        // the E' buffer is free again: the next tile streams in while this one is read
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            mbar_expect_tx(bar_e, 65536u);
            bulk_g2s(sm + L::buf, et + (size_t)(nt + 1) * ELG_TILE_BYTES, 65536u, bar_e);
          }
          {
            uint32_t xr[32];
            umma::ld32_nw(tl + TC_COL_S + sl2 * 128 + 32 * wsub, xr);
            umma::wait_ld();
            if (act) {
              const int jb = nt * 128 + 32 * wsub;
              const int nb = N1 - jb;
              const uint32_t vwin = ~gmask[4 * nt + wsub] & (nb >= 32 ? FULL : (nb > 0 ? ((1u << nb) - 1u) : 0u));
              const uint32_t nwin = gnb[4 * nt + wsub];
              const float* ebt = sEb + sl2 * 128 + 32 * wsub;
              float* scr = sSc + row * 128;
#pragma unroll
              for (int i = 0; i < 32; ++i) {
                if ((vwin >> i) & 1u) {
                  const float sc = umma::after_wait(xr[i]);
                  if ((nwin >> i) & 1u) scr[(32 * wsub + i) ^ lane] = sc + ebt[i];      // a neighbour: exact logit below
                  else consider((sc + ebt[i]) + A.xi, jb + i);
                }
              }
            }
          }
          umma::fence_before_sync();
          quad_sync(11 + q);      // the scratch row is written and read by the four threads of the row (one lane quadrant);
                                    // the CTA barrier at the end of the iteration still orders the accumulator reads of all
                                    // warps before the MMAs of the tile after next
          // the neighbours of this tile (and the depot) with their own penalty + local score; only the depot can be masked
          if (act) {
#pragma unroll
            for (int s = 0; s < SPT; ++s) {
              const int p = p0 + s;
              if (p < npr) {
                const int nd = sAddId[row * SKT + p];
                if ((nd >> 7) == nt) {
                  const bool masked = DEP && p == 0 && (gmask[0] & 1u);
                  if (!masked) consider(scr_at(sSc, row, nd & 127, lane) + sAdd[row * SKT + p], nd);
                  gnb[nd >> 5] = 0u;
                }
              }
            }
          }
          if (nt + 1 < NT) {
            const int j = (nt + 1) * 128 + (tid & 127);
            if (tid < 128) sEb[(sl2 ^ 1) * 128 + tid] = j < N1 ? pEb[j] : 0.f;
            __syncthreads();                     // scratch and eb slot may be rewritten by the next tile
          }
        }
        PHASE_MARK(8);
        sX2[wsub * 128 + row] = make_float2(vbest, __int_as_float(ibest));
        quad_sync(11 + q);        // candidates of a row: its lane quadrant only
        {
          float bv = -INFINITY;
          int bi = 0x7fffffff;
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const float2 cnd = sX2[c * 128 + row];
            const int oi = __float_as_int(cnd.y);
            if (cnd.x > bv || (cnd.x == bv && oi < bi)) { bv = cnd.x; bi = oi; }
          }
          sl = act ? bi : 0;
        }
      } else {
        sl = (CVRP && t == 0) ? 0 : A.start_nodes[min(row0 + row, A.M - 1)];
        __syncthreads();      // forced steps have no other barrier between the row-state reads above and phase C's rewrite
      }

      PHASE_MARK(9);
      // ================= phase C: environment step on the global bit masks; this thread owns words w = wsub mod 4 =========
      bool live_after = false;
      if (in_tile) {
        const bool was_fin = !act;
        bool fin = was_fin;
        float ld = 1.f;
        const int cntv = cnt0 + ((CVRP ? sl != 0 : true) && !was_fin ? 1 : 0);
        if (CVRP) {
          const bool at_depot = sl == 0;
          ld = at_depot ? 1.f : ld0 - pDem[sl];
          fin = was_fin || (at_depot && cntv == N1 - 1);
          const float lde = __fadd_rn(ld, 1e-6f);
          for (int w = wsub; w < Wp; w += 4) {
            uint32_t vw = gvis[w];
            if ((sl >> 5) == w) vw |= 1u << (sl & 31);
            if (w == 0) vw = at_depot ? (vw | 1u) : (vw & ~1u);
            uint32_t big = 0u;
            const int jb = w * 32;
            if (jb < N1) {
#pragma unroll 8
              for (int i = 0; i < 32; ++i) {
                const int j = jb + i;
                if (j < N1 && lde < cDem[j]) big |= 1u << i;
              }
            }
            uint32_t mk = vw | big;
            if (w == 0 && fin) mk &= ~1u;
            gvis[w] = vw;
            gmask[w] = mk;
          }
        } else {
          const int w = sl >> 5;
          if ((w & 3) == wsub) {
            const uint32_t vw = gvis[w] | (1u << (sl & 31));
            gvis[w] = vw;
            gmask[w] = vw;
          }
        }
        live_after = !fin;
        if (wsub == 0) {
          if (t > 0) {
            sTlen[row] += seg_cost(A.t, b, N1, pXY, cur0, sl);
          }
          if (!CVRP && t == 0) sFirst[row] = sl;
          sCur[row] = sl;
          sLoad[row] = ld;
          sFin[row] = fin ? 1 : 0;
          sCnt[row] = cntv;
          if (t < A.t_max) A.tours[((size_t)b * A.M + row0 + row) * A.t_max + t] = (int16_t)sl;
        }
      }
      PHASE_MARK(10);
      bool more = __syncthreads_or(live_after ? 1 : 0) != 0;
      PHASE_MARK(11);
      if (!CVRP) more = (t + 1) < N1;
      if (!more || t + 1 >= A.t_max) { ++t; break; }
    }

    // ---- epilogue: rewards ---------------------------------------------------------------------
    for (int r = tid; r < nrows; r += RT) {
      float len = sTlen[r];
      if (!CVRP) {
        len += seg_cost(A.t, b, N1, pXY, sCur[r], sFirst[r]);
      }
      const size_t gg = (size_t)b * A.M + row0 + r;
      A.reward[gg] = -len;
      if (A.logp) A.logp[gg] = 0.f;
    }
    if (tid == 0) A.n_steps[b * A.ns_stride + tile] = t;
    __syncthreads();
  }
  umma::fence_before_sync();
  __syncthreads();
  if (warp == 0) umma::tmem_dealloc(tm, 512);
#ifdef ELG_PHASE_TIMING
  if (tid == 0)
    for (int i = 0; i < 16; ++i) atomicAdd(&g_phase_clk[i], pclk[i]);
#endif
}

// ---- host side ----------------------------------------------------------------------------------
bool rollout_stc_eligible(const elg_model_desc* d, const RolloutArgs& a) {
  const int K1 = d->local_k + (d->problem == ELG_CVRP ? 1 : 0);
  return a.mode == ELG_GREEDY && !a.single_step && !(d->flags & ELG_FLAG_ATTN_FP32) && a.t.et && a.t.ws &&
         a.N1 > N_RES_MAX && a.N1 <= N_STREAM_MAX && K1 <= SKT - 4 && a.work_counter;
}

int launch_rollout_stc(const elg_model_desc* d, RolloutArgs& a, cudaStream_t st) {
  const size_t smem = (size_t)StcL::total * sizeof(float);
  int dev = 0, sms = 148;
  ELG_CUDA_OK(cudaGetDevice(&dev));
  ELG_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int work = a.B * ((a.M + 127) / 128);
  const int grid = work < sms ? work : sms;
  if (d->problem == ELG_CVRP) {
    ELG_CUDA_OK(cudaFuncSetAttribute(rollout_stc_kernel<ELG_CVRP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    rollout_stc_kernel<ELG_CVRP><<<grid, RT, smem, st>>>(a);
  } else {
    ELG_CUDA_OK(cudaFuncSetAttribute(rollout_stc_kernel<ELG_TSP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    rollout_stc_kernel<ELG_TSP><<<grid, RT, smem, st>>>(a);
  }
  ELG_LAUNCH_OK();
  return ELG_OK;
}

}  // namespace elg

extern "C" size_t elg_rollout_ws_bytes(const elg_model_desc* d, int B, int M, int N1) {
  if (elg::check_desc(d) || B <= 0 || M <= 0 || N1 <= elg::N_RES_MAX || N1 > elg::N_STREAM_MAX) return 0;
  return elg::stc_ws_layout((long long)B * M, N1).total;
}

#ifdef ELG_PHASE_TIMING
extern "C" int elg_debug_phase_clocks_stc(unsigned long long* out16, int reset) {
  ELG_CUDA_OK(cudaMemcpyFromSymbol(out16, elg::g_phase_clk, sizeof(unsigned long long) * 16));
  if (reset) { unsigned long long z[16] = {0}; ELG_CUDA_OK(cudaMemcpyToSymbol(elg::g_phase_clk, z, sizeof(z))); }
  return ELG_OK;
}
#endif
