// Persistent rollout kernel: the whole autoregressive construction loop of one aug-instance
// (decode step of the global POMO attention policy + local k-nearest attention policy + env step)
// runs inside one CTA.
//
// reference per-step path (file:line under the reference tree):
//   rollout                      CVRP/utils.py:7-29            TSP/utils.py:7-26
//   get_cur_feature              CVRP/CVRPEnv.py:291-318       TSP/TSPEnv.py:135-156
//   one_step_rollout             CVRP/CVRPModel.py:36-75       TSP/TSPModel.py:26-64
//   Decoder.forward              CVRP/models.py:322-423        TSP/models.py:244-303
//   local_policy_att.forward     CVRP/models.py:51-175         TSP/models.py:48-110
//   env.step                     CVRP/CVRPEnv.py:190-249       TSP/TSPEnv.py:108-133
//   reward                       CVRP/CVRPEnv.py:251-288       TSP/TSPEnv.py:158-184
//
// Work decomposition (DESIGN.md has the full story):
//   CTA   = one (aug-instance, tile of <= 64 POMO rows), 16 warps, persistent over work items.
//   RESIDENT (N1 <= 112): K', V, E' of the instance (3 x N1 x 128 fp32) are brought into shared
//           memory once per work item by cp.async.bulk (TMA) and stay there for the whole rollout.
//   STREAMING (N1 <= 8192): K', V, E' are read through L1/L2 every step (all warps of a CTA walk the
//           nodes in the same order, so a line is fetched from L2 about once per CTA per step).
//   phase A  thread = (row, head): q . K over the warp-union of unmasked nodes with a lazily rescaled
//            online softmax (log2 domain) and the weighted V sum; K/V rows are warp-broadcast loads.
//   phase B  warp = 4 rows.  B1: local policy with an octet of lanes per row (walk over the
//            distance-presorted neighbour list, polar features, 4-head attention with the constant
//            query folded into 3-vector dots + tables).  B2: score tile (4 rows x 4 node-chunks per
//            lane) against E', 128 nodes at a time.  B3: clip*tanh(score + penalty + local) + mask,
//            running first-max argmax (or Philox sampling when N1 <= 128).
//   phase C  env step on bit masks (fp32 load recurrence, visited / too-large masks by warp ballots).
#include "rollout_common.cuh"

namespace elg {

// Sampled decision of one row (one warp; node j = lane + 32 ch of the row's masked logits lg, N1 <= 128), the draw
// elg_rollout and elg_decode_step document: u = ((x >> 8) + 0.5) 2^-24, x the first word of Philox4x32-10 at counter
// (grow lo, grow hi, step lo, step hi) and key (seed lo, seed hi); the pick is the first node in index order with p > 0
// and running sum >= u * total.  The total (butterfly) and the running sums (scan) round differently, so at u = 1 the
// last running sum can end one ulp below u * total: the last node of positive probability is then the pick.
// samp / selp are written only when the row has a node of positive probability.
__device__ __forceinline__ void sample_row(const float (&lg)[4], float best, unsigned long long seed, unsigned long long grow,
                                           unsigned long long step, int lane, int& samp, float& selp) {
  float bv = best;
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) bv = fmaxf(bv, __shfl_xor_sync(FULL, bv, off));
  float pr[4], tot = 0.f;
#pragma unroll
  for (int ch = 0; ch < 4; ++ch) { pr[ch] = lg[ch] == -INFINITY ? 0.f : expf(lg[ch] - bv); tot += pr[ch]; }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) tot += __shfl_xor_sync(FULL, tot, off);
  const uint4 rnd = philox4x32(make_uint4((uint32_t)grow, (uint32_t)(grow >> 32), (uint32_t)step, (uint32_t)(step >> 32)),
                               make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
  const float target = ((rnd.x >> 8) + 0.5f) * (1.f / 16777216.f) * tot;
  float run = 0.f, pickp = 0.f;
  int pick = -1, last = -1;
#pragma unroll
  for (int ch = 0; ch < 4; ++ch) {
    float inc = pr[ch];
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const float nb = __shfl_up_sync(FULL, inc, off);
      if (lane >= off) inc += nb;
    }
    const float cum = run + inc;
    const uint32_t hit = __ballot_sync(FULL, pr[ch] > 0.f && cum >= target);
    const uint32_t pos = __ballot_sync(FULL, pr[ch] > 0.f);
    if (pick < 0 && pos) {          // the first hit, else this chunk's last node of positive probability
      const int src = hit ? __ffs(hit) - 1 : 31 - __clz(pos);
      last = src + 32 * ch;
      pickp = __shfl_sync(FULL, pr[ch], src);
      if (hit) pick = last;
    }
    run += __shfl_sync(FULL, inc, 31);
  }
  if (pick < 0) pick = last;
  if (pick >= 0) { samp = pick; selp = pickp / tot; }
}

// ---- shared-memory layout (offsets in floats) ---------------------------------------------------
struct SmemLayout {
  int k, v, e, o, eb, xy, dem, wl, u, tt, a, vpe, pw, pb, zw, zb;
  int cur, first, load, tlen, fin, logp, mask, vis, ids, dense, ctrl, bar;
  int total;     // floats
};
__host__ __device__ inline int r4(int x) { return (x + 3) & ~3; }
__host__ __device__ inline SmemLayout make_layout(int N1, int MT, int KT, bool resident) {
  SmemLayout L;
  const int W = (N1 + 31) >> 5;
  int o = 0;
  L.k = o; o += resident ? N1 * E : 0;
  L.v = o; o += resident ? N1 * E : 0;
  // resident: E' as fp16 hi/lo tcgen05 B operands (N1 padded to 16 rows); attention outputs as fp16 hi/lo
  // A operands (64 rows; +1 KB because the upper 64 MMA rows alias the next k-chunk); the staged scores alias them
  L.e = o; o += resident ? 2 * (((N1 + 15) & ~15) * 64) : 0;
  L.o = o; o += resident ? (2 * A_HALF + 1024) / 4 : MT * E;
  L.eb = o; o += resident ? r4(N1) : 0;
  L.xy = o; o += resident ? r4(2 * N1) : 0;
  L.dem = o; o += resident ? r4(N1) : 0;
  L.wl = o; o += E;
  L.u = o; o += LH * 4;
  L.tt = o; o += LH * KT_MAX;
  L.a = o; o += LE * 4;                     // (Wv We)[c][0..2], (Wv be)[c]
  L.vpe = o; o += KT * TS;
  L.pw = o; o += KT * TS;
  L.pb = o; o += KT_MAX;
  L.zw = o; o += LE * 4;
  L.zb = o; o += 4;
  L.cur = o; o += MT;
  L.first = o; o += MT;
  L.load = o; o += MT;
  L.tlen = o; o += MT;
  L.fin = o; o += MT;
  L.logp = o; o += MT;
  L.mask = o; o += r4(MT * W);
  L.vis = o; o += r4(MT * W);
  L.ids = o; o += RW * 4 * (KT_MAX / 2);            // per warp: 4 rows x 64 uint16 neighbour ids
  L.dense = o; o += resident ? 0 : RW * 4 * DS;     // resident: aliases the warp's dead attention rows
  L.ctrl = o; o += 4;
  L.bar = o; o += 8;                                // TMA mbarrier, MMA mbarrier, TMEM base address
  L.total = o;
  return L;
}

// =================================================================================================
template <int PROBLEM, int MAXE, bool RESIDENT>
__global__ void __launch_bounds__(RT, 1) rollout_kernel(const RolloutArgs A) {
  constexpr bool CVRP = PROBLEM == ELG_CVRP;
  constexpr int DEP = CVRP ? 1 : 0;
  extern __shared__ __align__(128) float sm[];
  const int N1 = A.N1;
  const int W = (N1 + 31) >> 5;                  // mask words per row
  const int KT = MAXE * 8;
  const SmemLayout L = make_layout(N1, A.MT, KT, RESIDENT);
  float* sO = sm + L.o;
  float* sWL = sm + L.wl;
  const float* sU = sm + L.u;
  const float* sT = sm + L.tt;
  const float* sA = sm + L.a;
  const float* sVPE = sm + L.vpe;
  const float* sPW = sm + L.pw;
  const float* sPB = sm + L.pb;
  const float* sZW = sm + L.zw;
  const float* sZB = sm + L.zb;
  int* sCur = reinterpret_cast<int*>(sm + L.cur);
  int* sFirst = reinterpret_cast<int*>(sm + L.first);
  float* sLoad = sm + L.load;
  float* sTlen = sm + L.tlen;
  int* sFin = reinterpret_cast<int*>(sm + L.fin);
  float* sLogp = sm + L.logp;
  uint32_t* sMask = reinterpret_cast<uint32_t*>(sm + L.mask);
  uint32_t* sVis = reinterpret_cast<uint32_t*>(sm + L.vis);
  int* sCtrl = reinterpret_cast<int*>(sm + L.ctrl);
  uint64_t* bar = reinterpret_cast<uint64_t*>(sm + L.bar);      // TMA completion
  uint64_t* bar_mma = bar + 1;                                    // tcgen05.commit completion
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bar + 2);
  const int N1p = (N1 + 15) & ~15;                                // E' rows padded for the MMA N dimension

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  // ---- one-time: folded local-policy tables and the load column of Wq_last ---------------------
  {
    const float* loc = A.derived + DER_LOC;
    float* w = sm;
    for (int i = tid; i < E; i += RT) w[L.wl + i] = A.derived[DER_WL + i];
    for (int i = tid; i < LH * 4; i += RT) w[L.u + i] = loc[LOC_U + i];
    for (int i = tid; i < LH * KT_MAX; i += RT) w[L.tt + i] = loc[LOC_T + i];
    for (int i = tid; i < LE * 4; i += RT) {
      w[L.a + i] = (i & 3) == 3 ? loc[LOC_CV + (i >> 2)] : loc[LOC_A + i];
      w[L.zw + i] = loc[LOC_ZW + i];
    }
    for (int i = tid; i < KT_MAX; i += RT) w[L.pb + i] = loc[LOC_PB + i];
    for (int i = tid; i < 4; i += RT) w[L.zb + i] = loc[LOC_ZB + i];
    for (int i = tid; i < KT * LE; i += RT) {
      int p = i / LE, c = i % LE;
      w[L.vpe + p * TS + c] = loc[LOC_VPE + i];
      w[L.pw + p * TS + c] = loc[LOC_PW + i];
    }
    if (RESIDENT && tid == 0) {
      mbar_init(bar, 1);
      mbar_init(bar_mma, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (RESIDENT && warp == 0) umma::tmem_alloc(tmem_ptr, 256);     // scores: hi*hi in cols [0,112), cross terms in [128,240)
    if (RESIDENT) umma::fence_before_sync();
  }
  __syncthreads();
  uint32_t tmem_d = 0;
  if (RESIDENT) { umma::fence_after_sync(); tmem_d = *tmem_ptr; }

  const int total_work = A.B * A.tiles;
  uint32_t bar_phase = 0, mma_phase = 0;
#ifdef ELG_PHASE_TIMING
  unsigned long long pclk[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#endif

  for (int iter = 0;; ++iter) {
    // ---- fetch work: dynamic (atomic counter) for rollouts, static for single decode steps ------
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

    // ---- the instance's tables: shared memory (resident) or global memory through L1/L2 ---------
    const float *pK, *pV, *pE, *pEb, *pXY, *pDem;
    if (RESIDENT) {
      float* sK = sm + L.k; float* sV = sm + L.v; float* sE = sm + L.e;
      float* sEb = sm + L.eb; float* sXY = sm + L.xy; float* sDem = sm + L.dem;
      if (tid == 0) {
        const uint32_t bytes = (uint32_t)N1 * E * sizeof(float);
        const uint32_t ebytes = (uint32_t)N1p * 512u;        // fp16 hi + lo, N1p rows x 128 k
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        mbar_expect_tx(bar, 2 * bytes + ebytes);
        bulk_g2s(sK, A.t.k + (size_t)b * N1 * E, bytes, bar);
        bulk_g2s(sV, A.t.v + (size_t)b * N1 * E, bytes, bar);
        bulk_g2s(sE, reinterpret_cast<const uint8_t*>(A.t.e) + (size_t)b * 3 * ebytes, ebytes, bar);      // segment 0 of [E' | K' | V^T]
      }
      for (int i = tid; i < N1; i += RT) {
        sEb[i] = A.t.eb[(size_t)b * N1 + i];
        sXY[2 * i] = A.t.xy[((size_t)b * N1 + i) * 2];
        sXY[2 * i + 1] = A.t.xy[((size_t)b * N1 + i) * 2 + 1];
        sDem[i] = CVRP ? A.t.demand[(size_t)b * N1 + i] : 0.f;
      }
      pK = sK; pV = sV; pE = sE; pEb = sEb; pXY = sXY; pDem = sDem;
    } else {
      pK = A.t.k + (size_t)b * N1 * E; pV = A.t.v + (size_t)b * N1 * E; pE = reinterpret_cast<const float*>(A.t.e) + (size_t)b * N1 * E;
      pEb = A.t.eb + (size_t)b * N1; pXY = A.t.xy + (size_t)b * N1 * 2;
      pDem = CVRP ? A.t.demand + (size_t)b * N1 : A.t.eb;
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
      sLogp[r] = 0.f;
    }
    for (int i = tid; i < A.MT * W; i += RT) {
      const int r = i / W, w = i % W;
      sVis[i] = 0u;
      sMask[i] = (A.single_step && r < nrows) ? A.st_mask[((size_t)b * A.M + row0 + r) * W + w] : 0u;
    }
    if (RESIDENT) {
      mbar_wait(bar, bar_phase);
      bar_phase ^= 1;
    }
    __syncthreads();

    // ---- the construction loop ----------------------------------------------------------------
    int t = 0;
    for (;; ++t) {
      const bool forced = !A.single_step && (t < 1 + DEP);
      PHASE_T0();
      if (!forced) {
        // ================= phase A: multi-head attention, thread = (row, head) ====================
        const int full_blocks = nrows >> 5, tail = nrows & 31;
        const int n_units = H * full_blocks + ((H * tail + 31) >> 5);
        for (int u = warp; u < n_units; u += RW) {
          int r, h;
          bool act;
          if (u < H * full_blocks) {
            h = u / full_blocks; r = (u % full_blocks) * 32 + lane; act = true;
          } else {
            int pi = (u - H * full_blocks) * 32 + lane;
            act = pi < H * tail;
            h = act ? pi / tail : 0;
            r = act ? full_blocks * 32 + pi % tail : 0;
          }
          act = act && !sFin[r];
          // q and o live as float2 pairs: the dot products and the p.V update run on packed FFMA2 (sm_100
          // fma.rn.f32x2: two IEEE fp32 FMAs per instruction, half the issue slots of scalar FFMA)
          float2 q2[D / 2], o2[D / 2];
          if (act) {
            const int cur = sCur[r];
            const float4* qp = reinterpret_cast<const float4*>(A.t.qtab + ((size_t)b * N1 + cur) * E + h * D);
            const float ld = sLoad[r];
#pragma unroll
            for (int d4 = 0; d4 < D / 4; ++d4) {
              float4 v4 = __ldg(qp + d4);
              if (CVRP) {
                float4 wl = *reinterpret_cast<const float4*>(sWL + h * D + d4 * 4);
                v4.x = fmaf(ld, wl.x, v4.x); v4.y = fmaf(ld, wl.y, v4.y);
                v4.z = fmaf(ld, wl.z, v4.z); v4.w = fmaf(ld, wl.w, v4.w);
              } else {
                float4 f4 = __ldg(reinterpret_cast<const float4*>(A.t.qfirst + ((size_t)b * N1 + sFirst[r]) * E + h * D) + d4);
                v4.x = f4.x + v4.x; v4.y = f4.y + v4.y; v4.z = f4.z + v4.z; v4.w = f4.w + v4.w;
              }
              q2[d4 * 2] = make_float2(v4.x, v4.y);
              q2[d4 * 2 + 1] = make_float2(v4.z, v4.w);
            }
          } else {
#pragma unroll
            for (int d = 0; d < D / 2; ++d) q2[d] = make_float2(0.f, 0.f);
          }
#pragma unroll
          for (int d = 0; d < D / 2; ++d) o2[d] = make_float2(0.f, 0.f);
          float m = -INFINITY, l = 0.f;
          const float* kp = pK + h * D;
          const float* vp = pV + h * D;
          // K is pre-scaled by log2(e)/sqrt(D): scores live in the log2 domain, weights are 2^(s-m).
          // Only nodes that at least one lane of the warp still needs are visited (warp-uniform loop).
          for (int w = 0; w < W; ++w) {
            const uint32_t mw = act ? sMask[r * W + w] : FULL;
            const int nb = N1 - w * 32;
            const uint32_t lim = nb >= 32 ? FULL : ((1u << nb) - 1u);
            uint32_t bits = __reduce_or_sync(FULL, ~mw) & lim;
            while (bits) {
              // NK nodes per iteration: all score dot products are in flight before the softmax update
              constexpr int NK = 4;
              int jb[NK];
              bool uu[NK];
              float2 sc2[NK];
#pragma unroll
              for (int n = 0; n < NK; ++n) {
                const bool have = bits != 0;
                jb[n] = have ? __ffs(bits) - 1 : jb[0];
                uu[n] = have && !((mw >> jb[n]) & 1u);
                bits &= bits - 1;
                sc2[n] = make_float2(0.f, 0.f);
              }
#pragma unroll
              for (int d4 = 0; d4 < D / 4; ++d4) {
#pragma unroll
                for (int n = 0; n < NK; ++n) {
                  const float4* kr = reinterpret_cast<const float4*>(kp + (size_t)(w * 32 + jb[n]) * E) + d4;
                  const float4 kk = RESIDENT ? *kr : __ldg(kr);
                  sc2[n] = __ffma2_rn(q2[d4 * 2], make_float2(kk.x, kk.y), sc2[n]);
                  sc2[n] = __ffma2_rn(q2[d4 * 2 + 1], make_float2(kk.z, kk.w), sc2[n]);
                }
              }
              float sc[NK];
              float smax = -INFINITY;
#pragma unroll
              for (int n = 0; n < NK; ++n) {
                sc[n] = sc2[n].x + sc2[n].y;
                smax = fmaxf(smax, uu[n] ? sc[n] : -INFINITY);
              }
              if (smax > m + 12.f) {          // lazy rescale of the running softmax reference
                const float c = exp2f(m - smax);
                l *= c;
#pragma unroll
                for (int d = 0; d < D / 2; ++d) o2[d] = __fmul2_rn(o2[d], make_float2(c, c));
                m = smax;
              }
              float pp[NK];
#pragma unroll
              for (int n = 0; n < NK; ++n) { pp[n] = uu[n] ? exp2f(sc[n] - m) : 0.f; l += pp[n]; }
              if (smax != -INFINITY) {
#pragma unroll
                for (int d4 = 0; d4 < D / 4; ++d4) {
#pragma unroll
                  for (int n = 0; n < NK; ++n) {
                    const float4* vr = reinterpret_cast<const float4*>(vp + (size_t)(w * 32 + jb[n]) * E) + d4;
                    const float4 vv = RESIDENT ? *vr : __ldg(vr);
                    const float2 p2 = make_float2(pp[n], pp[n]);
                    o2[d4 * 2] = __ffma2_rn(p2, make_float2(vv.x, vv.y), o2[d4 * 2]);
                    o2[d4 * 2 + 1] = __ffma2_rn(p2, make_float2(vv.z, vv.w), o2[d4 * 2 + 1]);
                  }
                }
              }
            }
          }
          if (act) {
            const float inv = 1.f / l;
            float o[D];
#pragma unroll
            for (int d = 0; d < D / 2; ++d) { o[2 * d] = o2[d].x; o[2 * d + 1] = o2[d].y; }
            if (RESIDENT) {
              // fp16 hi/lo A operand of the score MMA: row r, columns h*16 .. h*16+15 = k-chunks 2h, 2h+1
              uint32_t hw[8], lw[8];
#pragma unroll
              for (int d2 = 0; d2 < D / 2; ++d2) {
                __half h0, l0, h1, l1;
                umma::split_f16(o[2 * d2] * inv, h0, l0);
                umma::split_f16(o[2 * d2 + 1] * inv, h1, l1);
                hw[d2] = (uint32_t)__half_as_ushort(h0) | ((uint32_t)__half_as_ushort(h1) << 16);
                lw[d2] = (uint32_t)__half_as_ushort(l0) | ((uint32_t)__half_as_ushort(l1) << 16);
              }
              uint8_t* ah = reinterpret_cast<uint8_t*>(sO) + (2 * h) * 1024 + (r >> 3) * 128 + (r & 7) * 16;
              *reinterpret_cast<uint4*>(ah) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
              *reinterpret_cast<uint4*>(ah + 1024) = make_uint4(hw[4], hw[5], hw[6], hw[7]);
              *reinterpret_cast<uint4*>(ah + A_HALF) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
              *reinterpret_cast<uint4*>(ah + A_HALF + 1024) = make_uint4(lw[4], lw[5], lw[6], lw[7]);
            } else {
              float4* op = reinterpret_cast<float4*>(sO + r * E + h * D);
#pragma unroll
              for (int d4 = 0; d4 < D / 4; ++d4)
                op[d4] = make_float4(o[d4 * 4] * inv, o[d4 * 4 + 1] * inv, o[d4 * 4 + 2] * inv, o[d4 * 4 + 3] * inv);
            }
          }
        }
        if (RESIDENT) umma::fence_async_smem();     // generic-proxy operand writes -> tensor-core reads
        PHASE_MARK(0);
        __syncthreads();
        PHASE_MARK(1);
        if (RESIDENT && tid == 0) {
          // scores D[row][node] = o . E'  as  A_hi B_hi + A_hi B_lo + A_lo B_hi  (tcgen05, fp32 accumulate in TMEM)
          umma::fence_after_sync();
          const uint32_t idesc = umma::make_idesc_f16(128, N1p);
          const uint32_t a0 = umma::smem_addr(sO), b0 = umma::smem_addr(sm + L.e);
          const uint32_t lboB = (uint32_t)N1p * 16u, bhalf = (uint32_t)N1p * 256u;
          bool accum = false;
#pragma unroll
          for (int term = 0; term < 3; ++term) {
            const uint32_t aa = a0 + (term == 2 ? A_HALF : 0), bb = b0 + (term == 1 ? bhalf : 0);
#pragma unroll
            for (int ks = 0; ks < E / 16; ++ks) {
              // cross terms accumulate separately: added into the large hi*hi sums they would be truncated
              umma::mma_f16_ss(tmem_d + (term ? 128u : 0u), umma::make_desc(aa + ks * 2048, 1024, 128),
                               umma::make_desc(bb + ks * 2 * lboB, lboB, 128), idesc, accum && !(term == 1 && ks == 0));
              accum = true;
            }
          }
          umma::commit(bar_mma);
        }
      }

      // ================= phase B + C: warp = 4 rows ==============================================
      const int r0 = warp * 4;
      const bool own = r0 < nrows;
      const int rq = lane >> 3, s8 = lane & 7;         // octet (row within the warp), sub-lane
      const int myr = own ? min(r0 + rq, nrows - 1) : 0;
      const bool row_ok = own && (r0 + rq) < nrows;
      int warp_live = 0;
      // B1 results: penalty + local score of this lane's neighbour entries (rank p = s8 + 8 e)
      float addv[MAXE];
      int node[MAXE];
      int np = 0;
      bool rlive = false, any_live = false;
      if (own && !forced) {
        rlive = row_ok && !sFin[myr];
        any_live = __any_sync(FULL, rlive);
        if (any_live) {
          // ---- B1: local policy, octet of lanes per row --------------------------------------------
          uint16_t* ids = reinterpret_cast<uint16_t*>(sm + L.ids) + warp * 4 * KT_MAX + rq * KT_MAX;
          const int cur = sCur[myr];
          const float ldv = sLoad[myr];
          const float xc = pXY[2 * cur], yc = pXY[2 * cur + 1];
          const int NL = N1 - DEP, kloc = A.k_local;
          const uint32_t* mrow = sMask + myr * W;
          int cnt = 0;
          // neighbour walk: first k valid entries of the distance-presorted list of `cur`
          if (RESIDENT) {
            uint4 Lw = make_uint4(0, 0, 0, 0);
            if (rlive) Lw = __ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const uint8_t*>(A.t.nbr) + ((size_t)b * N1 + cur) * ELG_NBR_NODE_BYTES(N1)) + s8);
            const int iters = (NL + 7) >> 3;
#pragma unroll
            for (int it = 0; it < 16; ++it) {
              if (it >= iters) break;
              const uint32_t wsel = it < 4 ? Lw.x : (it < 8 ? Lw.y : (it < 12 ? Lw.z : Lw.w));
              const int id = (wsel >> ((it & 3) * 8)) & 0xff;
              const int e = it * 8 + s8;
              const bool valid = rlive && e < NL && cnt < kloc && !((mrow[id >> 5] >> (id & 31)) & 1u);
              const uint32_t bal = __ballot_sync(FULL, valid);
              const uint32_t mine = (bal >> (lane & 24)) & 0xffu;
              const int rank = cnt + __popc(mine & ((1u << s8) - 1u));
              if (valid && rank < kloc) ids[rank] = (uint16_t)id;
              cnt += __popc(mine);
              if (__all_sync(FULL, !rlive || cnt >= kloc)) break;
            }
          } else {
            const int stride = (NL + 63) & ~63;          // uint16 entries per node, 64-entry blocks
            const uint16_t* lst = reinterpret_cast<const uint16_t*>(A.t.nbr) + ((size_t)b * N1 + cur) * stride;
            const int iters = stride >> 6;
            for (int it = 0; it < iters; ++it) {
              uint4 Lw = make_uint4(0, 0, 0, 0);
              if (rlive && cnt < kloc) Lw = __ldg(reinterpret_cast<const uint4*>(lst + it * 64) + s8);
              const uint32_t wd[4] = {Lw.x, Lw.y, Lw.z, Lw.w};
              uint32_t vm = 0;
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                const int id = (wd[i >> 1] >> ((i & 1) * 16)) & 0xffff;
                const int e = it * 64 + s8 * 8 + i;
                const bool valid = rlive && cnt < kloc && e < NL && !((mrow[id >> 5] >> (id & 31)) & 1u);
                vm |= (valid ? 1u : 0u) << i;
              }
              const int c = __popc(vm);
              int incl = c;
              int tt = __shfl_up_sync(FULL, incl, 1); if (s8 >= 1) incl += tt;
              tt = __shfl_up_sync(FULL, incl, 2); if (s8 >= 2) incl += tt;
              tt = __shfl_up_sync(FULL, incl, 4); if (s8 >= 4) incl += tt;
              int rank = cnt + incl - c;
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                if ((vm >> i) & 1u) {
                  if (rank < kloc) ids[rank] = (uint16_t)((wd[i >> 1] >> ((i & 1) * 16)) & 0xffff);
                  ++rank;
                }
              }
              cnt += __shfl_sync(FULL, incl, (lane & 24) | 7);
              if (__all_sync(FULL, !rlive || cnt >= kloc)) break;
            }
          }
          const int kk = min(cnt, kloc);
          np = rlive ? kk + DEP : 0;
          __syncwarp();
          // features of this lane's entries.  Resident instances gather (distance, angle) from the pair table that
          // neighbour_kernel wrote next to the lists; streaming instances compute them here.
          const float2* feat = reinterpret_cast<const float2*>(reinterpret_cast<const uint8_t*>(A.t.nbr) +
                                                               ((size_t)b * N1 + cur) * ELG_NBR_NODE_BYTES(N1) + ELG_NBR_STRIDE);
          float dmax = 0.f;
          if (kk > 0) {
            const int nl = ids[kk - 1];
            dmax = RESIDENT ? __ldg(feat + nl).x : dist2(xc - pXY[2 * nl], yc - pXY[2 * nl + 1]);
          }
          const float r0d = CVRP ? (dmax != 0.f ? 1.f / (dmax + 1e-6f) : 1.f) : 1.f / (dmax + 1e-6f);      // cur_dist / (max + 1e-6)
          const float r1d = dmax != 0.f ? 1.f / dmax : 1.f;        // cvrp penalty -d / dmax (no eps, CVRP/models.py:380,403)
          const float rld = 1.f / ldv;
          float f0[MAXE], f1[MAXE], f2[MAXE];
#pragma unroll
          for (int e = 0; e < MAXE; ++e) {
            const int p = s8 + 8 * e;
            f0[e] = f1[e] = f2[e] = addv[e] = 0.f;
            node[e] = 0;
            if (p < np && !(DEP && p == 0)) {
              const int nd = ids[p - DEP];
              node[e] = nd;
              float dd, th;
              if (RESIDENT) {
                const float2 ft = __ldg(feat + nd);
                dd = ft.x; th = ft.y;
              } else {
                const float xn = pXY[2 * nd], yn = pXY[2 * nd + 1];
                dd = dist2(xc - xn, yc - yn);
                th = atan2f(yn - yc, xn - xc);
              }
              f0[e] = dd * r0d;
              f1[e] = th;
              if (CVRP) {
                addv[e] = -(dd * r1d);                             // distance penalty
                f2[e] = pDem[nd] * rld;
              } else {
                addv[e] = -f0[e];
              }
            }
          }
          // 4-head attention of the constant query over the local sequence.  Per head the octet reduces
          // (sum, g0..2) to every lane and the 8 value columns reduce-scatter, so lane d ends up owning ol[h*8 + d].
          float olh[LH];
#pragma unroll
          for (int h = 0; h < LH; ++h) {
            const float u0 = sU[h * 4], u1 = sU[h * 4 + 1], u2 = sU[h * 4 + 2];
            float sc[MAXE];
            float mx = -INFINITY;
#pragma unroll
            for (int e = 0; e < MAXE; ++e) {
              const int p = s8 + 8 * e;
              float v = -INFINITY;
              if (p < np) {
                v = fmaf(u2, f2[e], fmaf(u1, f1[e], u0 * f0[e])) + sT[h * KT_MAX + p];
                if (DEP && p == 0 && (mrow[0] & 1u)) v = -INFINITY;
              }
              sc[e] = v;
              mx = fmaxf(mx, v);
            }
            mx = octet_max(mx);
            const float mref = mx == -INFINITY ? 0.f : mx;
            float g0 = 0.f, g1 = 0.f, g2 = 0.f, sum = 0.f;
            float vp8[LD];
#pragma unroll
            for (int d = 0; d < LD; ++d) vp8[d] = 0.f;
#pragma unroll
            for (int e = 0; e < MAXE; ++e) {
              const int p = s8 + 8 * e;
              const float w = umma::ex2_raw(sc[e] - mref);          // -inf (masked / beyond np) -> 0
              sum += w;
              g0 = fmaf(w, f0[e], g0); g1 = fmaf(w, f1[e], g1); g2 = fmaf(w, f2[e], g2);
              if (p < np) {
                const float4 va = *reinterpret_cast<const float4*>(sVPE + p * TS + h * LD);
                const float4 vb = *reinterpret_cast<const float4*>(sVPE + p * TS + h * LD + 4);
                vp8[0] = fmaf(w, va.x, vp8[0]); vp8[1] = fmaf(w, va.y, vp8[1]);
                vp8[2] = fmaf(w, va.z, vp8[2]); vp8[3] = fmaf(w, va.w, vp8[3]);
                vp8[4] = fmaf(w, vb.x, vp8[4]); vp8[5] = fmaf(w, vb.y, vp8[5]);
                vp8[6] = fmaf(w, vb.z, vp8[6]); vp8[7] = fmaf(w, vb.w, vp8[7]);
              }
            }
            sum = octet_sum(sum);
            const float inv_s = sum > 0.f ? 1.f / sum : 0.f;
            g0 = octet_sum(g0) * inv_s; g1 = octet_sum(g1) * inv_s; g2 = octet_sum(g2) * inv_s;
            // reduce-scatter of vp8 over the octet: after three exchange steps lane s8 holds the total of vp8[s8]
            float r4[4], r2[2];
            {
              const bool up = (s8 & 4) != 0;
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const float send = up ? vp8[i] : vp8[i + 4];
                const float keep = up ? vp8[i + 4] : vp8[i];
                r4[i] = keep + __shfl_xor_sync(FULL, send, 4);
              }
            }
            {
              const bool up = (s8 & 2) != 0;
#pragma unroll
              for (int i = 0; i < 2; ++i) {
                const float send = up ? r4[i] : r4[i + 2];
                const float keep = up ? r4[i + 2] : r4[i];
                r2[i] = keep + __shfl_xor_sync(FULL, send, 2);
              }
            }
            const bool up1 = (s8 & 1) != 0;
            const float vps = ((up1 ? r2[1] : r2[0]) + __shfl_xor_sync(FULL, up1 ? r2[0] : r2[1], 1)) * inv_s;
            // ol[c] = (Wv We)[c] . g + (Wv be)[c] + sum_p w_p (Wv PE(p))[c],  c = h*8 + s8
            const float4 a4 = *reinterpret_cast<const float4*>(sA + (h * LD + s8) * 4);
            olh[h] = fmaf(a4.z, g2, fmaf(a4.y, g1, a4.x * g0)) + a4.w + vps;
          }
          // z = ZW^T ol + ZB (3 feature weights + constant), partial over this lane's four ol, then octet sum
          float z0 = 0.f, z1 = 0.f, z2 = 0.f, c0 = 0.f;
#pragma unroll
          for (int h = 0; h < LH; ++h) {
            const float4 zw = *reinterpret_cast<const float4*>(sZW + (h * LD + s8) * 4);
            z0 = fmaf(zw.x, olh[h], z0); z1 = fmaf(zw.y, olh[h], z1);
            z2 = fmaf(zw.z, olh[h], z2); c0 = fmaf(zw.w, olh[h], c0);
          }
          z0 = octet_sum(z0) + sZB[0]; z1 = octet_sum(z1) + sZB[1]; z2 = octet_sum(z2) + sZB[2]; c0 = octet_sum(c0) + sZB[3];
          // positional part PW[p] . ol of this lane's entries: ol broadcast four columns at a time
          float pem[MAXE];
#pragma unroll
          for (int e = 0; e < MAXE; ++e) pem[e] = sPB[min(s8 + 8 * e, KT - 1)];
#pragma unroll
          for (int h = 0; h < LH; ++h) {
#pragma unroll
            for (int dq = 0; dq < 2; ++dq) {
              const float o0 = __shfl_sync(FULL, olh[h], (lane & 24) | (dq * 4 + 0));
              const float o1 = __shfl_sync(FULL, olh[h], (lane & 24) | (dq * 4 + 1));
              const float o2 = __shfl_sync(FULL, olh[h], (lane & 24) | (dq * 4 + 2));
              const float o3 = __shfl_sync(FULL, olh[h], (lane & 24) | (dq * 4 + 3));
#pragma unroll
              for (int e = 0; e < MAXE; ++e) {
                const int p = min(s8 + 8 * e, KT - 1);
                const float4 pw = *reinterpret_cast<const float4*>(sPW + p * TS + h * LD + dq * 4);
                pem[e] = fmaf(pw.w, o3, fmaf(pw.z, o2, fmaf(pw.y, o1, fmaf(pw.x, o0, pem[e]))));
              }
            }
          }
#pragma unroll
          for (int e = 0; e < MAXE; ++e)      // penalty + local score (tables carry the 1/sqrt(32))
            addv[e] += fmaf(f2[e], z2, fmaf(f1[e], z1, f0[e] * z0)) + c0 + pem[e];

        }
      }

      PHASE_MARK(2);
      if (RESIDENT && !forced) {
        // ---- scores TMEM -> shared memory (+ eb): warps of TMEM lane quadrants 0/1 (rows 0..63), 4 column parts --
        if ((warp & 3) < 2) {
          mbar_wait(bar_mma, mma_phase);
          umma::fence_after_sync();
          const int q = warp & 3, part = warp >> 2, cp = N1p >> 2;
          const int row = 32 * q + lane;
          float* srow = sO + row * SS;
          for (int c = part * cp; c < (part + 1) * cp; c += 16) {
            const int cs = max(0, min(c, (part + 1) * cp - 16));
            float v[16], v2[16];
            umma::ld16(tmem_d + ((uint32_t)(32 * q) << 16) + cs, v);
            umma::ld16(tmem_d + ((uint32_t)(32 * q) << 16) + 128 + cs, v2);
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] += v2[i];
            if (row < nrows) {
#pragma unroll
              for (int i = 0; i < 16; ++i) {
                const int col = cs + i;
                if (col >= c && col < (part + 1) * cp && col < N1) srow[col] = v[i] + (sm + L.eb)[col];
              }
            }
          }
          umma::fence_before_sync();
        }
        mma_phase ^= 1;
        PHASE_MARK(3);
        __syncthreads();
        PHASE_MARK(4);
      }

      if (own) {
        int sel[4];
        float selp[4] = {1.f, 1.f, 1.f, 1.f};
        if (forced) {
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int gr = min(row0 + r0 + i, A.M - 1);
            sel[i] = (CVRP && t == 0) ? 0 : A.start_nodes[gr];
          }
        } else {
          float best[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
          int bidx[4] = {0x7fffffff, 0x7fffffff, 0x7fffffff, 0x7fffffff};
          int samp[4] = {-1, -1, -1, -1};
          if (any_live && RESIDENT) {
            // ---- B3 (resident): the octet adds penalty + local to its neighbours' staged scores and publishes a
            //      neighbour bit mask; every other unmasked node gets the default penalty xi
            {
              uint32_t nbw[4] = {0u, 0u, 0u, 0u};
              float* srow = sO + myr * SS;
#pragma unroll
              for (int e = 0; e < MAXE; ++e) {
                const int p = s8 + 8 * e;
                if (p < np) {
                  const int nd = node[e];
                  srow[nd] += addv[e];
                  const uint32_t bit = 1u << (nd & 31);
                  nbw[0] |= (nd >> 5) == 0 ? bit : 0u; nbw[1] |= (nd >> 5) == 1 ? bit : 0u;
                  nbw[2] |= (nd >> 5) == 2 ? bit : 0u; nbw[3] |= (nd >> 5) == 3 ? bit : 0u;
                }
              }
#pragma unroll
              for (int w = 0; w < 4; ++w) {
                nbw[w] |= __shfl_xor_sync(FULL, nbw[w], 1);
                nbw[w] |= __shfl_xor_sync(FULL, nbw[w], 2);
                nbw[w] |= __shfl_xor_sync(FULL, nbw[w], 4);
              }
              if (row_ok && s8 < 4) reinterpret_cast<uint32_t*>(srow)[112 + s8] = s8 == 0 ? nbw[0] : (s8 == 1 ? nbw[1] : (s8 == 2 ? nbw[2] : nbw[3]));
            }
            __syncwarp();
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const int r = r0 + i;
              const bool live = r < nrows && !sFin[min(r, nrows - 1)];
              if (live) {
                const float* srow = sO + r * SS;
                float lg[4];
#pragma unroll
                for (int ch = 0; ch < 4; ++ch) {
                  const int j = lane + 32 * ch;
                  float v = -INFINITY;
                  if (j < N1 && !((sMask[r * W + ch] >> lane) & 1u)) {
                    const bool isnb = (reinterpret_cast<const uint32_t*>(srow)[112 + ch] >> lane) & 1u;
                    v = A.clip * tanhf(isnb ? srow[j] : srow[j] + A.xi);
                  }
                  lg[ch] = v;
                  if (v > best[i]) { best[i] = v; bidx[i] = j; }
                }
                if (A.out_logits) {
                  float* lo = A.out_logits + ((size_t)b * A.M + row0 + r) * N1;
#pragma unroll
                  for (int ch = 0; ch < 4; ++ch)
                    if (lane + 32 * ch < N1) lo[lane + 32 * ch] = lg[ch];
                }
                if (A.mode == ELG_SAMPLE)         // host guarantees N1 <= 128 (one chunk) in this mode
                  sample_row(lg, best[i], A.seed, (unsigned long long)b * A.M + row0 + r,
                             A.single_step ? A.step_id : (unsigned long long)t, lane, samp[i], selp[i]);
              }
            }
          }
          if (any_live && !RESIDENT) {
            // ---- B2 + B3 over chunks of 128 nodes ------------------------------------------------------
          const float* ob = sO + r0 * E;
          float* dense = RESIDENT ? sO + r0 * E : sm + L.dense + warp * 4 * DS;     // [4][DS]
          const int rcl[4] = {0, min(1, nrows - 1 - r0), min(2, nrows - 1 - r0), min(3, nrows - 1 - r0)};
          for (int c0n = 0; c0n < N1; c0n += 128) {
            float acc[4][4];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
              for (int c = 0; c < 4; ++c) acc[i][c] = 0.f;
            int jj[4];
#pragma unroll
            for (int ch = 0; ch < 4; ++ch) jj[ch] = min(c0n + lane + 32 * ch, N1 - 1);
            const int nch = min(4, (N1 - c0n + 31) >> 5);
#pragma unroll 4
            for (int c4 = 0; c4 < E / 4; ++c4) {
              float4 ov[4];
#pragma unroll
              for (int i = 0; i < 4; ++i) ov[i] = *reinterpret_cast<const float4*>(ob + rcl[i] * E + c4 * 4);
#pragma unroll
              for (int ch = 0; ch < 4; ++ch) {
                if (ch < nch) {
                  const float4* ep = reinterpret_cast<const float4*>(pE + (size_t)jj[ch] * E + ((c4 ^ (jj[ch] & 7)) << 2));
                  const float4 ev = RESIDENT ? *ep : __ldg(ep);
#pragma unroll
                  for (int i = 0; i < 4; ++i) {
                    acc[i][ch] = fmaf(ov[i].x, ev.x, acc[i][ch]); acc[i][ch] = fmaf(ov[i].y, ev.y, acc[i][ch]);
                    acc[i][ch] = fmaf(ov[i].z, ev.z, acc[i][ch]); acc[i][ch] = fmaf(ov[i].w, ev.w, acc[i][ch]);
                  }
                }
              }
            }
#pragma unroll
            for (int ch = 0; ch < 4; ++ch) {
              const float ebv = pEb[jj[ch]];
#pragma unroll
              for (int i = 0; i < 4; ++i) acc[i][ch] += ebv;
            }
            __syncwarp();               // resident: every lane is done reading this warp's o rows
            // penalty + local for this chunk: xi by default, depot / neighbours overwritten by their octet
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
              for (int ch = 0; ch < 4; ++ch) dense[i * DS + lane + 32 * ch] = A.xi;
            __syncwarp();
#pragma unroll
            for (int e = 0; e < MAXE; ++e) {
              const int p = s8 + 8 * e;
              const int nd = node[e] - c0n;
              if (p < np && nd >= 0 && nd < 128) dense[rq * DS + nd] = addv[e];
            }
            __syncwarp();
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const int r = r0 + i;
              const bool live = r < nrows && !sFin[min(r, nrows - 1)];
              if (live) {
                float lg[4];
#pragma unroll
                for (int ch = 0; ch < 4; ++ch) {
                  const int j = c0n + lane + 32 * ch;
                  float v = -INFINITY;
                  if (j < N1 && !((sMask[r * W + (j >> 5)] >> lane) & 1u)) v = A.clip * tanhf(acc[i][ch] + dense[i * DS + lane + 32 * ch]);
                  lg[ch] = v;
                  if (v > best[i]) { best[i] = v; bidx[i] = j; }
                }
                if (A.out_logits) {
                  float* lo = A.out_logits + ((size_t)b * A.M + row0 + r) * N1;
#pragma unroll
                  for (int ch = 0; ch < 4; ++ch)
                    if (c0n + lane + 32 * ch < N1) lo[c0n + lane + 32 * ch] = lg[ch];
                }
                if (A.mode == ELG_SAMPLE)         // host guarantees N1 <= 128 (one chunk) in this mode
                  sample_row(lg, best[i], A.seed, (unsigned long long)b * A.M + row0 + r,
                             A.single_step ? A.step_id : (unsigned long long)t, lane, samp[i], selp[i]);
              }
            }
            __syncwarp();
          }
          }
          // ---- first-max argmax across the warp (ties -> lowest index, as torch.argmax); sampling -----
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int r = r0 + i;
            const bool live = r < nrows && !sFin[min(r, nrows - 1)];
            float bv = best[i];
            int bi = bidx[i];
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
              const float ov = __shfl_xor_sync(FULL, bv, off);
              const int oi = __shfl_xor_sync(FULL, bi, off);
              if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
            }
            int choice = live ? bi : 0;
            if (A.mode == ELG_SAMPLE && live && samp[i] >= 0) choice = samp[i];     // else (no node of positive probability): the mode
            sel[i] = choice;
          }
        }

        if (A.single_step) {
          if (lane < 4 && r0 + lane < nrows) {
            const size_t g = (size_t)b * A.M + row0 + r0 + lane;
            int sv = sel[0]; float pv = selp[0];
            if (lane == 1) { sv = sel[1]; pv = selp[1]; }
            if (lane == 2) { sv = sel[2]; pv = selp[2]; }
            if (lane == 3) { sv = sel[3]; pv = selp[3]; }
            A.out_selected[g] = sv;
            if (A.out_prob) A.out_prob[g] = pv;
          }
        } else {
          // ================= phase C: environment step (lanes = nodes for the too-large test) =======
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int r = r0 + i;
            if (r >= nrows) break;
            const int sl = sel[i];
            const int prev = sCur[r];
            const bool was_fin = sFin[r] != 0;
            __syncwarp();     // every lane has read the row state (and its mask words in B3) before lane 0 rewrites it
            bool fin = was_fin;
            float ld = 1.f;
            if (CVRP) {
              const bool at_depot = sl == 0;
              ld = at_depot ? 1.f : sLoad[r] - pDem[sl];
              bool allv = true;
              for (int w = 0; w < W; ++w) {
                uint32_t vw = sVis[r * W + w];
                if (w == (sl >> 5)) vw |= 1u << (sl & 31);
                if (w == 0) vw = at_depot ? (vw | 1u) : (vw & ~1u);
                const int j = w * 32 + lane;
                const uint32_t big = __ballot_sync(FULL, j < N1 && (__fadd_rn(ld, 1e-6f) < pDem[min(j, N1 - 1)]));
                const int nb = N1 - w * 32;
                const uint32_t fullw = nb >= 32 ? FULL : ((1u << nb) - 1u);
                allv = allv && ((vw & fullw) == fullw);
                __syncwarp();
                if (lane == 0) { sVis[r * W + w] = vw; sMask[r * W + w] = vw | big; }
              }
              fin = was_fin || allv;
              __syncwarp();
              if (fin && lane == 0) sMask[r * W] &= ~1u;       // finished rows may stay at the depot
            } else {
              if (lane == 0) {
                const uint32_t vw = sVis[r * W + (sl >> 5)] | (1u << (sl & 31));
                sVis[r * W + (sl >> 5)] = vw;
                sMask[r * W + (sl >> 5)] = vw;
              }
            }
            warp_live |= !fin;
            if (lane == 0) {
              if (t > 0) {
                float seg;
                if (A.t.unscaled) {
                  const float* ux = A.t.unscaled + (size_t)b * N1 * 2;
                  seg = rintf(seglen(ux[2 * prev] - ux[2 * sl], ux[2 * prev + 1] - ux[2 * sl + 1]));
                } else {
                  seg = seglen(pXY[2 * prev] - pXY[2 * sl], pXY[2 * prev + 1] - pXY[2 * sl + 1]);
                }
                sTlen[r] += seg;
              }
              if (!CVRP && t == 0) sFirst[r] = sl;
              sCur[r] = sl;
              sLoad[r] = ld;
              sFin[r] = fin ? 1 : 0;
              if (A.mode == ELG_SAMPLE && !was_fin) sLogp[r] += logf(selp[i]);
              if (t < A.t_max) A.tours[((size_t)b * A.M + row0 + r) * A.t_max + t] = (int16_t)sl;
            }
          }
        }
      }
      PHASE_MARK(5);
      if (A.single_step) break;
      // ---- all rows finished?  (the barrier also publishes the new row state to phase A) ---------
      bool more = __syncthreads_or(warp_live) != 0;
      PHASE_MARK(6);
      if (!CVRP) more = (t + 1) < N1;
      if (!more || t + 1 >= A.t_max) { ++t; break; }
    }

    // ---- epilogue: rewards ---------------------------------------------------------------------
    if (!A.single_step) {
      for (int r = tid; r < nrows; r += RT) {
        float len = sTlen[r];
        if (!CVRP) {                       // close the tour: last -> first
          const int a = sCur[r], f = sFirst[r];
          if (A.t.unscaled) {
            const float* ux = A.t.unscaled + (size_t)b * N1 * 2;
            len += rintf(seglen(ux[2 * a] - ux[2 * f], ux[2 * a + 1] - ux[2 * f + 1]));
          } else {
            len += seglen(pXY[2 * a] - pXY[2 * f], pXY[2 * a + 1] - pXY[2 * f + 1]);
          }
        }
        const size_t g = (size_t)b * A.M + row0 + r;
        A.reward[g] = -len;
        if (A.logp) A.logp[g] = sLogp[r];
      }
      if (tid == 0) A.n_steps[b * A.ns_stride + tile] = t;
    }
    __syncthreads();
  }
  if (RESIDENT) {
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 0) umma::tmem_dealloc(tmem_d, 256);
  }
#ifdef ELG_PHASE_TIMING
  if (tid == 0)
    for (int i = 0; i < 8; ++i) atomicAdd(&g_phase_clk[i], pclk[i]);
#endif
}

// ---- host side ----------------------------------------------------------------------------------
// Resident (K'/V/E' in shared memory for the whole rollout) iff the layout fits with the largest row tile.
// A function of (model, N1) only, because elg_encode must write E' and the neighbour lists in the matching format.
bool rollout_is_resident(const elg_model_desc* d, int N1) {
  if (N1 > N_RES_MAX) return false;
  const int KT = d->local_k + (d->problem == ELG_CVRP ? 1 : 0);
  const int maxe = KT <= 32 ? 4 : (KT <= 48 ? 6 : 8);
  return (size_t)make_layout(N1, MT_MAX, maxe * 8, true).total * sizeof(float) <= 227 * 1024;
}

struct Plan {
  bool resident;
  int maxe, tiles, MT;
  size_t smem;
};

static int make_plan(const elg_model_desc* d, int B, int M, int N1, Plan& p) {
  const int KT = d->local_k + (d->problem == ELG_CVRP ? 1 : 0);
  p.maxe = KT <= 32 ? 4 : (KT <= 48 ? 6 : 8);
  int sms = 148, dev = 0;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  auto tile_rows = [&](int tiles) { return (((M + tiles - 1) / tiles) + 3) & ~3; };
  p.tiles = (M + MT_MAX - 1) / MT_MAX;
  // few aug-instances (library instances: B = 8): use as many row tiles as fit one wave of CTAs
  if (B * p.tiles < sms) {
    int t2 = sms / B;
    int max_tiles = (M + 3) / 4;
    if (t2 > max_tiles) t2 = max_tiles;
    if (t2 > p.tiles) p.tiles = t2;
  }
  p.MT = tile_rows(p.tiles);
  p.tiles = (M + p.MT - 1) / p.MT;
  p.resident = rollout_is_resident(d, N1);      // the same predicate elg_encode used to choose the table formats
  if (p.resident) p.smem = (size_t)make_layout(N1, p.MT, p.maxe * 8, true).total * sizeof(float);
  if (!p.resident) {
    ELG_REQUIRE(N1 <= N_STREAM_MAX, ELG_EUNSUPPORTED, "rollout supports up to %d nodes (got %d)", N_STREAM_MAX, N1);
    p.smem = (size_t)make_layout(N1, p.MT, p.maxe * 8, false).total * sizeof(float);
    while (p.smem > 227 * 1024 && p.MT > 4) {      // huge N: shrink the row tile until the bit masks fit
      p.MT -= 4;
      p.tiles = (M + p.MT - 1) / p.MT;
      p.smem = (size_t)make_layout(N1, p.MT, p.maxe * 8, false).total * sizeof(float);
    }
    ELG_REQUIRE(p.smem <= 227 * 1024, ELG_EUNSUPPORTED, "row state does not fit in shared memory (N1=%d)", N1);
  }
  return ELG_OK;
}

int launch_rollout_tc(const elg_model_desc* d, RolloutArgs& a, cudaStream_t st);
int rollout_tc_tiles(const elg_model_desc* d, int B, int M, int N1, int* mt_out);
int launch_rollout_stc(const elg_model_desc* d, RolloutArgs& a, cudaStream_t st);      // rollout_stc.cu: large instances, streamed tiles
bool rollout_stc_eligible(const elg_model_desc* d, const RolloutArgs& a);

// Tensor-core attention kernel (rollout_tc.cu): resident instances, greedy decoding, and enough aug-instances that
// whole-instance CTAs fill the machine -- or when forced by ELG_FLAG_ATTN_TENSOR; ELG_FLAG_ATTN_FP32 forces this file's kernel.
static bool use_tensor_attention(const elg_model_desc* d, const RolloutArgs& a) {
  if (a.mode != ELG_GREEDY || (d->flags & ELG_FLAG_ATTN_FP32) || !rollout_is_resident(d, a.N1)) return false;
  const int tiles = rollout_tc_tiles(d, a.B, a.M, a.N1, nullptr);
  if (tiles <= 0) return false;
  if (d->flags & ELG_FLAG_ATTN_TENSOR) return true;
  int sms = 148, dev = 0;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  return a.B * tiles >= sms;      // few aug-instances (library runs, B = 8): small row tiles of the fp32-pipe kernel fill the machine better
}

static int launch_rollout(const elg_model_desc* d, RolloutArgs& a, cudaStream_t st) {
  if (use_tensor_attention(d, a)) return launch_rollout_tc(d, a, st);
  if (rollout_stc_eligible(d, a)) return launch_rollout_stc(d, a, st);
  Plan p;
  int rc = make_plan(d, a.B, a.M, a.N1, p);
  if (rc) return rc;
  ELG_REQUIRE(a.mode == ELG_GREEDY || a.N1 <= 128, ELG_EUNSUPPORTED, "sampling is implemented for up to 128 nodes (got %d)", a.N1);
  a.tiles = p.tiles;
  a.MT = p.MT;
  int dev = 0, sms = 148;
  ELG_CUDA_OK(cudaGetDevice(&dev));
  ELG_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int work = a.B * a.tiles;
  const int grid = work < sms ? work : sms;
#define ELG_RK(P, ME, RES)                                                                                   \
  do {                                                                                                       \
    ELG_CUDA_OK(cudaFuncSetAttribute(rollout_kernel<P, ME, RES>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                     (int)p.smem));                                                          \
    rollout_kernel<P, ME, RES><<<grid, RT, p.smem, st>>>(a);                                                 \
  } while (0)
#define ELG_RK_ME(P, RES)                                                                                    \
  do {                                                                                                       \
    if (p.maxe == 4) ELG_RK(P, 4, RES); else if (p.maxe == 6) ELG_RK(P, 6, RES); else ELG_RK(P, 8, RES);      \
  } while (0)
  if (d->problem == ELG_CVRP) {
    if (p.resident) ELG_RK_ME(ELG_CVRP, true); else ELG_RK_ME(ELG_CVRP, false);
  } else {
    if (p.resident) ELG_RK_ME(ELG_TSP, true); else ELG_RK_ME(ELG_TSP, false);
  }
#undef ELG_RK_ME
#undef ELG_RK
  ELG_LAUNCH_OK();
  return ELG_OK;
}


}  // namespace elg

using namespace elg;

extern "C" {

#ifdef ELG_PHASE_TIMING
int elg_debug_phase_clocks(unsigned long long* out8, int reset) {
  ELG_CUDA_OK(cudaMemcpyFromSymbol(out8, g_phase_clk, sizeof(unsigned long long) * 8));
  if (reset) { unsigned long long z[8] = {0}; ELG_CUDA_OK(cudaMemcpyToSymbol(g_phase_clk, z, sizeof(z))); }
  return ELG_OK;
}
#endif

int elg_rollout_tiles(const elg_model_desc* d, int B, int M, int N1) {
  if (check_desc(d) || M <= 0 || B <= 0) return -1;
  Plan p;
  if (make_plan(d, B, M, N1, p)) return -1;
  const int tc = rollout_tc_tiles(d, B, M, N1, nullptr);      // whichever kernel runs, n_steps is strided by this value
  return p.tiles > tc ? p.tiles : tc;
}

static int fill_common(const elg_model_desc* d, const float* derived, const elg_tables* t, int B, int M, int N1,
                       RolloutArgs& a) {
  int rc = check_desc(d);
  if (rc) return rc;
  ELG_REQUIRE(derived && t, ELG_EINVAL, "NULL pointer");
  ELG_REQUIRE(B > 0 && M > 0 && N1 > 1, ELG_EINVAL, "bad sizes B=%d M=%d N1=%d", B, M, N1);
  ELG_REQUIRE(t->xy && t->k && t->v && t->e && t->eb && t->qtab && t->nbr, ELG_EINVAL, "elg_tables has NULL members");
  ELG_REQUIRE(d->problem == ELG_TSP ? t->qfirst != nullptr : t->demand != nullptr, ELG_EINVAL,
              "tsp needs qfirst, cvrp needs demand");
  memset(&a, 0, sizeof(a));
  a.t = *t;
  a.derived = derived;
  a.problem = d->problem;
  a.B = B; a.M = M; a.N1 = N1;
  a.k_local = d->local_k;
  a.xi = d->xi; a.clip = d->clip;
  return ELG_OK;
}

int elg_rollout(const elg_model_desc* d, const float* derived, const elg_tables* t, int B, int M, int N1,
                const int32_t* start_nodes, int mode, uint64_t seed, int t_max, int16_t* tours, float* reward,
                int32_t* n_steps, float* logp, int32_t* work_counter, void* stream) {
  RolloutArgs a;
  int rc = fill_common(d, derived, t, B, M, N1, a);
  if (rc) return rc;
  ELG_REQUIRE(start_nodes && tours && reward && n_steps && work_counter, ELG_EINVAL, "NULL output/state pointer");
  ELG_REQUIRE(mode == ELG_GREEDY || mode == ELG_SAMPLE, ELG_EINVAL, "unknown mode %d", mode);
  const int need = d->problem == ELG_CVRP ? 2 * N1 + 2 : N1;
  ELG_REQUIRE(t_max >= need, ELG_EINVAL, "t_max=%d too small, need >= %d", t_max, need);
  a.start_nodes = start_nodes; a.mode = mode; a.seed = seed; a.t_max = t_max;
  a.tours = tours; a.reward = reward; a.n_steps = n_steps; a.logp = logp; a.work_counter = work_counter;
  a.ns_stride = elg_rollout_tiles(d, B, M, N1);
  return launch_rollout(d, a, (cudaStream_t)stream);
}

int elg_decode_step(const elg_model_desc* d, const float* derived, const elg_tables* t, int B, int M, int N1,
                    const int32_t* cur, const float* load, const int32_t* first, const uint32_t* mask_bits,
                    int mode, uint64_t seed, uint64_t step, int32_t* selected, float* prob, float* logits,
                    void* stream) {
  RolloutArgs a;
  int rc = fill_common(d, derived, t, B, M, N1, a);
  if (rc) return rc;
  ELG_REQUIRE(cur && mask_bits && selected, ELG_EINVAL, "NULL state pointer");
  ELG_REQUIRE(d->problem == ELG_TSP ? first != nullptr : load != nullptr, ELG_EINVAL, "tsp needs first, cvrp needs load");
  ELG_REQUIRE(mode == ELG_GREEDY || mode == ELG_SAMPLE, ELG_EINVAL, "unknown mode %d", mode);
  a.mode = mode; a.seed = seed; a.single_step = 1; a.step_id = step; a.t_max = 1;
  a.st_cur = cur; a.st_load = load; a.st_first = first; a.st_mask = mask_bits;
  a.out_selected = selected; a.out_prob = prob; a.out_logits = logits;
  a.work_counter = nullptr;   // static CTA -> work mapping
  return launch_rollout(d, a, (cudaStream_t)stream);
}

}  // extern "C"
