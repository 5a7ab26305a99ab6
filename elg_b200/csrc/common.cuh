// Shared definitions for the ELG B200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <math.h>
#include "../../include/elg_b200.h"

namespace elg {

// Fixed architecture of the released ELG configuration (config.yml model_params).
constexpr int E = 128;    // embedding_dim
constexpr int H = 8;      // head_num
constexpr int D = 16;     // qkv_dim
constexpr int LE = 32;    // local_att_hidden_dim
constexpr int LH = 4;     // local_att_head_num
constexpr int LD = 8;     // local_att_qkv_dim
constexpr int KT_MAX = 64;  // max local sequence length (local_k + depot)

// ---- derived-table layout (floats), produced by elg_prepare_model --------------------------
constexpr int DER_WQN = 0;                    // [E][E]  node part of Wq_last
constexpr int DER_WL = DER_WQN + E * E;       // [E]     load column of Wq_last (cvrp) / zeros
constexpr int DER_WQF = DER_WL + E;           // [E][E]  Wq_first (tsp) / zeros
constexpr int DER_WK4 = DER_WQF + E * E;      // [E][E]  Wk * log2(e) / sqrt(D)
constexpr int DER_WET = DER_WK4 + E * E;      // [E][E]  WET[i][k] = Wo[k][i] / sqrt(E)
constexpr int DER_BE = DER_WET + E * E;       // [E]     bo / sqrt(E)
constexpr int DER_LOC = DER_BE + E;           // local-policy tables
constexpr int LOC_U = 0;                      // [LH][4]      u_h[f]      (x log2 e)
constexpr int LOC_T = LOC_U + LH * 4;         // [LH][KT_MAX] t_h[p]      (x log2 e)
constexpr int LOC_A = LOC_T + LH * KT_MAX;    // [LE][4]      (Wv We)[c][f]
constexpr int LOC_CV = LOC_A + LE * 4;        // [LE]         Wv be
constexpr int LOC_VPE = LOC_CV + LE;          // [KT_MAX][LE] Wv PE(p)
constexpr int LOC_PE = LOC_VPE + KT_MAX * LE; // [KT_MAX][LE] PE(p)
constexpr int LOC_WCT = LOC_PE + KT_MAX * LE; // [LE][LE]     WCT[c][c'] = Wo_l[c'][c]
constexpr int LOC_BC = LOC_WCT + LE * LE;     // [LE]
constexpr int LOC_WE = LOC_BC + LE;           // [LE][4]      We[c][f]
constexpr int LOC_BE = LOC_WE + LE * 4;       // [LE]
// everything downstream of the local attention output ol is linear in it; folded for rollout_tc.cu (x 1/sqrt(LE)):
//   local score of entry p = f_p . z + z3 + PW[p] . ol + PB[p],   z = ZW^T ol + ZB
constexpr int LOC_PW = LOC_BE + LE;           // [KT_MAX][LE] sum_c' PE(p)[c'] Wo_l[c'][c] / sqrt(LE)
constexpr int LOC_PB = LOC_PW + KT_MAX * LE;  // [KT_MAX]     PE(p) . bo_l / sqrt(LE)
constexpr int LOC_ZW = LOC_PB + KT_MAX;       // [LE][4]      f < 3: sum_c' We[c'][f] Wo_l[c'][c];  f = 3: sum_c' be[c'] Wo_l[c'][c]   (/ sqrt(LE))
constexpr int LOC_ZB = LOC_ZW + LE * 4;       // [4]          We^T bo_l, be . bo_l                                                    (/ sqrt(LE))
// the two local-policy contractions of rollout_tc.cu as tcgen05 B operands (fp16 hi | lo, K-major core matrices, one
// 32-bit word per float slot):
//   OP1 per local head h: rows n < 8: (Wv PE(p))[h*8 + n] over k = p < KT_MAX (rows 8..15 zero); 16 x KT_MAX, LBO 256 B
//   OP2: rows n < K1: PW[n][k]; rows K1..K1+3: ZW[k][n - K1]; zero up to N2 = ceil16(K1 + 4); N2 x 32, LBO N2 * 16 B
constexpr int LOC_OP1 = LOC_ZB + 4;           // [LH][hi 16*KT_MAX halves | lo]
constexpr int LOC_OP2 = LOC_OP1 + LH * KT_MAX * 16;   // [hi N2*32 halves | lo], at most N2 = 80
constexpr int LOC_TOTAL = LOC_OP2 + 80 * LE;
constexpr int DER_FOLD_TOTAL = DER_LOC + LOC_TOTAL;
// After the folds: every GEMM weight matrix pre-split into fp16 hi/lo tcgen05 B-operand tiles (one float's worth
// of bytes per weight element).  Matrix W[N][K] -> tiles (n/128, k/64), each [hi 16 KB | lo 16 KB] in the K-major
// core-matrix layout of umma.cuh.  Order: per layer {Wq|Wk|Wv (3E x E), Wo, W1, W2}; then K' weights, Wv_dec,
// Wq_node, Wq_first.
__host__ __device__ inline long long split_layer_floats(int ff) { return 3LL * E * E + (long long)E * E + 2LL * ff * E; }
__host__ __device__ inline long long split_off_layer(int l, int ff) { return DER_FOLD_TOTAL + l * split_layer_floats(ff); }
__host__ __device__ inline long long split_off_dec(int layers, int ff) { return DER_FOLD_TOTAL + layers * split_layer_floats(ff); }
__host__ __device__ inline long long derived_total(int layers, int ff) { return split_off_dec(layers, ff) + 4LL * E * E; }

// ---- activations kept by elg_encode_train for the backward pass (floats; rows = B * N1) ---------------
// per layer: xin [E] | qkv [3E] | att [E] | t1 = xin + att Wo^T + bo [E] | x1 = IN(t1) [E] | hid [ff] | t2 = x1 + ffn [E];
// after the layers: plain fp32 score matrix E' = enc Wo-fold / sqrt(E) [rows][E].
enum { TS_XIN = 0, TS_QKV = 1, TS_ATT = 2, TS_T1 = 3, TS_X1 = 4, TS_HID = 5, TS_T2 = 6 };
__host__ __device__ inline long long train_layer_floats(int ff) { return 8LL * E + ff; }
__host__ __device__ inline long long train_saved_off(int l, long long rows, int ff, int which) {
  const long long part[7] = {0, E, 4LL * E, 5LL * E, 6LL * E, 7LL * E, 7LL * E + ff};
  return ((long long)l * train_layer_floats(ff) + part[which]) * rows;
}
__host__ __device__ inline long long train_saved_eplain(int layers, long long rows, int ff) { return (long long)layers * train_layer_floats(ff) * rows; }
__host__ __device__ inline long long train_saved_total(int layers, long long rows, int ff) { return train_saved_eplain(layers, rows, ff) + rows * E; }

// ---- error plumbing -------------------------------------------------------------------------
void set_error(const char* fmt, ...);
void count_launch(int n = 1);
int check_desc(const elg_model_desc* d);

#define ELG_CUDA_OK(call)                                                        \
  do {                                                                           \
    cudaError_t _e = (call);                                                     \
    if (_e != cudaSuccess) {                                                     \
      elg::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return (int)_e;                                                            \
    }                                                                            \
  } while (0)

#define ELG_LAUNCH_OK()                                                          \
  do {                                                                           \
    elg::count_launch();                                                         \
    cudaError_t _e = cudaGetLastError();                                         \
    if (_e != cudaSuccess) {                                                     \
      elg::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), __FILE__, __LINE__); \
      return (int)_e;                                                            \
    }                                                                            \
  } while (0)

#define ELG_REQUIRE(cond, code, ...)                                             \
  do {                                                                           \
    if (!(cond)) {                                                               \
      elg::set_error(__VA_ARGS__);                                               \
      return (code);                                                             \
    }                                                                            \
  } while (0)

// ---- device helpers -------------------------------------------------------------------------
// Euclidean distance exactly as torch's CPU `norm(p=2)` accumulates a 2-vector:
// acc = dx*dx (rounded); acc = fma(dy, dy, acc); sqrt.  Used everywhere a distance is needed so
// that neighbour ordering, features and tour lengths all see the same value.
__device__ __forceinline__ float dist2(float dx, float dy) {
  return __fsqrt_rn(__fmaf_rn(dy, dy, __fmul_rn(dx, dx)));
}

// Tour segment length exactly as the reference's reward: ((a-b)**2).sum(-1).sqrt() -- two rounded
// squares, one rounded add (no fused multiply-add), then sqrt (CVRP/CVRPEnv.py:261, TSP/TSPEnv.py:168).
__device__ __forceinline__ float seglen(float dx, float dy) {
  return __fsqrt_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)));
}

// ---- local search (two_opt.cu, cvrp_ls.cu, tsp_ls.cu) ----------------------------------------------------
constexpr float LS_MIN_GAIN = -1e-6f;  // a move is applied only if its gain is below this

// d(a, b) of nodes a, b: the reward's seglen, rint()-ed under the library metric
__device__ __forceinline__ float edge_len(const float2* __restrict__ xy, int a, int b, int round_edges) {
  const float2 p = xy[a], q = xy[b];
  const float d = seglen(p.x - q.x, p.y - q.y);
  return round_edges ? rintf(d) : d;
}

// (gain, key) ordered by gain, then by key: torch.argmin's first-index tie-break.  K is int, or unsigned where the keys
// can pass 2^31-1 (cvrp_ls.cu with segment moves).
template <typename K>
__device__ __forceinline__ bool gain_better(float g, K key, float bg, K bkey) {
  return g < bg || (g == bg && key < bkey);
}

// CTA-wide minimum of every thread's (bg, bkey) under gain_better, returned to every thread.  red_g / red_k hold one
// entry per warp; a barrier must separate the reads here from the next writes to them.
template <typename K>
__device__ __forceinline__ void cta_min_gain(float& bg, K& bkey, float* red_g, K* red_k) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  for (int o = 16; o > 0; o >>= 1) {
    const float g = __shfl_xor_sync(0xffffffffu, bg, o);
    const K k = __shfl_xor_sync(0xffffffffu, bkey, o);
    if (gain_better(g, k, bg, bkey)) { bg = g; bkey = k; }
  }
  if (lane == 0) { red_g[warp] = bg; red_k[warp] = bkey; }
  __syncthreads();
  bg = red_g[0]; bkey = red_k[0];
  for (int w = 1; w < nwarps; ++w)
    if (gain_better(red_g[w], red_k[w], bg, bkey)) { bg = red_g[w]; bkey = red_k[w]; }
}

// reverses row[a..b] with the threads of the CTA; the caller synchronises
__device__ __forceinline__ void reverse_span(int16_t* row, int a, int b) {
  for (int k = threadIdx.x; k < (b - a + 1) / 2; k += blockDim.x) {
    const int16_t t = row[a + k]; row[a + k] = row[b - k]; row[b - k] = t;
  }
}

// xy instance of row r: inst[r], else 0 when one instance is shared by all rows, else r
__device__ __forceinline__ int ls_instance(const int32_t* __restrict__ inst, int Bxy, int r) {
  return inst ? inst[r] : (Bxy == 1 ? 0 : r);
}

// Result of row r: the n positions of `tour` back to `row`; length[r] = edge[0..n-1] summed in the order of
// tour_length_kernel (sequential from the edge leaving position 0, on thread 0); iterations[r] = moves.  tour and edge
// must be final (behind a barrier); the closing barrier lets the next row reuse shared memory.  nthr is the kernel's
// blockDim.x: reading it again here costs tsp_ls_kernel a register.
__device__ __forceinline__ void ls_store_row(const int16_t* tour, const float* edge, int n, int16_t* __restrict__ row,
                                             int r, int moves, float* __restrict__ length,
                                             int32_t* __restrict__ iterations, int nthr) {
  for (int p = threadIdx.x; p < n; p += nthr) row[p] = tour[p];
  if (threadIdx.x == 0) {
    float sum = 0.f;
    for (int p = 0; p < n; ++p) sum += edge[p];
    length[r] = sum;
    iterations[r] = moves;
  }
  __syncthreads();
}

// The checks every local-search entry point makes; `what` names the search in the messages.
inline int ls_check_args(const char* what, const float* xy, int Bxy, int N1, const int32_t* inst, const int16_t* tours,
                         int R, int max_iterations, const int32_t* iterations, const float* length) {
  ELG_REQUIRE(N1 > 0 && R >= 0 && Bxy > 0, ELG_EINVAL, "bad sizes N1=%d R=%d Bxy=%d", N1, R, Bxy);
  ELG_REQUIRE(N1 <= ELG_MAX_NODES, ELG_EUNSUPPORTED, "%s supports up to %d nodes (got %d)", what, ELG_MAX_NODES, N1);
  ELG_REQUIRE(max_iterations >= 0, ELG_EINVAL, "max_iterations must be >= 0 (got %d)", max_iterations);
  ELG_REQUIRE(xy && tours && iterations && length, ELG_EINVAL, "NULL pointer");
  ELG_REQUIRE(inst || Bxy == 1 || Bxy == R, ELG_EINVAL, "without inst the xy batch must be 1 or R (Bxy=%d, R=%d)", Bxy, R);
  return ELG_OK;
}

// Persistent launch of a local-search kernel over R rows: one CTA per row at a time, 256 threads for rows of at most
// 512 positions and 512 above, as many CTAs as fit on the device (at most R).
template <typename... Params, typename... Args>
int ls_launch(void (*kernel)(Params...), size_t smem, int positions, int R, void* stream, const char* what, int N1, int L,
              Args... args) {
  if (R == 0) return ELG_OK;
  const int threads = positions <= 512 ? 256 : 512;
  ELG_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int dev = 0, sms = 0, per_sm = 0;
  ELG_CUDA_OK(cudaGetDevice(&dev));
  ELG_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  ELG_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem));
  ELG_REQUIRE(per_sm > 0, ELG_EUNSUPPORTED, "%s: %zu bytes of shared memory do not fit (N1=%d, L=%d)", what, smem, N1, L);
  const int grid = (int)((long long)R < (long long)sms * per_sm ? R : sms * per_sm);
  kernel<<<grid, threads, smem, (cudaStream_t)stream>>>(args...);
  ELG_LAUNCH_OK();
  return ELG_OK;
}

// Swizzled column of the score matrix E' (row j): XOR the 16-byte chunk index with (j & 7) so
// that 8 consecutive rows read by a quarter-warp hit 8 different bank groups.
__host__ __device__ __forceinline__ int eswz(int j, int c) { return c ^ ((j & 7) << 2); }

// Position of neighbour-list entry e (rank by distance) inside a node's ELG_NBR_STRIDE-byte row:
// 8-way interleaved so lane s of an octet reads its entries e = s, s+8, ... with one 16-byte load.
__host__ __device__ __forceinline__ int nbr_pos(int e) { return (e & 7) * 16 + (e >> 3); }

}  // namespace elg
