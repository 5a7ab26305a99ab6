// Best-improvement TSP local search with 2-opt and Or-opt moves (elg_tsp_local_search).
//
// One CTA refines one tour at a time and is persistent over the R tours.  Everything the search touches lives in shared
// memory, and global memory is touched only to load the tour and to write the result:
//   xy   [N1] float2  coordinates by node            (64 KB at N1 = 8192)
//   edge [N1] float   edge[p] = d(t_p, t_p+1 mod N1) (32 KB)
//   tour [N1] int16   the tour                       (16 KB)
// 14*N1 bytes: 112 KB at N1 = 8192.
//
// A task is one position i and a chunk of TSP_LS_CHUNK consecutive positions j; the lanes of a warp take consecutive i
// and the same chunk, so every read indexed by j is a broadcast.  For each j the task computes the distances from t_j to
// t_i, t_i+1 and t_i+2 (A0_j, A1_j, A2_j), and every term of every variant is one of them or the next j's:
//   v = 0  2-opt      (A0_j - e_i) + (A1_j+1 - e_j)
//   v = 1  s = 1      rem_1 + ((A0_j - e_j) + A0_j+1)
//   v = 2  s = 2      rem_2 + ((A0_j - e_j) + A1_j+1)     v = 3, reversed: rem_2 + ((A1_j - e_j) + A0_j+1)
//   v = 4  s = 3      rem_3 + ((A0_j - e_j) + A2_j+1)     v = 5, reversed: rem_3 + ((A2_j - e_j) + A0_j+1)
// with rem_s = (d(t_i-1, t_i+s) - e_i-1) - e_i+s-1 once per task.  So a pair costs three seglen, plus three per chunk.
// The CTA reduces (gain, v*N1^2 + i*N1 + j) to its minimum.  A move is a composition of span reversals (an Or-opt move
// rotates the segment past its neighbours: reverse the segment, reverse the rest, reverse both), after which the edges
// of the changed span are recomputed.  Position 0 is never inside a span.
#include "common.cuh"

namespace elg {

constexpr int TSP_LS_CHUNK = 16;           // positions j per task (three extra seglen per chunk)

__device__ __forceinline__ void take(float g, int key, float& bg, int& bk) {
  if (gain_better(g, key, bg, bk)) { bg = g; bk = key; }
}

__global__ void __launch_bounds__(512, 2) tsp_ls_kernel(const float* __restrict__ xy_g, int Bxy, int N1,
                                                        const int32_t* __restrict__ inst, int16_t* __restrict__ tours,
                                                        int R, int L, int max_segment, int round_edges,
                                                        int max_iterations, int32_t* __restrict__ iterations,
                                                        float* __restrict__ length) {
  extern __shared__ __align__(16) unsigned char smem[];
  __shared__ float red_g[32];
  __shared__ int red_i[32];
  float2* xy = reinterpret_cast<float2*>(smem);
  float* edge = reinterpret_cast<float*>(xy + N1);
  int16_t* tour = reinterpret_cast<int16_t*>(edge + N1);
  const int tid = threadIdx.x, nthr = blockDim.x;
  const int NN = N1 * N1;
  const int nch = (N1 + TSP_LS_CHUNK - 1) / TSP_LS_CHUNK;
  const int tasks = N1 * nch;

  for (int r = blockIdx.x; r < R; r += gridDim.x) {
    const int b = inst ? inst[r] : (Bxy == 1 ? 0 : r);
    const float2* src = reinterpret_cast<const float2*>(xy_g) + (long long)b * N1;
    int16_t* row = tours + (long long)r * L;
    for (int p = tid; p < N1; p += nthr) xy[p] = src[p];
    for (int p = tid; p < N1; p += nthr) tour[p] = row[p];
    __syncthreads();
    for (int p = tid; p < N1; p += nthr) edge[p] = edge_len(xy, tour[p], tour[p + 1 == N1 ? 0 : p + 1], round_edges);
    __syncthreads();

    int moves = 0;
    while (moves < max_iterations) {
      float bg = INFINITY;
      int bk = 0x7fffffff;
      for (int task = tid; task < tasks; task += nthr) {
        const int i = task % N1, c = task / N1;
        const int j0 = max(c * TSP_LS_CHUNK, max_segment ? 0 : i + 2), j1 = min(c * TSP_LS_CHUNK + TSP_LS_CHUNK, N1);
        if (j0 >= j1) continue;
        const float2 p0 = xy[tour[i]], p1 = xy[tour[min(i + 1, N1 - 1)]], p2 = xy[tour[min(i + 2, N1 - 1)]];
        const float e_i = edge[i];
        // removal part of the Or-opt variants: segment i..i+s-1 taken out, t_i-1 joined to t_i+s
        float rem1 = 0.f, rem2 = 0.f, rem3 = 0.f;
        const bool ok1 = max_segment >= 1 && i >= 1, ok2 = max_segment >= 2 && i >= 1 && i + 1 <= N1 - 1,
                   ok3 = max_segment >= 3 && i >= 1 && i + 2 <= N1 - 1;
        if (ok1) {
          const int prev = tour[i - 1];
          const float e_prev = edge[i - 1];
          rem1 = (edge_len(xy, prev, tour[i + 1 == N1 ? 0 : i + 1], round_edges) - e_prev) - e_i;
          if (ok2) rem2 = (edge_len(xy, prev, tour[i + 2 == N1 ? 0 : i + 2], round_edges) - e_prev) - edge[i + 1];
          if (ok3) rem3 = (edge_len(xy, prev, tour[i + 3 == N1 ? 0 : i + 3], round_edges) - e_prev) - edge[i + 2];
        }
        const auto dist = [round_edges](float2 p, float2 q) {
          const float d = seglen(p.x - q.x, p.y - q.y);
          return round_edges ? rintf(d) : d;
        };
        float2 q = xy[tour[j0]];
        float a0 = dist(q, p0), a1 = dist(q, p1), a2 = max_segment >= 3 ? dist(q, p2) : 0.f;
        for (int j = j0; j < j1; ++j) {
          const int jn = j + 1 == N1 ? 0 : j + 1;
          q = xy[tour[jn]];
          const float n0 = dist(q, p0), n1 = dist(q, p1), n2 = max_segment >= 3 ? dist(q, p2) : 0.f;
          const float e_j = edge[j];
          const int base = i * N1 + j;
          if (j >= i + 2 && !(i == 0 && j == N1 - 1)) take((a0 - e_i) + (n1 - e_j), base, bg, bk);
          if (ok1 && (j < i - 1 || j > i)) take(rem1 + ((a0 - e_j) + n0), NN + base, bg, bk);
          if (ok2 && (j < i - 1 || j > i + 1)) {
            take(rem2 + ((a0 - e_j) + n1), 2 * NN + base, bg, bk);
            take(rem2 + ((a1 - e_j) + n0), 3 * NN + base, bg, bk);
          }
          if (ok3 && (j < i - 1 || j > i + 2)) {
            take(rem3 + ((a0 - e_j) + n2), 4 * NN + base, bg, bk);
            take(rem3 + ((a2 - e_j) + n0), 5 * NN + base, bg, bk);
          }
          a0 = n0; a1 = n1; a2 = n2;
        }
      }
      cta_min_gain(bg, bk, red_g, red_i);
      if (!(bg < LS_MIN_GAIN)) break;                   // every thread reads the same reduction: uniform exit
      const int v = bk / NN, i = bk % NN / N1, j = bk % N1;
      int lo, hi;                                       // the span of positions the move changes
      if (v == 0) {
        lo = i + 1; hi = j;
        reverse_span(tour, lo, hi);
      } else {
        // segment S = i..i+s-1 and the run T between it and the insertion edge: [S T] -> [T S] (j > i) or
        // [T S] -> [S T] (j < i) is reverse S, reverse T, reverse both; a reversed insertion skips reversing S
        const int s = v / 2 + 1, last = i + s - 1;
        lo = j > i ? i : j + 1;
        hi = j > i ? j : last;
        if (v == 1 || !(v & 1)) reverse_span(tour, i, last);
        if (j > i) reverse_span(tour, last + 1, j); else reverse_span(tour, j + 1, i - 1);
        __syncthreads();
        reverse_span(tour, lo, hi);
      }
      __syncthreads();
      for (int p = lo - 1 + tid; p <= hi; p += nthr) edge[p] = edge_len(xy, tour[p], tour[p + 1 == N1 ? 0 : p + 1], round_edges);
      ++moves;
      __syncthreads();
    }

    for (int p = tid; p < N1; p += nthr) row[p] = tour[p];
    if (tid == 0) {
      // the summation order of tour_length_kernel: sequential from the edge leaving position 0
      float sum = 0.f;
      for (int p = 0; p < N1; ++p) sum += edge[p];
      length[r] = sum;
      iterations[r] = moves;
    }
    __syncthreads();                                    // shared memory is reused by the next tour
  }
}

size_t tsp_ls_smem_bytes(int N1) { return (size_t)N1 * (sizeof(float2) + sizeof(float) + sizeof(int16_t)); }

}  // namespace elg

using namespace elg;

extern "C" {

int elg_tsp_local_search(const float* xy, int Bxy, int N1, const int32_t* inst, int16_t* tours, int R, int L,
                         int max_segment, int round_edges, int max_iterations, int32_t* iterations, float* length,
                         void* stream) {
  ELG_REQUIRE(N1 > 0 && R >= 0 && Bxy > 0, ELG_EINVAL, "bad sizes N1=%d R=%d Bxy=%d", N1, R, Bxy);
  ELG_REQUIRE(N1 <= ELG_MAX_NODES, ELG_EUNSUPPORTED, "tsp local search supports up to %d nodes (got %d)", ELG_MAX_NODES,
              N1);
  ELG_REQUIRE(L >= N1, ELG_EINVAL, "tours need L >= N1 (L=%d, N1=%d)", L, N1);
  ELG_REQUIRE(max_segment >= 0 && max_segment <= 3, ELG_EINVAL, "max_segment must be in 0..3 (got %d)", max_segment);
  ELG_REQUIRE(max_iterations >= 0, ELG_EINVAL, "max_iterations must be >= 0 (got %d)", max_iterations);
  ELG_REQUIRE(xy && tours && iterations && length, ELG_EINVAL, "NULL pointer");
  ELG_REQUIRE(inst || Bxy == 1 || Bxy == R, ELG_EINVAL, "without inst the xy batch must be 1 or R (Bxy=%d, R=%d)", Bxy, R);
  if (R == 0) return ELG_OK;
  const size_t smem = tsp_ls_smem_bytes(N1);
  const int threads = N1 <= 512 ? 256 : 512;
  ELG_CUDA_OK(cudaFuncSetAttribute(tsp_ls_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int dev = 0, sms = 0, per_sm = 0;
  ELG_CUDA_OK(cudaGetDevice(&dev));
  ELG_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  ELG_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, tsp_ls_kernel, threads, smem));
  ELG_REQUIRE(per_sm > 0, ELG_EUNSUPPORTED, "tsp local search: %zu bytes of shared memory do not fit (N1=%d)", smem, N1);
  const int grid = (int)((long long)R < (long long)sms * per_sm ? R : sms * per_sm);
  tsp_ls_kernel<<<grid, threads, smem, (cudaStream_t)stream>>>(xy, Bxy, N1, inst, tours, R, L, max_segment, round_edges,
                                                               max_iterations, iterations, length);
  ELG_LAUNCH_OK();
  return ELG_OK;
}

}  // extern "C"
