// Best-improvement 2-opt local search on TSP tours and CVRP routes (elg_two_opt).
//
// One CTA refines one tour at a time and is persistent over the R tours.  Everything the search touches lives in
// shared memory: the coordinates indexed by node, the tour (int16 node ids), the length of every tour edge, and for
// CVRP the position of the last depot visit at or before every position.  Per move the CTA evaluates every admissible
// pair (i, j), reduces (gain, i*L + j) to its minimum, reverses positions i+1..j and patches the edge array; global
// memory is touched only to load the tour and to write the result.
//
// Pairs are swept along diagonals (j - i = d constant) in chunks of CHUNK: the edge (t_i, t_j) of a pair is the edge
// (t_{i+1}, t_{j+1}) of the pair before it, so each pair costs one seglen.  For CVRP a pair is admissible only if
// positions i+1..j are all customers, so d never exceeds the longest run of customers; route lengths do not change
// under such moves, which bounds the sweep for the whole search.
#include "common.cuh"

namespace elg {

constexpr int TWO_OPT_CHUNK = 16;          // pairs per diagonal chunk (one extra seglen per chunk)

template <int PROBLEM>
__global__ void __launch_bounds__(512) two_opt_kernel(const float* __restrict__ xy_g, int Bxy, int N1,
                                                       const int32_t* __restrict__ inst, int16_t* __restrict__ tours,
                                                       int R, int L, int round_edges, int max_iterations,
                                                       int32_t* __restrict__ iterations, float* __restrict__ length) {
  extern __shared__ __align__(16) unsigned char smem[];
  __shared__ float red_g[32];
  __shared__ int red_i[32];
  __shared__ int s_dmax;
  const int n = PROBLEM == ELG_CVRP ? L : N1;           // positions of the cyclic tour
  float2* xy = reinterpret_cast<float2*>(smem);
  float* edge = reinterpret_cast<float*>(xy + N1);     // edge[p] = d(t_p, t_{p+1 mod n})
  int16_t* tour = reinterpret_cast<int16_t*>(edge + n);
  int16_t* lastdep = tour + n;                          // cvrp: last position <= p holding the depot, -1 if none
  const int tid = threadIdx.x, nthr = blockDim.x, lane = tid & 31, warp = tid >> 5;

  for (int r = blockIdx.x; r < R; r += gridDim.x) {
    const int b = inst ? inst[r] : (Bxy == 1 ? 0 : r);
    const float2* src = reinterpret_cast<const float2*>(xy_g) + (long long)b * N1;
    int16_t* row = tours + (long long)r * L;
    for (int p = tid; p < N1; p += nthr) xy[p] = src[p];
    for (int p = tid; p < n; p += nthr) tour[p] = row[p];
    __syncthreads();
    for (int p = tid; p < n; p += nthr) edge[p] = edge_len(xy, tour[p], tour[p + 1 == n ? 0 : p + 1], round_edges);

    int dmax = n - 1;                                   // largest diagonal j - i worth sweeping
    if (PROBLEM == ELG_CVRP) {
      // max-scan of depot positions: each thread scans a contiguous slice, then the slices are combined
      const int per = (n + nthr - 1) / nthr, p0 = min(tid * per, n), p1 = min(p0 + per, n);
      int last = -1;
      for (int p = p0; p < p1; ++p) if (tour[p] == 0) last = p;
      int incl = last;                                  // inclusive max-scan over threads
      for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl = max(incl, v);
      }
      if (lane == 31) red_i[warp] = incl;
      if (tid == 0) s_dmax = 0;
      __syncthreads();
      int prev = -1;
      for (int w = 0; w < warp; ++w) prev = max(prev, red_i[w]);
      const int up = __shfl_up_sync(0xffffffffu, incl, 1);
      if (lane > 0) prev = max(prev, up);
      int run = 0;
      for (int p = p0; p < p1; ++p) {
        if (tour[p] == 0) prev = p;
        lastdep[p] = (int16_t)prev;
        run = max(run, p - prev);
      }
      atomicMax(&s_dmax, run);
      __syncthreads();
      dmax = min(s_dmax, n - 1);
    }
    __syncthreads();

    const int nd = dmax - 1;                            // diagonals d = 2..dmax
    const int nchunks = (n - 2 + TWO_OPT_CHUNK - 1) / TWO_OPT_CHUNK;
    const int tasks = nd > 0 ? nd * nchunks : 0;
    int moves = 0;
    while (moves < max_iterations) {
      float bg = INFINITY;
      int bidx = 0x7fffffff;
      for (int task = tid; task < tasks; task += nthr) {
        const int d = 2 + task % nd;
        const int i0 = (task / nd) * TWO_OPT_CHUNK, i1 = min(i0 + TWO_OPT_CHUNK, n - d);
        if (i0 >= i1) continue;
        float dij = edge_len(xy, tour[i0], tour[i0 + d], round_edges);
        for (int i = i0; i < i1; ++i) {
          const int j = i + d, j1 = j + 1 == n ? 0 : j + 1;
          const float dnext = edge_len(xy, tour[i + 1], tour[j1], round_edges);
          const bool ok = PROBLEM == ELG_CVRP ? lastdep[j] <= i : !(i == 0 && j == n - 1);
          if (ok) {
            const float g = (dij - edge[i]) + (dnext - edge[j]);
            const int idx = i * L + j;
            if (gain_better(g, idx, bg, bidx)) { bg = g; bidx = idx; }
          }
          dij = dnext;
        }
      }
      cta_min_gain(bg, bidx, red_g, red_i);
      if (!(bg < LS_MIN_GAIN)) break;                   // every thread reads the same reduction: uniform exit
      const int i = bidx / L, j = bidx % L;
      // reverse tour[i+1..j] and, with it, the edges strictly inside the segment, edge[i+1..j-1]
      for (int k = tid; k < (j - i) / 2; k += nthr) {
        const int16_t t = tour[i + 1 + k]; tour[i + 1 + k] = tour[j - k]; tour[j - k] = t;
      }
      for (int k = tid; k < (j - i - 1) / 2; k += nthr) {
        const float e = edge[i + 1 + k]; edge[i + 1 + k] = edge[j - 1 - k]; edge[j - 1 - k] = e;
      }
      __syncthreads();
      if (tid == 0) edge[i] = edge_len(xy, tour[i], tour[i + 1], round_edges);
      if (tid == 1) edge[j] = edge_len(xy, tour[j], tour[j + 1 == n ? 0 : j + 1], round_edges);
      ++moves;
      __syncthreads();
    }

    for (int p = tid; p < n; p += nthr) row[p] = tour[p];
    if (tid == 0) {
      // the summation order of tour_length_kernel: sequential from the edge leaving position 0
      float sum = 0.f;
      for (int p = 0; p < n; ++p) sum += edge[p];
      length[r] = sum;
      iterations[r] = moves;
    }
    __syncthreads();                                    // shared memory is reused by the next tour
  }
}

size_t two_opt_smem_bytes(int problem, int N1, int L) {
  const size_t n = problem == ELG_CVRP ? L : N1;
  return (size_t)N1 * sizeof(float2) + n * sizeof(float) + n * sizeof(int16_t) * (problem == ELG_CVRP ? 2 : 1);
}

}  // namespace elg

using namespace elg;

extern "C" {

int elg_two_opt(int problem, const float* xy, int Bxy, int N1, const int32_t* inst, int16_t* tours, int R, int L,
                int round_edges, int max_iterations, int32_t* iterations, float* length, void* stream) {
  ELG_REQUIRE(problem == ELG_TSP || problem == ELG_CVRP, ELG_EINVAL, "unknown problem %d", problem);
  ELG_REQUIRE(N1 > 0 && R >= 0 && Bxy > 0, ELG_EINVAL, "bad sizes N1=%d R=%d Bxy=%d", N1, R, Bxy);
  ELG_REQUIRE(N1 <= ELG_MAX_NODES, ELG_EUNSUPPORTED, "2-opt supports up to %d nodes (got %d)", ELG_MAX_NODES, N1);
  ELG_REQUIRE(problem == ELG_CVRP || L >= N1, ELG_EINVAL, "tsp tours need L >= N1 (L=%d, N1=%d)", L, N1);
  ELG_REQUIRE(problem == ELG_TSP || (L > 0 && L <= 2 * N1 + 2), ELG_EINVAL,
              "cvrp tours need 0 < L <= 2*N1+2 (L=%d, N1=%d)", L, N1);
  ELG_REQUIRE(max_iterations >= 0, ELG_EINVAL, "max_iterations must be >= 0 (got %d)", max_iterations);
  ELG_REQUIRE(xy && tours && iterations && length, ELG_EINVAL, "NULL pointer");
  ELG_REQUIRE(inst || Bxy == 1 || Bxy == R, ELG_EINVAL, "without inst the xy batch must be 1 or R (Bxy=%d, R=%d)", Bxy, R);
  if (R == 0) return ELG_OK;
  const size_t smem = two_opt_smem_bytes(problem, N1, L);
  const int n = problem == ELG_CVRP ? L : N1;
  const int threads = n <= 512 ? 256 : 512;
  auto kernel = problem == ELG_CVRP ? two_opt_kernel<ELG_CVRP> : two_opt_kernel<ELG_TSP>;
  ELG_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int dev = 0, sms = 0, per_sm = 0;
  ELG_CUDA_OK(cudaGetDevice(&dev));
  ELG_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  ELG_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem));
  ELG_REQUIRE(per_sm > 0, ELG_EUNSUPPORTED, "2-opt: %zu bytes of shared memory do not fit (N1=%d, L=%d)", smem, N1, L);
  const int grid = (int)((long long)R < (long long)sms * per_sm ? R : sms * per_sm);
  kernel<<<grid, threads, smem, (cudaStream_t)stream>>>(xy, Bxy, N1, inst, tours, R, L, round_edges, max_iterations,
                                                        iterations, length);
  ELG_LAUNCH_OK();
  return ELG_OK;
}

}  // extern "C"
