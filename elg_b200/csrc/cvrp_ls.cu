// Best-improvement CVRP local search with capacity (elg_cvrp_local_search): 2-opt inside a route, relocate of one
// customer, swap of two customers of different routes, and 2-opt* (tail exchange) between two routes.
//
// One CTA refines one row at a time and is persistent over the R rows.  The whole solution lives in shared memory and
// global memory is touched only to load the row and to write the result:
//   xy   [N1] float2   coordinates by node                                 (64 KB at N1 = 8192)
//   pref [L]  int32    demand of the route's customers up to the position; at a depot position the route's total
//   dem  [N1] int32    demands by node
//   row  [L]  int16    the canonical row: routes in order, each preceded by one 0, no empty route, zero padding
//   rs   [L]  int16    position of the route's depot visit (the last 0 at or before the position)
// 12*N1 + 8*L bytes: 224 KB for N1 = 8192, L = 2*N1+2.  There is no room for an edge array, so edges are recomputed.
//
// Per move every position i (positions 0..P-1, P = 1 + last customer position) sweeps the positions j in chunks of
// CVRP_LS_CHUNK; consecutive j share d(t_j, t_i) and d(t_j, t_j+1), so a pair costs two distances plus one to three for
// the move types that apply to it.  The CTA reduces (gain, type*L^2 + i*L + j) to its minimum.  Every applied move is a
// composition of reversals of row spans; a route emptied by it leaves two adjacent depot visits, one of which is rotated
// to the end of the used positions.  The route starts and load prefixes are then rebuilt from the first changed route
// to the end of the used positions with one segmented scan.
#include <climits>

#include "common.cuh"

namespace elg {

constexpr int CVRP_LS_CHUNK = 16;   // positions j per task

// rs and pref of positions lo..hi, where row[lo] == 0 and position hi+1 starts a route or is L.  One segmented scan over
// contiguous per-thread slices: the carry of a slice is (last depot position in it or -1, demand after that depot).
__device__ __forceinline__ void rebuild_routes(const int16_t* row, const int32_t* dem, int16_t* rs, int32_t* pref, int lo, int hi, int L,
                               int* red_a, int* red_b) {
  const int tid = threadIdx.x, nthr = blockDim.x, lane = tid & 31, warp = tid >> 5;
  const int len = hi - lo + 1, per = (len + nthr - 1) / nthr;
  const int p0 = lo + min(tid * per, len), p1 = lo + min((tid + 1) * per, len);
  int last = -1, sum = 0;
  for (int p = p0; p < p1; ++p) {
    const int v = row[p];
    if (v == 0) { last = p; sum = 0; } else sum += dem[v];
  }
  for (int o = 1; o < 32; o <<= 1) {                    // inclusive scan within the warp
    const int l2 = __shfl_up_sync(0xffffffffu, last, o), s2 = __shfl_up_sync(0xffffffffu, sum, o);
    if (lane >= o && last < 0) { last = l2; sum += s2; }
  }
  if (lane == 31) { red_a[warp] = last; red_b[warp] = sum; }
  __syncthreads();
  int cur = -1, run = 0;                                // exclusive carry: earlier warps, then the lane before
  for (int w = 0; w < warp; ++w) {
    if (red_a[w] >= 0) { cur = red_a[w]; run = red_b[w]; } else run += red_b[w];
  }
  const int l1 = __shfl_up_sync(0xffffffffu, last, 1), s1 = __shfl_up_sync(0xffffffffu, sum, 1);
  if (lane > 0) {
    if (l1 >= 0) { cur = l1; run = s1; } else run += s1;
  }
  for (int p = p0; p < p1; ++p) {
    const int v = row[p];
    if (v == 0) { cur = p; run = 0; } else run += dem[v];
    rs[p] = (int16_t)cur;
    pref[p] = run;
  }
  __syncthreads();
  for (int p = lo + tid; p <= hi; p += nthr)            // the route's total at its depot position
    if (row[p] != 0 && (p + 1 == L || row[p + 1] == 0)) pref[rs[p]] = pref[p];
  __syncthreads();
}

__global__ void __launch_bounds__(512, 1) cvrp_ls_kernel(const float* __restrict__ xy_g, int Bxy, int N1,
                                                       const int32_t* __restrict__ dem_g, int capacity,
                                                       const int32_t* __restrict__ inst, int16_t* __restrict__ tours,
                                                       int R, int L, int round_edges, int max_iterations,
                                                       int32_t* __restrict__ iterations, float* __restrict__ length) {
  extern __shared__ __align__(16) unsigned char smem[];
  __shared__ float red_g[32];
  __shared__ int red_a[32], red_b[32];
  __shared__ int s_pos[2];
  float2* xy = reinterpret_cast<float2*>(smem);
  int32_t* pref = reinterpret_cast<int32_t*>(xy + N1);
  int32_t* dem = pref + L;
  int16_t* row = reinterpret_cast<int16_t*>(dem + N1);
  int16_t* rs = row + L;
  const int tid = threadIdx.x, nthr = blockDim.x, lane = tid & 31, warp = tid >> 5;
  const int LL = L * L;

  for (int r = blockIdx.x; r < R; r += gridDim.x) {
    const int b = inst ? inst[r] : (Bxy == 1 ? 0 : r);
    const float2* src_xy = reinterpret_cast<const float2*>(xy_g) + (long long)b * N1;
    const int32_t* src_dem = dem_g + (long long)b * N1;
    int16_t* grow = tours + (long long)r * L;
    for (int p = tid; p < N1; p += nthr) { xy[p] = src_xy[p]; dem[p] = src_dem[p]; }

    // canonical form: keep position 0, every customer, and a depot visit right after a customer (stream compaction)
    {
      const int per = (L + nthr - 1) / nthr, p0 = min(tid * per, L), p1 = min(p0 + per, L);
      int cnt = 0;
      for (int p = p0; p < p1; ++p) cnt += (p == 0 || grow[p] != 0 || grow[p - 1] != 0);
      int incl = cnt;
      for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
      }
      if (lane == 31) red_a[warp] = incl;
      __syncthreads();
      int out = incl - cnt;
      for (int w = 0; w < warp; ++w) out += red_a[w];
      for (int p = p0; p < p1; ++p)
        if (p == 0 || grow[p] != 0 || grow[p - 1] != 0) row[out++] = grow[p];
      if (tid == nthr - 1) s_pos[0] = out;
      __syncthreads();
    }
    const int kept = s_pos[0];
    for (int p = kept + tid; p < L; p += nthr) row[p] = 0;
    __syncthreads();
    int P = kept > 1 && row[kept - 1] == 0 ? kept - 1 : kept;   // used positions: up to the last customer
    rebuild_routes(row, dem, rs, pref, 0, L - 1, L, red_a, red_b);

    int moves = 0;
    while (moves < max_iterations) {
      float bg = INFINITY;
      int bk = INT_MAX;
      const int nch = (P + CVRP_LS_CHUNK - 1) / CVRP_LS_CHUNK;
      for (int task = tid; task < P * nch; task += nthr) {
        const int i = task / nch, j0 = (task % nch) * CVRP_LS_CHUNK, j1 = min(j0 + CVRP_LS_CHUNK, P);
        const int u = row[i], a = i > 0 ? row[i - 1] : 0, bn = i + 1 < P ? row[i + 1] : 0, ri = rs[i];
        const float e_im1 = edge_len(xy, a, u, round_edges), e_i = edge_len(xy, u, bn, round_edges);
        const float rem = edge_len(xy, a, bn, round_edges) - e_im1 - e_i;        // relocate: u taken out
        const int du = dem[u], load_a = pref[ri], pre_a = u ? pref[i] : 0;
        const int t0 = row[j0], tm1 = j0 > 0 ? row[j0 - 1] : 0;
        float dju = edge_len(xy, t0, u, round_edges);                             // d(t_j, u)
        float djm1u = edge_len(xy, tm1, u, round_edges);                          // d(t_j-1, u)
        float ejm1 = edge_len(xy, tm1, t0, round_edges);                          // d(t_j-1, t_j)
        for (int j = j0; j < j1; ++j) {
          const int tj = row[j], tj1 = j + 1 < P ? row[j + 1] : 0, rj = rs[j];
          const float dj1u = edge_len(xy, tj1, u, round_edges), ej = edge_len(xy, tj, tj1, round_edges);
          if (j >= i + 2 && rj <= i) {                                            // 0: reverse i+1..j inside a route
            const float g = (dju - e_i) + (edge_len(xy, bn, tj1, round_edges) - ej);
            if (gain_better(g, i * L + j, bg, bk)) { bg = g; bk = i * L + j; }
          }
          if (u != 0 && j != i - 1 && j != i && (rj == ri || pref[rj] + du <= capacity)) {   // 1: u onto (t_j, t_j+1)
            const float g = rem + ((dju + dj1u) - ej);
            const int key = LL + i * L + j;
            if (gain_better(g, key, bg, bk)) { bg = g; bk = key; }
          }
          if (j > i && rj != ri) {
            const float dvb = edge_len(xy, tj, bn, round_edges);
            const int dv = dem[tj], load_b = pref[rj], pre_b = tj ? pref[j] : 0;
            if (u != 0 && tj != 0 && load_a - du + dv <= capacity && load_b - dv + du <= capacity) {   // 2: swap
              const float g = ((edge_len(xy, a, tj, round_edges) + dvb) - (e_im1 + e_i)) + ((djm1u + dj1u) - (ejm1 + ej));
              const int key = 2 * LL + i * L + j;
              if (gain_better(g, key, bg, bk)) { bg = g; bk = key; }
            }
            if (pre_a + load_b - pre_b <= capacity && pre_b + load_a - pre_a <= capacity) {          // 3: 2-opt*
              const float g = (dj1u - e_i) + (dvb - ej);
              const int key = 3 * LL + i * L + j;
              if (gain_better(g, key, bg, bk)) { bg = g; bk = key; }
            }
          }
          djm1u = dju; dju = dj1u; ejm1 = ej;
        }
      }
      cta_min_gain(bg, bk, red_g, red_a);
      if (!(bg < LS_MIN_GAIN)) break;                   // every thread reads the same reduction: uniform exit
      const int type = bk / LL, i = bk % LL / L, j = bk % L;
      const int lo = rs[min(i, j)];                     // first route the move changes
      if (type == 0) {
        reverse_span(row, i + 1, j);
      } else if (type == 1) {                           // rotate u from i to j (j > i) or to j+1 (j < i)
        if (j > i) { reverse_span(row, i, j); __syncthreads(); reverse_span(row, i, j - 1); }
        else { reverse_span(row, j + 1, i); __syncthreads(); reverse_span(row, j + 2, i); }
      } else if (type == 2) {
        if (tid == 0) { const int16_t t = row[i]; row[i] = row[j]; row[j] = t; }
      } else {
        // [X Z Y] -> [Y Z X] with X = A after i, Z = the routes between up to B's head, Y = B after j
        if (tid == 0) { s_pos[0] = P; s_pos[1] = P; }
        __syncthreads();
        for (int q = i + 1 + tid; q < P; q += nthr)
          if (row[q] == 0) atomicMin(&s_pos[q > j ? 1 : 0], q);
        __syncthreads();
        const int ea = s_pos[0] - 1, eb = s_pos[1] - 1, ny = eb - j, nz = j - ea;
        reverse_span(row, i + 1, eb);
        __syncthreads();
        reverse_span(row, i + 1, i + ny);
        reverse_span(row, i + 1 + ny, i + ny + nz);
        reverse_span(row, i + 1 + ny + nz, eb);
      }
      __syncthreads();
      if (tid == 0) s_pos[0] = P;                       // an emptied route: two adjacent depot visits
      __syncthreads();
      for (int q = lo + 1 + tid; q < P; q += nthr)
        if (row[q] == 0 && row[q - 1] == 0) atomicMin(&s_pos[0], q);
      __syncthreads();
      const int z = s_pos[0];
      if (z < P) { reverse_span(row, z, P - 1); __syncthreads(); reverse_span(row, z, P - 2); }
      __syncthreads();
      const int p_old = P;
      if (row[p_old - 1] == 0) --P;
      rebuild_routes(row, dem, rs, pref, lo, p_old - 1, L, red_a, red_b);
      ++moves;
    }

    // closed length in the summation order of tour_length_kernel: sequential from the edge leaving position 0
    float* edge = reinterpret_cast<float*>(pref);       // the prefixes are not needed any more
    for (int p = tid; p < L; p += nthr) {
      edge[p] = edge_len(xy, row[p], row[p + 1 == L ? 0 : p + 1], round_edges);
      grow[p] = row[p];
    }
    __syncthreads();
    if (tid == 0) {
      float sum = 0.f;
      for (int p = 0; p < L; ++p) sum += edge[p];
      length[r] = sum;
      iterations[r] = moves;
    }
    __syncthreads();                                    // shared memory is reused by the next row
  }
}

size_t cvrp_ls_smem_bytes(int N1, int L) {
  return (size_t)N1 * (sizeof(float2) + sizeof(int32_t)) + (size_t)L * (sizeof(int32_t) + 2 * sizeof(int16_t));
}

}  // namespace elg

using namespace elg;

extern "C" {

int elg_cvrp_local_search(const float* xy, int Bxy, int N1, const int32_t* demand, int32_t capacity, const int32_t* inst,
                          int16_t* tours, int R, int L, int round_edges, int max_iterations, int32_t* iterations,
                          float* length, void* stream) {
  ELG_REQUIRE(N1 > 0 && R >= 0 && Bxy > 0, ELG_EINVAL, "bad sizes N1=%d R=%d Bxy=%d", N1, R, Bxy);
  ELG_REQUIRE(N1 <= ELG_MAX_NODES, ELG_EUNSUPPORTED, "cvrp local search supports up to %d nodes (got %d)", ELG_MAX_NODES,
              N1);
  ELG_REQUIRE(L > 0 && L <= 2 * N1 + 2, ELG_EINVAL, "rows need 0 < L <= 2*N1+2 (L=%d, N1=%d)", L, N1);
  ELG_REQUIRE(capacity > 0, ELG_EINVAL, "capacity must be > 0 (got %d)", capacity);
  ELG_REQUIRE(max_iterations >= 0, ELG_EINVAL, "max_iterations must be >= 0 (got %d)", max_iterations);
  ELG_REQUIRE(xy && demand && tours && iterations && length, ELG_EINVAL, "NULL pointer");
  ELG_REQUIRE(inst || Bxy == 1 || Bxy == R, ELG_EINVAL, "without inst the xy batch must be 1 or R (Bxy=%d, R=%d)", Bxy, R);
  if (R == 0) return ELG_OK;
  const size_t smem = cvrp_ls_smem_bytes(N1, L);
  const int threads = L <= 512 ? 256 : 512;
  ELG_CUDA_OK(cudaFuncSetAttribute(cvrp_ls_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int dev = 0, sms = 0, per_sm = 0;
  ELG_CUDA_OK(cudaGetDevice(&dev));
  ELG_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  ELG_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, cvrp_ls_kernel, threads, smem));
  ELG_REQUIRE(per_sm > 0, ELG_EUNSUPPORTED, "cvrp local search: %zu bytes of shared memory do not fit (N1=%d, L=%d)", smem,
              N1, L);
  const int grid = (int)((long long)R < (long long)sms * per_sm ? R : sms * per_sm);
  cvrp_ls_kernel<<<grid, threads, smem, (cudaStream_t)stream>>>(xy, Bxy, N1, demand, capacity, inst, tours, R, L,
                                                                round_edges, max_iterations, iterations, length);
  ELG_LAUNCH_OK();
  return ELG_OK;
}

}  // extern "C"
