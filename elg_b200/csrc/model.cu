// Weight layout + one-time weight folds (elg_prepare_model) + library bookkeeping.
#include <stdarg.h>
#include <string.h>
#include <atomic>
#include <cuda_fp16.h>
#include "common.cuh"
#include "umma.cuh"

namespace elg {

static thread_local char g_err[512] = "";
static std::atomic<uint64_t> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
void count_launch(int n) { g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed); }

int check_desc(const elg_model_desc* d) {
  ELG_REQUIRE(d != nullptr, ELG_EINVAL, "model desc is NULL");
  ELG_REQUIRE(d->problem == ELG_TSP || d->problem == ELG_CVRP, ELG_EINVAL, "unknown problem %d", d->problem);
  ELG_REQUIRE(d->emb == E && d->heads == H && d->qkv == D, ELG_EUNSUPPORTED,
              "kernels are built for embedding_dim=128, head_num=8, qkv_dim=16 (got %d/%d/%d)", d->emb, d->heads, d->qkv);
  ELG_REQUIRE(d->local_emb == LE && d->local_heads == LH && d->local_qkv == LD, ELG_EUNSUPPORTED,
              "kernels are built for local_att 32/4/8 (got %d/%d/%d)", d->local_emb, d->local_heads, d->local_qkv);
  ELG_REQUIRE(d->layers >= 1 && d->layers <= ELG_MAX_LAYERS, ELG_EUNSUPPORTED, "encoder_layer_num %d not in [1,%d]", d->layers, ELG_MAX_LAYERS);
  ELG_REQUIRE(d->ff > 0 && d->ff % 128 == 0, ELG_EUNSUPPORTED, "ff_hidden_dim must be a positive multiple of 128");
  const int k_max = KT_MAX - (d->problem == ELG_CVRP ? 1 : 0);      // the cvrp local sequence also holds the depot
  ELG_REQUIRE(d->local_k >= 1 && d->local_k <= k_max, ELG_EUNSUPPORTED, "local_size %d outside [1,%d] for %s", d->local_k,
              k_max, d->problem == ELG_CVRP ? "cvrp" : "tsp");
  ELG_REQUIRE(d->flags & ELG_FLAG_DISTANCE_PENALTY, ELG_EUNSUPPORTED,
              "distance_penalty=False is not implemented (ensemble may be on or off)");
  return ELG_OK;
}

// ---------------------------------------------------------------------------------------------
// One block; every output element is an independent short dot product (double accumulation).
__global__ void prepare_kernel(elg_model_desc d, elg_weight_layout_t L, const float* __restrict__ w,
                               float* __restrict__ der) {
  const int tid = threadIdx.x, nt = blockDim.x;
  const bool cvrp = d.problem == ELG_CVRP;
  const int ldq = cvrp ? E + 1 : E;
  const int F = cvrp ? 3 : 2;
  const float inv_sqrt_e = 11.313708498984761f;  // sqrt(128)
  for (int i = tid; i < E * E; i += nt) {
    int o = i / E, c = i % E;
    der[DER_WQN + i] = w[L.dec_wq_last + (int64_t)o * ldq + c];
    der[DER_WQF + i] = cvrp ? 0.f : w[L.dec_wq_first + i];
    der[DER_WK4 + i] = w[L.dec_wk + i] * 0.36067376022224085f;   // log2(e) / sqrt(D): phase A works in the log2 domain
    der[DER_WET + i] = w[L.dec_wo + (int64_t)c * E + o] / inv_sqrt_e;   // WET[o=i][c=k] = Wo[k][i]/sqrt(E)
  }
  for (int i = tid; i < E; i += nt) {
    der[DER_WL + i] = cvrp ? w[L.dec_wq_last + (int64_t)i * ldq + E] : 0.f;
    der[DER_BE + i] = w[L.dec_bo + i] / inv_sqrt_e;
  }
  float* loc = der + DER_LOC;
  __shared__ float ql[LE];
  __shared__ float pe[KT_MAX][LE];
  __shared__ float we[LE][4];
  for (int c = tid; c < LE; c += nt) {
    double a = 0;
    for (int i = 0; i < LE; ++i) a += (double)w[L.loc_wq + c * LE + i] * (double)w[L.loc_token + i];
    ql[c] = (float)a;
    for (int f = 0; f < 4; ++f) we[c][f] = f < F ? w[L.loc_we + c * F + f] : 0.f;
  }
  const float inc = (float)(-(log(10000.0) / 15.0));
  for (int i = tid; i < KT_MAX * LE; i += nt) {
    int p = i / LE, c = i % LE;
    float v = 0.f;
    if (d.flags & ELG_FLAG_POSITIONAL) {
      float inv = expf((float)(c % (LE / 2)) * inc);
      float ang = (float)p * inv;
      v = c < LE / 2 ? sinf(ang) : cosf(ang);
    }
    pe[p][c] = v;
    loc[LOC_PE + i] = v;
  }
  __syncthreads();
  const double inv_sqrt_d = 1.4426950408889634 / sqrt((double)LD);   // log2(e)/sqrt(d): local softmax runs in the log2 domain
  // u_h[f] and t_h[p]
  for (int i = tid; i < LH * 4; i += nt) {
    int h = i / 4, f = i % 4;
    double a = 0;
    for (int dd = 0; dd < LD; ++dd) {
      double kf = 0;
      for (int c = 0; c < LE; ++c) kf += (double)w[L.loc_wk + (h * LD + dd) * LE + c] * (double)we[c][f];
      a += (double)ql[h * LD + dd] * kf;
    }
    loc[LOC_U + i] = (float)(a * inv_sqrt_d);
  }
  for (int i = tid; i < LH * KT_MAX; i += nt) {
    int h = i / KT_MAX, p = i % KT_MAX;
    double a = 0;
    for (int dd = 0; dd < LD; ++dd) {
      double kb = 0;
      for (int c = 0; c < LE; ++c)
        kb += (double)w[L.loc_wk + (h * LD + dd) * LE + c] * ((double)w[L.loc_be + c] + (double)pe[p][c]);
      a += (double)ql[h * LD + dd] * kb;
    }
    loc[LOC_T + i] = (float)(a * inv_sqrt_d);
  }
  for (int i = tid; i < LE * 4; i += nt) {
    int c = i / 4, f = i % 4;
    double a = 0;
    for (int k = 0; k < LE; ++k) a += (double)w[L.loc_wv + c * LE + k] * (double)we[k][f];
    loc[LOC_A + i] = (float)a;
    loc[LOC_WE + i] = we[c][f];
  }
  for (int c = tid; c < LE; c += nt) {
    double a = 0;
    for (int k = 0; k < LE; ++k) a += (double)w[L.loc_wv + c * LE + k] * (double)w[L.loc_be + k];
    loc[LOC_CV + c] = (float)a;
    loc[LOC_BC + c] = w[L.loc_bo + c];
    loc[LOC_BE + c] = w[L.loc_be + c];
  }
  for (int i = tid; i < KT_MAX * LE; i += nt) {
    int p = i / LE, c = i % LE;
    double a = 0;
    for (int k = 0; k < LE; ++k) a += (double)w[L.loc_wv + c * LE + k] * (double)pe[p][k];
    loc[LOC_VPE + i] = (float)a;
  }
  for (int i = tid; i < LE * LE; i += nt) {
    int c = i / LE, c2 = i % LE;                 // WCT[c][c2] = Wo_l[c2][c]
    loc[LOC_WCT + i] = w[L.loc_wo + c2 * LE + c];
  }
  // folds of everything downstream of ol (mh = Wo_l ol + bo_l; z = We^T mh; c0 = be . mh; pem_p = PE(p) . mh), x 1/sqrt(LE)
  const double isl = 1.0 / sqrt((double)LE);
  for (int i = tid; i < KT_MAX * LE; i += nt) {
    int p = i / LE, c = i % LE;
    double a = 0;
    for (int k = 0; k < LE; ++k) a += (double)pe[p][k] * (double)w[L.loc_wo + k * LE + c];
    loc[LOC_PW + i] = (float)(a * isl);
  }
  for (int p = tid; p < KT_MAX; p += nt) {
    double a = 0;
    for (int k = 0; k < LE; ++k) a += (double)pe[p][k] * (double)w[L.loc_bo + k];
    loc[LOC_PB + p] = (float)(a * isl);
  }
  for (int i = tid; i < LE * 4; i += nt) {
    int c = i / 4, f = i % 4;
    double a = 0;
    for (int k = 0; k < LE; ++k) a += (f < 3 ? (double)we[k][f] : (double)w[L.loc_be + k]) * (double)w[L.loc_wo + k * LE + c];
    loc[LOC_ZW + i] = (float)(a * isl);
  }
  for (int f = tid; f < 4; f += nt) {
    double a = 0;
    for (int k = 0; k < LE; ++k) a += (f < 3 ? (double)we[k][f] : (double)w[L.loc_be + k]) * (double)w[L.loc_bo + k];
    loc[LOC_ZB + f] = (float)(a * isl);
  }
  // tcgen05 B operands of the two local-policy contractions (rollout_tc.cu), from the fp32 tables above
  __syncthreads();
  uint8_t* op1 = reinterpret_cast<uint8_t*>(loc + LOC_OP1);
  for (int i = tid; i < LH * 16 * KT_MAX; i += nt) {
    const int h = i / (16 * KT_MAX), n = (i / KT_MAX) % 16, p = i % KT_MAX;
    __half hi, lo;
    umma::split_f16(n < LD ? loc[LOC_VPE + p * LE + h * LD + n] : 0.f, hi, lo);
    const uint32_t off = umma::elem_off(n, p, 256);
    *reinterpret_cast<__half*>(op1 + h * (KT_MAX * 64) + off) = hi;
    *reinterpret_cast<__half*>(op1 + h * (KT_MAX * 64) + KT_MAX * 32 + off) = lo;
  }
  const int K1 = d.local_k + (cvrp ? 1 : 0);
  const int N2 = (K1 + 4 + 15) & ~15;
  uint8_t* op2 = reinterpret_cast<uint8_t*>(loc + LOC_OP2);
  for (int i = tid; i < N2 * LE; i += nt) {
    const int n = i / LE, k = i % LE;
    float v = 0.f;
    if (n < K1) v = loc[LOC_PW + n * LE + k];
    else if (n < K1 + 4) v = loc[LOC_ZW + k * 4 + (n - K1)];
    __half hi, lo;
    umma::split_f16(v, hi, lo);
    const uint32_t off = umma::elem_off(n, k, (uint32_t)N2 * 16u);
    *reinterpret_cast<__half*>(op2 + off) = hi;
    *reinterpret_cast<__half*>(op2 + N2 * 64 + off) = lo;
  }
}

// W[N][K] (fp32, leading dimension ld) -> fp16 hi/lo B-operand tiles for tc_gemm_kernel
__global__ void split_weights_kernel(const float* __restrict__ w, int N, int K, int ld, uint8_t* __restrict__ out) {
  const long long total = (long long)N * K;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int n = (int)(i / K), k = (int)(i % K);
    __half hi, lo;
    umma::split_f16(w[(long long)n * ld + k], hi, lo);
    uint8_t* tile = out + ((long long)(n >> 7) * (K >> 6) + (k >> 6)) * 32768;
    const uint32_t off = umma::elem_off(n & 127, k & 63, 2048);
    *reinterpret_cast<__half*>(tile + off) = hi;
    *reinterpret_cast<__half*>(tile + 16384 + off) = lo;
  }
}

}  // namespace elg

using namespace elg;

extern "C" {

int elg_abi_version(void) { return ELG_ABI_VERSION; }
const char* elg_last_error(void) { return g_err; }
uint64_t elg_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int elg_weight_layout(const elg_model_desc* d, elg_weight_layout_t* L) {
  int rc = check_desc(d);
  if (rc) return rc;
  ELG_REQUIRE(L != nullptr, ELG_EINVAL, "layout out pointer is NULL");
  memset(L, 0xff, sizeof(*L));
  const bool cvrp = d->problem == ELG_CVRP;
  const int F = d->ff, F_loc = cvrp ? 3 : 2;
  int64_t o = 0;
  auto take = [&](int64_t n) { int64_t r = o; o += (n + 3) & ~(int64_t)3; return r; };   // 16-byte aligned slots
  if (cvrp) {
    L->emb_depot_w = take(E * 2);
    L->emb_depot_b = take(E);
    L->emb_node_w = take(E * 3);
  } else {
    L->emb_node_w = take(E * 2);
  }
  L->emb_node_b = take(E);
  for (int l = 0; l < d->layers; ++l) {
    auto& y = L->layer[l];
    y.wq = take(E * E); y.wk = take(E * E); y.wv = take(E * E);      // contiguous: one [3E][E] GEMM operand
    y.wo = take(E * E); y.bo = take(E);
    y.n1w = take(E); y.n1b = take(E);
    y.w1 = take((int64_t)F * E); y.b1 = take(F);
    y.w2 = take((int64_t)E * F); y.b2 = take(E);
    y.n2w = take(E); y.n2b = take(E);
  }
  if (!cvrp) L->dec_wq_first = take(E * E);
  L->dec_wq_last = take((int64_t)E * (cvrp ? E + 1 : E));
  L->dec_wk = take(E * E); L->dec_wv = take(E * E);
  L->dec_wo = take(E * E); L->dec_bo = take(E);
  L->loc_token = take(LE);
  L->loc_we = take(LE * F_loc); L->loc_be = take(LE);
  L->loc_wq = take(LE * LE); L->loc_wk = take(LE * LE); L->loc_wv = take(LE * LE);
  L->loc_wo = take(LE * LE); L->loc_bo = take(LE);
  L->total = o;
  return ELG_OK;
}

int64_t elg_derived_floats(const elg_model_desc* d) { return check_desc(d) ? -1 : (int64_t)derived_total(d->layers, d->ff); }

int elg_prepare_model(const elg_model_desc* d, const float* weights, float* derived, void* stream) {
  elg_weight_layout_t L;
  int rc = elg_weight_layout(d, &L);
  if (rc) return rc;
  ELG_REQUIRE(weights && derived, ELG_EINVAL, "NULL weights/derived");
  cudaStream_t st = (cudaStream_t)stream;
  prepare_kernel<<<1, 256, 0, st>>>(*d, L, weights, derived);
  ELG_LAUNCH_OK();
  // No local policy (model_params['ensemble'] False, or the reference's decoder before add_local_policy: the warm-up
  // phase of `training: joint`, CVRP/models.py:409-413): every local table is zero, so the decode kernels add exactly
  // 0 to the global score + distance penalty whatever the local weight slots hold.
  if (!(d->flags & ELG_FLAG_ENSEMBLE)) ELG_CUDA_OK(cudaMemsetAsync(derived + DER_LOC, 0, sizeof(float) * LOC_TOTAL, st));
  // pre-split every GEMM weight into tcgen05 operand tiles (read back by TMA in tc_gemm_kernel)
  auto split = [&](const float* w, int N, int K, long long off_floats) -> int {
    split_weights_kernel<<<148, 256, 0, st>>>(w, N, K, K, reinterpret_cast<uint8_t*>(derived + off_floats));
    ELG_LAUNCH_OK();
    return ELG_OK;
  };
  for (int l = 0; l < d->layers; ++l) {
    long long o = split_off_layer(l, d->ff);
    if ((rc = split(weights + L.layer[l].wq, 3 * E, E, o))) return rc;          // Wq|Wk|Wv are contiguous
    o += 3LL * E * E;
    if ((rc = split(weights + L.layer[l].wo, E, E, o))) return rc;
    o += (long long)E * E;
    if ((rc = split(weights + L.layer[l].w1, d->ff, E, o))) return rc;
    o += (long long)d->ff * E;
    if ((rc = split(weights + L.layer[l].w2, E, d->ff, o))) return rc;
  }
  long long o = split_off_dec(d->layers, d->ff);
  if ((rc = split(derived + DER_WK4, E, E, o))) return rc;
  if ((rc = split(weights + L.dec_wv, E, E, o + 1LL * E * E))) return rc;
  if ((rc = split(derived + DER_WQN, E, E, o + 2LL * E * E))) return rc;
  if ((rc = split(derived + DER_WQF, E, E, o + 3LL * E * E))) return rc;
  return ELG_OK;
}

}  // extern "C"
