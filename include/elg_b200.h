/*
 * elg_b200.h — C ABI of the B200-native ELG rollout path (libelg_b200.so).
 *
 * Drop-in boundary.  The reference (gaocrr/ELG) has no FFI layer: its hot path is
 * reached through Python classes.  Each entry point below replaces one of those
 * Python-level operations (cited as file:line under the reference tree) and is
 * what a ctypes binding inside the reference would call; INTEGRATION.md shows the
 * stubs.  Conventions:
 *   - every pointer is a DEVICE pointer unless its name ends in _host;
 *   - tensors are dense, row-major, fp32 unless stated; indices are int32;
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*); no entry
 *     point synchronises the device;
 *   - the return value is 0 on success, a negative ELG_E* code for argument /
 *     capability errors, or a positive cudaError_t; elg_last_error() describes it;
 *   - the caller owns every buffer; nothing is allocated behind the ABI.
 *
 * "B" below is the number of aug-instances (instances x augmentation factor, row
 * index a*n+i as in the reference's augment_xy_data_by_8_fold), "M" the POMO width
 * (rows per aug-instance), "N1" the node count (problem_size+1 with the depot at
 * index 0 for CVRP, problem_size for TSP).
 */
#ifndef ELG_B200_H
#define ELG_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ELG_ABI_VERSION 4   /* 2: training path, data generators; 3: elg_tables.et / .ws (streamed tensor-core decode);
                               4: elg_two_opt, then elg_cvrp_local_search, then elg_tsp_local_search, then
                                  elg_cvrp_local_search_ex (purely additive,
                                  so the version stays 4: a library without one fails on the missing symbol when the
                                  binding loads) */

enum { ELG_TSP = 0, ELG_CVRP = 1 };
enum { ELG_GREEDY = 0, ELG_SAMPLE = 1 };
enum {
  ELG_FLAG_ENSEMBLE = 1,          /* model_params['ensemble'] and the local policy is present (decoder.local); off = global
                                     policy + distance penalty only: local tables are zeroed, local parameters get no gradient */
  ELG_FLAG_DISTANCE_PENALTY = 2,  /* model_params['distance_penalty']  */
  ELG_FLAG_POSITIONAL = 4,        /* model_params['positional']        */
  /* kernel selection for elg_rollout / elg_decode_step (diagnostics; default = automatic) */
  ELG_FLAG_ATTN_FP32 = 8,         /* always the fp32-pipe attention kernel (rollout.cu)                     */
  ELG_FLAG_ATTN_TENSOR = 16       /* tensor-core attention kernel (rollout_tc.cu) whenever it is eligible   */
};
enum {
  ELG_OK = 0,
  ELG_EINVAL = -1,       /* bad argument                                         */
  ELG_EUNSUPPORTED = -2, /* model/problem shape outside what the kernels support */
  ELG_ENOMEM = -3        /* workspace too small                                  */
};

/* model_params of the reference's config.yml (CVRP/config.yml:32-48, TSP/config.yml:31-47). */
typedef struct elg_model_desc {
  int32_t problem;      /* ELG_TSP | ELG_CVRP                        */
  int32_t emb;          /* embedding_dim            (128)            */
  int32_t heads;        /* head_num                 (8)              */
  int32_t qkv;          /* qkv_dim                  (16)             */
  int32_t ff;           /* ff_hidden_dim            (512)            */
  int32_t layers;       /* encoder_layer_num        (6)              */
  int32_t local_k;      /* local_size[0]            (40 cvrp/30 tsp) */
  int32_t local_emb;    /* local_att_hidden_dim     (32)             */
  int32_t local_heads;  /* local_att_head_num       (4)              */
  int32_t local_qkv;    /* local_att_qkv_dim        (8)              */
  float xi;             /* xi                       (-1)             */
  float clip;           /* logit_clipping           (50)             */
  int32_t flags;        /* ELG_FLAG_*                                */
} elg_model_desc;

/* Offsets (in floats) of each parameter inside the packed weight buffer.  All matrices keep
 * PyTorch's [out][in] layout.  Filled by elg_weight_layout(); names follow the reference
 * state_dict (CVRP/models.py:199-209,232-247,276-297,7-25; TSP/models.py:134-142,156-172,206-225). */
#define ELG_MAX_LAYERS 16
typedef struct elg_weight_layout_t {
  int64_t total;                  /* number of floats in the packed buffer */
  int64_t emb_depot_w, emb_depot_b;   /* cvrp: encoder.embedding_depot (E x 2), tsp: unused (-1) */
  int64_t emb_node_w, emb_node_b;     /* cvrp: encoder.embedding_node (E x 3); tsp: encoder.embedding (E x 2) */
  struct {
    int64_t wq, wk, wv;           /* E x E, no bias */
    int64_t wo, bo;               /* multi_head_combine */
    int64_t n1w, n1b;             /* first instance-norm affine */
    int64_t w1, b1, w2, b2;       /* feed-forward */
    int64_t n2w, n2b;
  } layer[ELG_MAX_LAYERS];
  int64_t dec_wq_first;           /* tsp only (E x E) */
  int64_t dec_wq_last;            /* cvrp: E x (E+1); tsp: E x E */
  int64_t dec_wk, dec_wv;         /* E x E */
  int64_t dec_wo, dec_bo;         /* decoder.multi_head_combine */
  int64_t loc_token;              /* cur_token_emb (e) */
  int64_t loc_we, loc_be;         /* init_emb (e x F, F = 3 cvrp / 2 tsp) */
  int64_t loc_wq, loc_wk, loc_wv; /* e x e */
  int64_t loc_wo, loc_bo;         /* multi_head_combine (e x e) */
} elg_weight_layout_t;

/* Device pointers describing one encoded batch (outputs of elg_encode, inputs of the decode path).
 * Replaces the tensors the reference caches on its modules: CVRPModel.encoded_nodes
 * (CVRP/CVRPModel.py:32), decoder.k / .v / .single_head_key (CVRP/models.py:300-308),
 * decoder.q_first (TSP/models.py:237-242) and env.dist (CVRP/CVRPEnv.py:148). */
typedef struct elg_tables {
  const float* xy;        /* [B][N1][2]   augmented, scaled coordinates                         */
  const float* demand;    /* [B][N1]      cvrp (demand[.,0] = 0); NULL for tsp                   */
  const float* unscaled;  /* [B][N1][2]   library instances: unscaled coordinates, else NULL     */
  float* enc;             /* [B][N1][E]   encoded nodes                                          */
  float* k;               /* [B][N1][E]   decoder keys, pre-scaled by log2(e)/sqrt(qkv)          */
  float* v;               /* [B][N1][E]   decoder values                                         */
  void* e;                /* score matrix E' = enc * Wo-fold / sqrt(E); elg_e_bytes() per batch:
                             resident variant: three fp16 hi/lo tcgen05 B operands per aug-instance,
                                               [B][E' | K' | V^T][2][..], N1p*512 bytes each (N1p = N1 rounded up to 16)
                             larger:                       fp32 [B][N1][E], 16-byte chunks XOR-swizzled by (j & 7)  */
  float* eb;              /* [B][N1]      score bias    enc . bo / sqrt(E)                       */
  float* qtab;            /* [B][N1][E]   per-node last-node query  Wq_last[:, :E] * enc         */
  float* qfirst;          /* [B][N1][E]   tsp: per-node first-node query; NULL for cvrp          */
  void* nbr;              /* neighbour lists sorted by (distance, index); elg_nbr_bytes() per batch:
                             resident variant (elg_rollout_resident() == 1): per node ELG_NBR_NODE_BYTES(N1) bytes =
                               uint8 [ELG_NBR_STRIDE] list, 8-way interleaved, then float2 [N1] (distance, angle) to every node,
                               then float4 [N1] per list entry in rank order: (distance, angle, demand, node id bits)
                             larger:                       uint16 [B][N1][ELG_NBR16_STRIDE(NL)], rank order  */
  void* et;               /* streaming variant only, may be NULL: K' / V / E' once more as tcgen05 B operands in tiles of
                             ELG_TILE_NODES nodes, [B][tiles][E' | K' | V^T][hi | lo], ELG_TILE_BYTES per tile
                             (elg_et_bytes() per batch); written by elg_encode when non-NULL; with it (and ws) greedy
                             rollouts of large instances run on the streamed tensor-core kernel (rollout_stc.cu)          */
  void* ws;               /* scratch of that kernel, elg_rollout_ws_bytes(): per-row bit masks (masked / visited /
                             neighbour), one word per 32 nodes; contents need not be preserved                           */
} elg_tables;

#define ELG_TILE_NODES 128                          /* nodes per operand tile of elg_tables.et        */
#define ELG_TILE_BYTES (3 * 65536)                  /* E' | K' | V^T, 32 KB hi + 32 KB lo each        */

#define ELG_NBR_STRIDE 128                          /* list bytes per node, resident variant          */
#define ELG_NBR_PAIR_BYTES(N1) (8 * (((N1) + 1) & ~1))                     /* pair features indexed by node id       */
#define ELG_NBR_NODE_BYTES(N1) (ELG_NBR_STRIDE + ELG_NBR_PAIR_BYTES(N1) + 16 * (N1))   /* list + pair features + rank-ordered records */
#define ELG_NBR16_STRIDE(NL) (((NL) + 63) & ~63)    /* uint16 entries per node, streaming variant     */
#define ELG_MAX_NODES_RESIDENT 112                  /* upper bound of the resident variant (also needs to fit smem) */
#define ELG_MAX_NODES 8192                          /* largest instance the rollout supports          */
#define ELG_MASK_WORDS(N1) (((N1) + 31) / 32)       /* uint32 words per row of every bit mask         */

/* ---- introspection ------------------------------------------------------------------- */
int elg_abi_version(void);
const char* elg_last_error(void);
/* number of kernels this library has launched since load (bench.py's gpu_launches) */
uint64_t elg_launch_count(void);

/* ---- weights ---------------------------------------------------------------------------
 * elg_weight_layout: where each state_dict tensor goes inside the packed buffer
 *   (replaces model.load_state_dict, CVRP/test.py:75-78).
 * elg_derived_floats / elg_prepare_model: one-time fold of the decoder / local-policy
 *   weights into the tables the decode kernel reads (constant local query, positional
 *   tables, Wq_last split into node and load parts, Wo folded into the score matrix). */
int elg_weight_layout(const elg_model_desc* desc, elg_weight_layout_t* out_host);
int64_t elg_derived_floats(const elg_model_desc* desc);
int elg_prepare_model(const elg_model_desc* desc, const float* weights, float* derived, void* stream);

/* ---- problem loading ----------------------------------------------------------------------
 * x8 augmentation + depot/node concatenation: CVRPEnv.load_random_problems (CVRP/CVRPEnv.py:125-150),
 * TSPEnv.load_random_problems (TSP/TSPEnv.py:53-67), augment_xy_data_by_8_fold (CVRP/utils.py:69-87).
 * depot may be NULL (tsp).  aug is 1 or 8.  Outputs: xy [aug*n][N1][2], demand [aug*n][N1]. */
int elg_load_problems(int problem, const float* depot_xy, const float* node_xy, const float* node_demand,
                      int n, int n_nodes, int aug, float* xy_out, float* demand_out, void* stream);
/* full pairwise distance matrix [B][N1][N1] (env.dist / reset_state.dist); API compatibility only */
int elg_pairwise_dist(const float* xy, int B, int N1, float* dist_out, void* stream);

/* ---- encoder + decoder caches -----------------------------------------------------------
 * model.pre_forward: CVRP_Encoder.forward + decoder.set_kv (CVRP/CVRPModel.py:21-34,
 * CVRP/models.py:211-229,249-269,300-308; TSP/TSPModel.py:21-24, TSP/models.py:144-194,227-235),
 * plus the per-node query tables and distance-sorted neighbour lists the decode kernel uses. */
size_t elg_encode_workspace_bytes(const elg_model_desc* desc, int B, int N1);
int elg_encode(const elg_model_desc* desc, const float* weights, const float* derived, const elg_tables* t,
               int B, int N1, void* workspace, size_t workspace_bytes, void* stream);

/* ---- rollout ----------------------------------------------------------------------------
 * The whole construction loop of utils.rollout (CVRP/utils.py:7-29, TSP/utils.py:7-26):
 * env.reset, then per step get_cur_feature/get_local_feature + one_step_rollout + env.step,
 * and the final reward (CVRPEnv._get_reward / compute_unscaled_reward, CVRP/CVRPEnv.py:251-288;
 * TSPEnv._get_travel_distance / compute_unscaled_distance, TSP/TSPEnv.py:158-184).
 *   start_nodes [M]      POMO start permutation (python random.sample on the host)
 *   tours [B][M][t_max]  int16, must be zero-filled by the caller; t_max >= 2*N1+2 (cvrp) / N1 (tsp)
 *   reward [B][M]        minus tour length (rounded unscaled length if t->unscaled != NULL)
 *   n_steps [B*tiles]    zero-initialised by the caller; entry [b*tiles + tile] = steps that row tile ran (tiles =
 *                        elg_rollout_tiles(); unused entries stay 0); the batch length T is the maximum
 *   logp [B][M]          sample mode: sum of log-probabilities of the sampled actions (may be NULL)
 *   work_counter         one zero-initialised int32 (dynamic CTA scheduler)
 * elg_rollout_tiles() returns the number of row tiles per aug-instance used for (B, M, N1);
 * elg_nbr_bytes() / elg_e_bytes() the sizes of elg_tables.nbr / .e.  Sampling mode needs N1 <= 128.
 * Sampled decision (elg_rollout and elg_decode_step, mode = ELG_SAMPLE) of row m of aug-instance b: x = word 0 of
 * Philox4x32-10 with counter (grow lo, grow hi, step lo, step hi), grow = b*M + m, and key (seed lo, seed hi);
 * u = ((x >> 8) + 0.5f) * 2^-24 in fp32, in [2^-25, 1]; the pick is the first node in node-index order with p > 0 and
 * running sum of p >= u * sum of p (inverse CDF of softmax(logits)), or the last node with p > 0 when fp32 rounding
 * leaves every running sum below u * sum.  elg_rollout uses the tour position t as the step (cvrp: t = 0 depot and
 * t = 1 start node are forced, sampled from t = 2; tsp: sampled from t = 1); elg_decode_step uses its step argument. */
int elg_rollout_tiles(const elg_model_desc* desc, int B, int M, int N1);
int elg_rollout_resident(const elg_model_desc* desc, int N1);   /* 1 = resident variant, 0 = streaming, <0 = error */
size_t elg_nbr_bytes(const elg_model_desc* desc, int B, int N1);
size_t elg_e_bytes(const elg_model_desc* desc, int B, int N1);
size_t elg_et_bytes(const elg_model_desc* desc, int B, int N1);              /* 0 for resident instances */
size_t elg_rollout_ws_bytes(const elg_model_desc* desc, int B, int M, int N1);   /* 0 for resident instances */
int elg_rollout(const elg_model_desc* desc, const float* derived, const elg_tables* t, int B, int M, int N1,
                const int32_t* start_nodes, int mode, uint64_t seed, int t_max, int16_t* tours, float* reward,
                int32_t* n_steps, float* logp, int32_t* work_counter, void* stream);

/* ---- single decode step -----------------------------------------------------------------
 * model.one_step_rollout for the non-forced steps (CVRP/CVRPModel.py:52-73, TSP/TSPModel.py:40-62)
 * = _get_encoding + Decoder.forward + local_policy_att.forward + argmax / multinomial.
 *   cur [B][M] int32; load [B][M] (cvrp); first [B][M] int32 (tsp);
 *   mask_bits [B][M][ELG_MASK_WORDS(N1)] uint32, bit j set = node j masked (-inf in the reference's ninf_mask)
 *   selected [B][M] int32 out; prob [B][M] out (sample mode, may be NULL);
 *   logits [B][M][N1] out (masked logits = input of the reference's final softmax), may be NULL */
int elg_decode_step(const elg_model_desc* desc, const float* derived, const elg_tables* t, int B, int M, int N1,
                    const int32_t* cur, const float* load, const int32_t* first, const uint32_t* mask_bits,
                    int mode, uint64_t seed, uint64_t step, int32_t* selected, float* prob, float* logits,
                    void* stream);

/* ---- environment step ---------------------------------------------------------------------
 * CVRPEnv.step (CVRP/CVRPEnv.py:190-249) / TSPEnv.step (TSP/TSPEnv.py:108-133) on bit-mask state.
 *   visited_bits, mask_bits [B][M][ELG_MASK_WORDS(N1)] uint32 in/out; load [B][M] in/out; finished [B][M] uint8 in/out
 *   ninf_mask [B][M][N1] optional fp32 {0,-inf} view for API compatibility (may be NULL)
 *   n_unfinished: one int32, incremented per unfinished row (caller zeroes it) */
int elg_env_step(int problem, const float* demand, int B, int M, int N1, const int32_t* selected, float* load,
                 uint32_t* visited_bits, uint32_t* mask_bits, uint8_t* finished, float* ninf_mask,
                 int32_t* n_unfinished, void* stream);

/* ---- features (API compatibility) -------------------------------------------------------
 * CVRPEnv.get_cur_feature (CVRP/CVRPEnv.py:291-318) / TSPEnv.get_local_feature (TSP/TSPEnv.py:135-156):
 * cur_dist, cur_theta [B][M][N1], rel_xy [B][M][N1][2], norm_demand [B][M][N1] (cvrp, may be NULL). */
int elg_cur_feature(const float* xy, const float* demand, const float* load, const int32_t* cur, int B, int M,
                    int N1, float* cur_dist, float* cur_theta, float* rel_xy, float* norm_demand, void* stream);

/* ---- tour length ---------------------------------------------------------------------------
 * closed-tour length of [B][M][T] int64 tours over xy [Bxy][N1][2] (Bxy = B, or 1 = shared by all
 * aug-instances as in TSPEnv.compute_unscaled_distance); round_edges applies rint() per edge. */
int elg_tour_length(const float* xy, int Bxy, const int64_t* tours, int B, int M, int T, int N1, int round_edges,
                    float* out, void* stream);

/* ---- 2-opt local search ------------------------------------------------------------------------
 * Best-improvement 2-opt on R tours, refined in place; the counterpart of the reference's batched_two_opt_torch
 * (TSP/utils.py:28-70, CVRP/utils.py:31-67), except that every tour stops on its own.
 *   xy [Bxy][N1][2]   coordinates; inst [R] int32 picks the xy instance of each tour (NULL: r when Bxy == R, 0 when Bxy == 1)
 *   tours [R][L]      int16 node ids.  tsp: positions 0..N1-1 hold a permutation, closed implicitly (L >= N1; positions
 *                     N1.. are ignored and left as they are).  cvrp: a rollout row (depot visits as 0, trailing zero
 *                     padding), closed implicitly, L <= 2*N1+2.
 *   A move picks positions i < j, reverses positions i+1..j and gains d(t_i,t_j) + d(t_i+1,t_j+1) - d(t_i,t_i+1) -
 *   d(t_j,t_j+1) (j+1 wraps to 0); d is the reward's segment length, rint()-ed per edge when round_edges is set.  Every
 *   move evaluates all admissible pairs and applies the smallest gain (ties: lowest i*L + j) if it is below -1e-6, at most
 *   max_iterations times.  tsp: admissible j >= i+2 except (0, N1-1), so position 0 never moves.  cvrp: admissible j >= i+2
 *   with positions i+1..j all customers, so every move stays inside one route and every route keeps its customers (and its load).
 *   iterations [R]    moves applied;  length [R]  closed length of the refined tour, summed as elg_tour_length sums it */
int elg_two_opt(int problem, const float* xy, int Bxy, int N1, const int32_t* inst, int16_t* tours, int R, int L,
                int round_edges, int max_iterations, int32_t* iterations, float* length, void* stream);

/* ---- TSP local search: 2-opt and Or-opt ------------------------------------------------------------
 * Best-improvement local search on R TSP tours, refined in place; every tour stops on its own.
 *   xy, Bxy, N1, inst, tours [R][L], round_edges, max_iterations, iterations [R]: as elg_two_opt with problem = ELG_TSP
 *   (positions 0..N1-1 a permutation, closed implicitly; positions N1.. ignored and left as they are; position 0 never
 *   moves).  d is the reward's seglen, rint()-ed per edge when round_edges is set; e_p = d(t_p, t_p+1), p+1 wrapping to 0.
 * Move variants, keyed v*N1^2 + i*N1 + j:
 *   v = 0, 2-opt, exactly the TSP move of elg_two_opt: i < j, j >= i+2, not (0, N1-1); reverses positions i+1..j;
 *          gain (d(t_i,t_j) - e_i) + (d(t_i+1,t_j+1) - e_j).
 *   v = 1..5, Or-opt: move the segment at positions i..i+s-1 onto the edge (t_j, t_j+1); v = 1: s = 1; v = 2 / 3: s = 2
 *          forward / reversed; v = 4 / 5: s = 3 forward / reversed.  Admissible for 1 <= i, i+s-1 <= N1-1 and
 *          j in 0..N1-1 outside {i-1, .., i+s-1} (either side of the segment); only s <= max_segment (0..3) is evaluated.
 *          Gain ((d(t_i-1, t_i+s) - e_i-1) - e_i+s-1) + ((d(t_j, a) - e_j) + d(b, t_j+1)), i+s wrapping to 0, with
 *          (a, b) = (t_i, t_i+s-1) forward and (t_i+s-1, t_i) reversed.
 * Gains are fp32 in the order written.  Every iteration evaluates every admissible variant and applies the smallest gain,
 * ties to the lowest key, if it is below -1e-6, at most max_iterations times.  max_segment = 0 runs
 * elg_two_opt(ELG_TSP).  length is the closed length of the returned tour as elg_tour_length sums it.
 * N1 <= 8192 (shared memory: 14*N1 bytes). */
int elg_tsp_local_search(const float* xy, int Bxy, int N1, const int32_t* inst, int16_t* tours, int R, int L,
                         int max_segment, int round_edges, int max_iterations, int32_t* iterations, float* length,
                         void* stream);

/* ---- capacity-aware CVRP local search ------------------------------------------------------------
 * Best-improvement local search on R CVRP solutions, refined in place; every row stops on its own.
 *   xy [Bxy][N1][2], inst, round_edges, max_iterations, iterations [R], length [R]: as elg_two_opt
 *   demand [Bxy][N1]  int32 demand units, demand[., 0] = 0; capacity in the same units.  A route is feasible iff the
 *                     integer sum of its demands is <= capacity; there is no tolerance.  Input routes must be feasible.
 *   tours [R][L]      int16 rollout rows: position 0 the depot, every customer 1..N1-1 exactly once, depot visits as 0,
 *                     trailing zero padding, L <= 2*N1+2.  The output row is canonical even without a move: routes in
 *                     their order, each preceded by one 0, no empty route, zero padding to L.
 *   max_segment       1, 2 or 3: the longest chain of customers an Or-opt move (types 4..7) carries; 1 evaluates
 *                     types 0..3 only.  Any other value is ELG_EINVAL.
 * A route is a maximal run of customers.  Positions refer to the current canonical row, P = 1 + last customer position,
 * e_p = d(t_p, t_p+1) with t_P = 0:
 *   type 0, 2-opt inside a route: reverse positions i+1..j (j >= i+2), all customers of one route.
 *   type 1, relocate: move the customer at i onto the edge (t_j, t_j+1), j < P, j not i-1 or i; feasible within its
 *           route, or if the target route's load + its demand <= capacity.  A route emptied by the move disappears.
 *   type 2, swap: exchange the customers at i < j of two different routes; both new loads <= capacity.
 *   type 3, 2-opt*: cut positions i < j (a route's depot position or a customer) of different routes A and B;
 *           A' = A[..i] + B(j..] takes A's slot, B' = B[..j] + A(i..] takes B's; both loads <= capacity; an empty
 *           result disappears, so two routes can merge.
 *   types 4 / 5 (s = 2) and 6 / 7 (s = 3), Or-opt: move the segment at positions i..i+s-1, all customers (so one route),
 *           onto the edge (t_j, t_j+1), forward / reversed; j < P, j not in i-1..i+s-1, s <= max_segment.  Feasible
 *           within its route, or if the target route's load + the segment's load <= capacity.  Gain
 *           ((d(t_i-1, t_i+s) - e_i-1) - e_i+s-1) + ((d(t_j, a) - e_j) + d(b, t_j+1)), fp32 in that order, with
 *           (a, b) = (t_i, t_i+s-1) forward and (t_i+s-1, t_i) reversed.  A segment that is its whole route empties it
 *           and the route disappears.
 * No move opens a route.  Gains of types 0..3 are added minus removed edges of d (the reward's seglen, rint()-ed when
 * round_edges is set).  Every iteration evaluates every admissible move and applies the smallest gain, ties to the
 * lowest type*L^2 + i*L + j (unsigned: up to 8*L^2 - 1), if it is below -1e-6, at most max_iterations times.  length is
 * the closed length of the returned row as elg_tour_length sums it.  N1 <= 8192 (shared memory: 12*N1 + 8*L bytes). */
int elg_cvrp_local_search_ex(const float* xy, int Bxy, int N1, const int32_t* demand, int32_t capacity,
                             const int32_t* inst, int16_t* tours, int R, int L, int max_segment, int round_edges,
                             int max_iterations, int32_t* iterations, float* length, void* stream);

/* elg_cvrp_local_search_ex with max_segment = 1 (types 0..3). */
int elg_cvrp_local_search(const float* xy, int Bxy, int N1, const int32_t* demand, int32_t capacity, const int32_t* inst,
                          int16_t* tours, int R, int L, int round_edges, int max_iterations, int32_t* iterations,
                          float* length, void* stream);

/* ---- training path (REINFORCE with the POMO shared baseline) ----------------------------------
 * Replaces the body of the reference's training loop, CVRP/train.py:104-125 (TSP/train.py:100-122):
 *   model.pre_forward            -> elg_encode_train   (elg_encode that also keeps every layer's activations)
 *   rollout(eval_type='sample')  -> elg_rollout(mode = ELG_SAMPLE), which records tours, rewards and sum log p
 *   J = mean(-(r - mean_m r) * log_prob / max_m(r - mean_m r));  J.backward()
 *                                -> elg_reinforce_backward  (gradient of J w.r.t. every parameter, packed like the
 *                                   weight buffer of elg_weight_layout; overwritten, not accumulated)
 *   optimizer.step()             -> elg_adam_step  (torch.optim.Adam with L2 weight decay; CVRP/train.py:87)
 * followed by elg_prepare_model on the updated weights.  Data-parallel training all-reduces `grads` (NCCL) between
 * elg_reinforce_backward and elg_adam_step; grad_scale = 1 / world_size turns the sum into the mean.
 *   saved      elg_train_saved_bytes() bytes, 16-byte aligned; written by elg_encode_train
 *   tours      [B][M][t_max] int16 as written by elg_rollout;  T = number of steps of the rollout (max n_steps)
 *   reward     [B][M];  logp [B][M] (only used for the reported loss, may be NULL);  loss: one float (may be NULL)
 *   scale_norm config params.scale_norm (tsp: applied only if every instance has a non-zero maximum advantage)
 *   workspace  256-byte aligned, at least elg_train_workspace_bytes(..., chunk_steps = 1); a larger chunk_steps (up
 *              to 256; 832 bytes per row-step at 101 nodes) lets the decode backward process that many rollout steps per launch.  Its head holds the
 *              gradients of the decoder tables (float offsets from elg_train_workspace_layout: d E', d K', d V,
 *              d qtab, d qfirst, d eb, d w_load, local-policy accumulators), left in place for inspection.
 * Resident instances only (elg_rollout_resident() == 1: up to 112 nodes, 108 for cvrp with local_size 40), M <= 128. */
size_t elg_train_saved_bytes(const elg_model_desc* desc, int B, int N1);
int elg_encode_train(const elg_model_desc* desc, const float* weights, const float* derived, const elg_tables* t,
                     int B, int N1, void* saved, size_t saved_bytes, void* stream);
size_t elg_train_workspace_bytes(const elg_model_desc* desc, int B, int M, int N1, int t_max, int chunk_steps);
int elg_train_workspace_layout(const elg_model_desc* desc, int B, int M, int N1, int t_max, int64_t* out8);
int elg_reinforce_backward(const elg_model_desc* desc, const float* weights, const float* derived, const elg_tables* t,
                           const void* saved, int B, int M, int N1, const int16_t* tours, int t_max, int T,
                           const float* reward, const float* logp, int scale_norm, float* grads, float* loss,
                           void* workspace, size_t workspace_bytes, void* stream);
int elg_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, int64_t step,
                  float lr, float beta1, float beta2, float eps, float weight_decay, float grad_scale, void* stream);

/* ---- training-data generators ------------------------------------------------------------------
 * generate_vrp_data (CVRP/generate_data.py:9-92) / generate_tsp_data (TSP/generate_data.py:9-57) on the device.
 *   kind: 0 uniform, 1 cluster, 2 mixed (config.yml distribution.data_type); n_cluster = distribution.n_cluster
 *   (cluster) or n_cluster_mix (mixed); lower / upper / std as in config.yml; capacity = CAPACITIES[problem_size].
 * Outputs: depot_xy [n][2] and node_demand [n][n_nodes] (cvrp; NULL for tsp), node_xy [n][n_nodes][2].
 * Counter-based Philox streams keyed by (seed, instance): same distributions as the reference, not its bit stream. */
int elg_generate_problems(int problem, int kind, int n, int n_nodes, int n_cluster, float lower, float upper, float std,
                          float capacity, uint64_t seed, float* depot_xy, float* node_xy, float* node_demand, void* stream);

/* ---- diagnostics -----------------------------------------------------------------------------
 * One split-precision tcgen05 GEMM  D[128][n] = A[rows_a][k] * B[n][k]^T  (fp16 hi/lo operands, fp32
 * accumulation in TMEM; terms = 1: hi*hi only, 3: + hi*lo + lo*hi; alias: 64-row A operand whose upper
 * rows alias the next k-chunk).  Pins the UMMA descriptor / TMEM conventions the kernels rely on. */
int elg_selftest_umma(const float* a, const float* b, float* d, int rows_a, int n, int k, int alias, int terms,
                      void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ELG_B200_H */
