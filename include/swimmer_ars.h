/*
 * swimmer_ars.h -- C ABI of libswimmer_ars.so, the B200 (sm_100a) implementation of the
 * batched Coulom swimmer + Augmented Random Search hot path.
 *
 * This is the drop-in boundary: plain C, pointers and sizes only (no torch / C++ types).
 * The Python host layer (safe-exploration-with-simulator-in-rl-algorithms_b200/) binds these
 * symbols with ctypes and mirrors the reference's Python plugin surface on top of them.
 * Each entry point names the reference interface it replaces (paths relative to the
 * reference repository root).
 *
 * Conventions
 *   - every `double*` / `int*` data argument is a DEVICE pointer unless it says "host";
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream); all calls only
 *     enqueue work on that stream and return without synchronising;
 *   - return value: 0 = ok, negative = swm_status (swm_strerror gives text); no exceptions
 *     and no hidden device allocations cross this boundary;
 *   - observation layout is the reference's: [Gdot_x, Gdot_y, th_1, thd_1, ..., th_n, thd_n]
 *     (remy_swimmer_env.py:216-224, SwimmerEnvironment.cpp:109-116), row-major [B, 2n+2];
 *   - a linear policy is row-major [(n-1), (2n+2)] (ars/ars_agent.py:72-73).
 */
#ifndef SWIMMER_ARS_H
#define SWIMMER_ARS_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define SWM_API __attribute__((visibility("default")))
#else
#define SWM_API
#endif

#define SWM_ABI_VERSION 3
#define SWM_MIN_SEGMENTS 2
#define SWM_MAX_SEGMENTS 10

typedef enum {
  SWM_OK = 0,
  SWM_ERR_BAD_ARG = -1,        /* NULL / out-of-range argument */
  SWM_ERR_UNSUPPORTED = -2,    /* valid request this build has no kernel for */
  SWM_ERR_CUDA = -3,           /* a CUDA runtime call failed: swm_last_cuda_error() */
  SWM_ERR_NO_DEVICE = -4
} swm_status;

/* Dynamics variant. */
typedef enum {
  SWM_DYN_GYM = 0,    /* envs/gym_swimmer/swimmer/remy_swimmer_env.py:69-214: explicit Euler */
  SWM_DYN_RLGLUE = 1  /* rlglue/environment/SwimmerEnvironment.cpp:102-271: semi-implicit Euler,
                         literal 5n+2 system including its column/weight quirks */
} swm_variant;

/* Physical parameters of one swimmer model (host struct, passed by pointer, read during the call).
 * Replaces SwimmerEnv.__init__ kwargs (remy_swimmer_env.py:16-29) and the RL-Glue globals
 * n_seg,max_u,l_i,k,m_i,h_global,direction (SwimmerEnvironment.cpp:3-9). */
typedef struct {
  int32_t n;            /* number of segments, SWM_MIN_SEGMENTS..SWM_MAX_SEGMENTS */
  int32_t _pad;
  double l_i, m_i, k, h, max_u;
  double direction[2];
} swm_params_t;

/* How each environment of a rollout obtains its action. */
typedef enum {
  SWM_POLICY_FIXED_ACTION = 0, /* actions[B, n-1] held constant for all H steps (BASELINE config 2) */
  SWM_POLICY_EXPLICIT = 1,     /* policies[P, (n-1)(2n+2)], env e uses policy e / rollouts_per_policy */
  SWM_POLICY_PHILOX = 2,       /* W +/- nu*delta_k, delta regenerated in-kernel from Philox4x32-10;
                                  policy index q = e / rollouts_per_policy, direction k = dir0 + q/2,
                                  sign + for even q, - for odd q  (ars_agent.py:140-142 ordering) */
  SWM_POLICY_DELTAS = 3        /* as PHILOX but delta_k is read from deltas[D, (n-1)(2n+2)] (row q/2):
                                  lets a caller replay the reference's own MT19937 draws */
} swm_policy_mode;

/* Which rollout kernel runs a launch.  Both implement the same equations and differ by rounding only
 * (summation order); AUTO picks LANES for batches too small to fill the chip with one thread per env. */
typedef enum {
  SWM_KERNEL_AUTO = 0,
  SWM_KERNEL_THREAD = 1, /* one thread = one environment (throughput: BASELINE configs 2 and 5) */
  SWM_KERNEL_LANES = 2,  /* one environment spread over 4/8/16 lanes, lane = segment (latency: the 2,048-env
                            ARS iteration of config 3, the 512-env safe-exploration rollouts of config 4);
                            gym dynamics without per-step screening / clipping, else SWM_ERR_UNSUPPORTED
                            (LANES2 / LANES3 also run per-step screening of plain linear policies) */
  SWM_KERNEL_LANES2 = 3, /* LANES cut into two warps per lane group (main warp + factorisation warp on separate
                            SM sub-partitions): batches so small that sub-partitions would otherwise idle */
  SWM_KERNEL_LANES3 = 4  /* LANES2 with two factorisation warps taking alternate steps: the smallest batches */
} swm_rollout_kernel;

/* Distribution of the Philox perturbations. */
typedef enum {
  SWM_DELTA_UNIFORM_PM1 = 0, /* 2*U[0,1)-1  (ars_agent.py:137, safe_ars/ars.py:84) */
  SWM_DELTA_UNIFORM_01 = 1   /* U[0,1)      (rlglue/agent/SwimmerAgent.py:208) */
} swm_delta_dist;

/* Philox4x32-10 addressing shared by the rollout and the update kernels (and the oracle):
 * key = (seed lo32, seed hi32), counter = (pair j, direction k, iteration, stream);
 * one call yields elements 2j and 2j+1 of delta_k;  u = ((a>>5)*2^26 + (b>>6)) * 2^-53. */
typedef struct {
  uint64_t seed;
  uint32_t iteration;
  uint32_t dir0;       /* global index of this shard's first direction */
  int32_t dist;        /* swm_delta_dist */
  int32_t _pad;
  const uint32_t* iteration_dev; /* optional DEVICE counter: the kernels use iteration + *iteration_dev.
                                    Lets a captured CUDA graph of one ARS iteration be replayed: the
                                    graph's arguments are frozen, the counter lives in device memory
                                    and is advanced by swm_counter_add inside the graph. */
} swm_philox_t;

/* Per-step state-constraint screening (safe_ars/ars.py:111-153, Safe_ARS.isSafe/rollout) with the
 * built-in cost of safe_ars/experiment.py:44, cost(obs) = max_i |thd_i|. */
typedef struct {
  int32_t enabled;
  int32_t _pad;
  swm_params_t sim;       /* simulator model; n must equal the real model's n */
  double sim_thresh;      /* take the real step iff cost(sim step) <= sim_thresh */
  double real_thresh;     /* real steps with cost > real_thresh are counted in violations[] */
  int32_t* violations;    /* [B] or NULL */
  int32_t* frozen_at;     /* [B] or NULL: first step index judged unsafe, H if never */
} swm_screen_t;

/* One fused H-step rollout of B environments.  Replaces Environment.rollout
 * (ars/environment.py:37-57), Basic_ARS.rollout / Safe_ARS.rollout (safe_ars/ars.py:13-35,
 * 124-153) and the 2N-rollout loop of ARSAgent.runOneIteration (ars/ars_agent.py:140-172). */
typedef struct {
  int32_t variant;              /* swm_variant */
  int32_t policy_mode;          /* swm_policy_mode */
  int32_t normalize;            /* 0 = ARS V1; 1 = ARS V2: action = (W diag(inv_sigma)) (obs - mean)
                                   (ars/environment.py:31-35) */
  int32_t clip_actions;         /* 1 = clip to +-max_u (rlglue/agent/SwimmerAgent.py:192-196) */
  int32_t H;                    /* steps */
  int32_t rollouts_per_policy;  /* R >= 1 consecutive envs share one policy */
  int64_t B;                    /* number of environments */
  const double* actions;        /* FIXED_ACTION: [B, n-1] */
  const double* policies;       /* EXPLICIT: [B/R, (n-1)(2n+2)];  PHILOX/DELTAS: base W [(n-1)(2n+2)] */
  const double* deltas;         /* DELTAS: [B/(2R), (n-1)(2n+2)] */
  double nu;                    /* PHILOX/DELTAS: perturbation scale */
  swm_philox_t philox;
  const int32_t* dir_mask;      /* PHILOX/DELTAS, optional [B/(2R)]: directions with mask 0 are NOT
                                   rolled out (their returns are set to NaN) -- the reward-constraint
                                   safe exploration of ars_agent.py:144-159 */
  const double* mean;           /* [2n+2], normalize only */
  const double* inv_sigma;      /* [2n+2], normalize only: diag(cov)^(-1/2) */
  const double* init_state;     /* NULL = reset() (gym: remy_swimmer_env.py:58-67; rlglue: env_start
                                   cpp:39-42), else [B or R or 1, 2n+2] */
  int64_t init_state_count;     /* rows in init_state: env e uses row e % init_state_count */
  double init_perturb;          /* != 0: add init_perturb * U[0,1) to every entry of the initial state,
                                   Philox stream 1, counter (pair j, e % R, iteration, 1): the same R
                                   perturbed starts for every policy (declared synthetic extension for
                                   BASELINE config 5; the reference's reset() is deterministic) */
  double* returns;              /* [B] sum of rewards */
  double* final_state;          /* [B, 2n+2] or NULL */
  double* trajectory;           /* [H, B, 2n+2] time-major post-step observations, or NULL
                                   (saved_states of ars/environment.py:53) */
  double* stats_partial;        /* NULL, or [swm_rollout_stats_blocks(B), 2, 2n+2]: per-block
                                   sums of (x-pivot) and (x-pivot)^2 over all visited states */
  const double* stats_pivot;    /* [2n+2], required with stats_partial */
  swm_screen_t screen;
  int32_t accumulate_returns;   /* 1: returns[e] += this launch's sum instead of overwriting it.  Lets a caller
                                   cut one rollout into time-chunks (final_state of one launch = init_state of the
                                   next) and sub-batches on several streams, which removes the quantisation of
                                   mid-size batches over SM sub-partitions; chunk lengths that are multiples of 64
                                   keep the visited states bit-identical to the single launch. */
  int32_t kernel;               /* swm_rollout_kernel: 0 = chosen from (B, n, SM count) */
  int32_t schedule_sub;         /* 0: the library decides between one plain launch and a chunked schedule (sub-batches x
                                   64-step-aligned time chunks on internal streams, joined back into `stream`; needs
                                   final_state as the chaining buffer; results: states bit-identical, returns equal up to
                                   the rounding of the partial sums) from (B, n, SM count) -- see swm_rollout_schedule;
                                   -1: always one plain launch;  1..32: this many sub-batches (SWM_ERR_UNSUPPORTED if the
                                   request cannot be scheduled: trajectory / screening / no final_state / H <= chunk) */
  int32_t schedule_chunk;       /* steps per chunk when schedule_sub > 0: a positive multiple of 64 */
} swm_rollout_t;

SWM_API int swm_abi_version(void);
SWM_API const char* swm_strerror(int status);
SWM_API const char* swm_last_cuda_error(void);
SWM_API int swm_device_info(int* sm_count, int* cc_major, int* cc_minor); /* host out-pointers */
/* sizeof() of the ABI structs in this build, so that a binding can verify its own layout */
SWM_API int swm_abi_struct_sizes(int* params, int* philox, int* screen, int* rollout);

/* Batched single step.  Replaces SwimmerEnv.step / next_observation (remy_swimmer_env.py:41-93)
 * and updateState (SwimmerEnvironment.cpp:102-137) for B independent environments.
 * state_out may alias state_in.  reward may be NULL. */
SWM_API int swm_step_batched(const swm_params_t* params, int variant, const double* state_in,
                     const double* action, double* state_out, double* reward, int64_t B,
                     void* stream);

/* Batched single step with SEVERAL models in one launch: environment e uses params[e / envs_per_model]
 * (host array of n_models <= SWM_MAX_MODELS_PER_STEP structs with the same n).  This is the shape of the
 * parameter-estimation objective Estimator.I (ars/estimator.py:36-62): every CMA-ES candidate
 * (m_i, l_i, k) predicts the same recorded states one step ahead.  gym variant only. */
#define SWM_MAX_MODELS_PER_STEP 24
SWM_API int swm_step_batched_models(const swm_params_t* params, int n_models, int64_t envs_per_model,
                                    const double* state_in, const double* action, double* state_out,
                                    double* reward, void* stream);

/* Accelerations only (compute_accelerations, remy_swimmer_env.py:95-114 / cpp:139-226):
 * acc[B, n+2] = [Gdd_x, Gdd_y, thdd_1..thdd_n]. */
SWM_API int swm_accelerations_batched(const swm_params_t* params, int variant, const double* state,
                              const double* action, double* acc, int64_t B, void* stream);

SWM_API int swm_rollout(const swm_params_t* params, const swm_rollout_t* cfg, void* stream);
/* number of per-block rows swm_rollout writes into stats_partial for this cfg when launched on `stream` of the
 * current device (depends on the kernel and the schedule it will choose; the schedule may differ while `stream`
 * is capturing a CUDA graph) */
SWM_API int64_t swm_rollout_stats_blocks(const swm_params_t* params, const swm_rollout_t* cfg, void* stream);
/* which kernel swm_rollout would run for this cfg on the current device: SWM_KERNEL_THREAD / _LANES,
 * or a negative swm_status */
SWM_API int swm_rollout_kernel_choice(const swm_params_t* params, const swm_rollout_t* cfg);
/* the schedule swm_rollout would use on `stream`: *n_sub = 0 for one plain launch, else sub-batches x *chunk
 * steps (finer while the stream is capturing a CUDA graph: replayed launches have no host cost) */
SWM_API int swm_rollout_schedule(const swm_params_t* params, const swm_rollout_t* cfg, void* stream, int* n_sub,
                                 int* chunk);

/* Deterministic Welford bookkeeping for ARS V2 (replaces np.mean / np.cov over the growing
 * saved_states list, ars/ars_agent.py:179-182).  A statistics record is
 * [count, mean[F], M2[F]] (1+2F doubles).
 *  - swm_stats_finalize: sums the per-block partial rows in a fixed order and converts them into a
 *    record (count, mean, M2) -- `out_record`.  count = samples, or samples * (*units) when the
 *    optional device int32 `units` is given (e.g. samples = 2*R*H per direction, units = the
 *    number of directions that survived screening).
 *  - swm_stats_merge: folds `n_records` records (contiguous, e.g. one per rank after an
 *    all-gather, merged in index order) into `running` (Chan et al.), then writes
 *    mean[F] and inv_sigma[F] = (M2/(count-1))^(-1/2) if those pointers are non-NULL. */
SWM_API int swm_stats_finalize(const double* partial, int64_t n_blocks, int n_features, double samples,
                               const int32_t* units, const double* pivot, double* out_record,
                               void* stream);
SWM_API int swm_stats_merge(double* running, const double* records, int n_records, int n_features,
                    double* mean_out, double* inv_sigma_out, void* stream);

/* Mean of each group of R consecutive returns (per-direction return when R rollouts share a
 * policy; BASELINE config 5). out[B/R]. */
SWM_API int swm_reduce_returns(const double* returns, int64_t n_groups, int R, double* out, void* stream);

/* order[N]: directions sorted by max(r+_k, r-_k) descending == sort_directions
 * (ars_agent.py:97-108, safe_ars/ars.py:37-46).  Ties: higher index first
 * (np.argsort(kind='stable')[::-1]); NaN keys first.  returns[2N] = [r+_0, r-_0, r+_1, ...].
 * mask (optional, [N] int32): directions with mask==0 sort after all others (screened out). */
SWM_API int swm_ars_topb(const double* returns, const int32_t* mask, int N, int32_t* order, void* stream);

/* update_policy (ars_agent.py:110-130, safe_ars/ars.py:48-65, rlglue/agent/SwimmerAgent.py:223-241):
 *   used    = order[0 .. n_order)            (order == NULL: identity, i.e. index order)
 *             if mask != NULL: only the first min(n_order, #mask!=0) entries (order must come from
 *             swm_ars_topb with the same mask, which sorts screened-out directions last)
 *   sigma_R = std of the 2*|used| returns with `ddof` (0: np.std, 1: statistics.stdev)
 *   W      += alpha * ( sum_{k in used} (r+_k - r-_k) delta_k / (divisor * sigma_R) )
 *             divisor <= 0 means |used| (safe_ars/ars.py:64 len(order)); ars_agent.py:128 passes b.
 * The three reference semantics (SURVEY appendix C) are therefore
 *   ars/ars_agent.py   : n_order = N, divisor = b, ddof = 0      (sorts, then uses ALL directions)
 *   safe_ars/ars.py    : n_order = b, divisor = 0 (=b), ddof = 0 (true top-b)
 *   rlglue agent       : order = NULL, n_order = b, divisor = b, ddof = 1
 * delta_k is regenerated from Philox (deltas == NULL; direction index dir0 + k) or read from
 * deltas[N, wsize].  If nothing is used W is unchanged (ars_agent.py:174).  sigma_out: optional
 * device double. */
SWM_API int swm_ars_update(double* W, int wsize, const double* returns, int N, const int32_t* order,
                           int n_order, const int32_t* mask, double divisor, int ddof, double alpha,
                           const swm_philox_t* philox, const double* deltas, double* sigma_out,
                           void* stream);

/* mask[k] = (sim_returns[2k] > threshold) && (sim_returns[2k+1] > threshold): the screening rule of
 * ars_agent.py:150-157 (a direction is rolled out in the real world only if both simulated
 * returns exceed the simulator threshold; a NaN return is screened out as well -- declared deviation from
 * the reference's `<=`).  n_pass: optional device int32 = number of survivors; n_pass_total: optional
 * device int64 running total (+= survivors), e.g. the screened fraction of a whole training run. */
SWM_API int swm_screen_mask(const double* sim_returns, int N, double threshold, int32_t* mask,
                            int32_t* n_pass, int64_t* n_pass_total, void* stream);

/* select_action for a batch (ars/environment.py:19-35): actions[B, n-1] = W_e obs_e (V1) or
 * (W_e diag(inv_sigma)) (obs_e - mean) (V2); env e uses policy e / rollouts_per_policy of
 * policies[P, (n-1)(2n+2)].  clip != 0 clips to +-max_u. */
SWM_API int swm_policy_actions(const swm_params_t* params, const double* obs, const double* policies,
                               int rollouts_per_policy, const double* mean, const double* inv_sigma,
                               int clip, double* actions, int64_t B, void* stream);

/* Writes delta_k (k = dir0 .. dir0+count-1) into out[count, wsize]: lets tests and the host API
 * see exactly the perturbations the kernels use. */
SWM_API int swm_philox_deltas(const swm_philox_t* philox, int count, int wsize, double* out, void* stream);

/* *counter += inc on the stream (device uint32): the iteration counter of swm_philox_t.iteration_dev. */
SWM_API int swm_counter_add(uint32_t* counter, uint32_t inc, void* stream);

/* curve[min(*index, capacity-1)] = mean of the non-NaN entries of x[n] (NaN if there is none):
 * the learning-curve entry of ARSAgent.runTraining (ars_agent.py:195-201: mean of the returns of the
 * directions that were rolled out), recorded on the device so that a training loop never has to
 * synchronise with the host.  index == NULL writes curve[0]. */
SWM_API int swm_record_nanmean(const double* x, int n, double* curve, const uint32_t* index,
                               uint32_t capacity, void* stream);

/* ---- Per-iteration record exchange of a sharded ARS iteration (SURVEY 8e) --------------------------------
 * Directions are sharded contiguously over `world` ranks (one process per GPU).  Each iteration every rank
 * packs ONE record [returns (2 n_local) | mask (n_local, optional) | count, mean[F], M2[F]], all ranks
 * exchange them, and every rank unpacks returns_all[2N] / mask_all[N] / records[world, 1+2F] for the
 * redundant, bit-identical ranking, update and Welford merge (replaces the 2N sequential rollouts'
 * `rewards.append` of ars_agent.py:161-172 and the cumulative np.mean/np.cov of :179-182 across ranks).
 *
 * swm_ars_pack_exchange does pack + exchange + unpack in ONE kernel launch:
 *   - h == NULL, gathered_world <= 1: single process, pack and unpack only;
 *   - h != NULL (world > 1): the record is stored into every rank's gather buffer over NVLink through
 *     CUDA-IPC peer pointers, epoch flags are published and awaited inside the kernel -- no NCCL call on
 *     the data path, so the whole iteration can be captured in a CUDA graph.  Setup (once): every rank
 *     calls swm_exchange_create, exports swm_exchange_ipc_handle (SWM_IPC_HANDLE_BYTES bytes), the host
 *     layer all-gathers the handles (torch.distributed / MPI / files) and passes the table to
 *     swm_exchange_open_peers.  A peer that does not answer within ~10 s sets a sticky status
 *     (swm_exchange_status) instead of hanging the device;
 *   - collective fallback (no peer access): call once with record_out set and gathered_world = world
 *     (pack only), all-gather record_out with the host's collective, then call with gathered_in. */
typedef struct swm_exchange swm_exchange_t;
#define SWM_IPC_HANDLE_BYTES 64
typedef struct {
  const double* returns_local;  /* [2 n_local R] per-env returns of this rank's rollouts */
  int32_t n_local;              /* directions owned by this rank */
  int32_t rollouts_per_policy;  /* R: record carries the mean over the R rollouts of a policy */
  const int32_t* mask_local;    /* [n_local] or NULL: screening mask of this rank's directions; the returns of a
                                   direction with mask 0 are packed as NaN whether or not its rollouts ran */
  const double* stats_partial;  /* [n_blocks, 2, F] from swm_rollout, or NULL (count 0) */
  int64_t n_blocks;
  int32_t n_features;           /* F = 2n+2, or 0 for ARS V1 (no statistics in the record) */
  int32_t gathered_world;       /* ranks in gathered_in / expected by the collective fallback */
  double samples;               /* states behind stats_partial (x *units if given) */
  const int32_t* units;         /* optional device int32 multiplier of samples */
  const double* pivot;          /* [F] */
  double* returns_all;          /* out [2 N] (NULL: pack only) */
  int32_t* mask_all;            /* out [N] or NULL */
  double* records;              /* out [world, 1+2F] or NULL */
  double* record_out;           /* out, optional: this rank's packed record [swm_pack_record_doubles] */
  const double* gathered_in;    /* in, optional: [gathered_world, record_doubles]; skips pack + exchange */
} swm_pack_t;
SWM_API int64_t swm_pack_record_doubles(int n_local, int has_mask, int n_features);
SWM_API int swm_exchange_create(int world, int rank, int64_t record_doubles, swm_exchange_t** out);
SWM_API int swm_exchange_ipc_handle(swm_exchange_t* h, void* handle_out /* host, SWM_IPC_HANDLE_BYTES */);
SWM_API int swm_exchange_open_peers(swm_exchange_t* h, const void* handles /* host, world x SWM_IPC_HANDLE_BYTES */);
SWM_API int swm_exchange_status(swm_exchange_t* h, uint64_t* epoch, uint64_t* status); /* host out; synchronises */
SWM_API int swm_exchange_destroy(swm_exchange_t* h);
SWM_API int swm_ars_pack_exchange(swm_exchange_t* h, const swm_pack_t* p, void* stream);

/* ---- The RL-Glue ARS experiment with the reference's literal step-level state machine -------------------
 * Replaces the four-process loop of rlglue/experiment/SwimmerExperiment.cpp:65-100 (2 N H training RL_steps
 * with "load state" every H steps, "freeze training", one H-step evaluation rollout per iteration) driving
 * rlglue/agent/SwimmerAgent.py:79-241 against rlglue/environment/SwimmerEnvironment.cpp.  The reference's
 * bookkeeping couples consecutive rollouts (see csrc/rlglue_protocol.cu), so an experiment is sequential: one
 * thread per replica.  state[replicas, swm_rlglue_protocol_state_doubles(n)] = [policy | pending action |
 * running total | iterations done]; all zeros = a fresh experiment (agent_start); calls continue where the
 * previous one stopped.  deltas: [iterations done + n_it, N, (n-1)(2n+2)] U[0,1) draws shared by all replicas
 * (replaying the agent's np.random.rand), or NULL: Philox, key seed + replica, counter (pair, direction,
 * iteration0 + iteration, 0). */
typedef struct {
  int32_t N, b, H, n_it;
  double alpha, nu;
  const double* deltas;
  uint64_t seed;
  uint32_t iteration0;
  int32_t _pad;
  double* state;    /* in/out */
  double* results;  /* out [replicas, n_it]: evaluation totals = the lines of rlglue/plot/results.txt */
  double* table;    /* out [replicas, n_it, 2N]: the agent's reward table at each update */
  int64_t replicas;
} swm_rlglue_protocol_t;
SWM_API int64_t swm_rlglue_protocol_state_doubles(int n);
SWM_API int swm_rlglue_protocol(const swm_params_t* params, const swm_rlglue_protocol_t* cfg, void* stream);

/* ---- Simulator-model estimation: prediction-error objective and CMA-ES on the device ---------------------
 * Replaces Estimator.I / estimate_real_env_param (ars/estimator.py:36-62, :89-110).  The objective of a
 * candidate x (d = 1..3 physical parameters) over K recorded trajectories of H observations is
 *   err(x) = sum_k sum_{t < H-1} || step_x(s_{k,t}, W_k s_{k,t}) - s_{k,t+1} ||_2
 * with the gym dynamics and the V1 policy product W_k s (as the reference, also for V2-recorded data).
 * A candidate is the base model with fields[i] replaced by x[i]; a candidate with m_i <= 0 or l_i <= 0 is
 * not stepped and gets +inf, and every non-finite sum becomes +inf.  Each err[c] is summed in a fixed order
 * (transitions within a CTA, then CTAs in index order) that depends on neither M nor the candidate's index:
 * results are bit-identical from run to run and permute with the candidates. */
#define SWM_MAX_CANDIDATES 1024
typedef enum { SWM_FIELD_M_I = 0, SWM_FIELD_L_I = 1, SWM_FIELD_K = 2 } swm_field;
typedef struct {
  const double* trajectories; /* [K, H, 2n+2] recorded observations */
  const double* policies;     /* [K, (n-1)(2n+2)] the policy that recorded each trajectory */
  int32_t K, H;               /* K >= 1, H >= 2 */
  int32_t d;                  /* unknowns, 1..3 */
  int32_t fields[3];          /* swm_field replaced by coordinate i < d; each field at most once */
  double* workspace;          /* [swm_prediction_error_workspace_doubles(K, H, M)] scratch of the two-pass sum */
} swm_estimate_data_t;
SWM_API int64_t swm_prediction_error_workspace_doubles(int K, int H, int M);
/* err[M] = err(candidates[c, 0..d)) for M (1..SWM_MAX_CANDIDATES) candidates, base->n in 2..10 */
SWM_API int swm_prediction_error(const swm_params_t* base, const swm_estimate_data_t* data,
                                 const double* candidates, int M, double* err, void* stream);

/* CMA-ES (Hansen, "The CMA Evolution Strategy: A Tutorial", 2016) with the tutorial's default strategy
 * parameters: mu = floor(lambda/2) positive log weights, c_sigma, d_sigma, c_c, c_1, c_mu, the h_sigma stall,
 * rank-one + rank-mu covariance update, cumulative step-size adaptation; no active (negative-weight) update.
 * All of its state is one device buffer of swm_cmaes_state_doubles(d, lambda) doubles, so that a CUDA graph of
 * several generations can be replayed.  Layout (offsets in doubles; L = 10 + ceil(30 d / lambda)):
 *   0 generation   1 status (swm_cmaes_status)   2 sigma   3 best f   4 max generations   5 tolfun   6 tolx
 *   7 mean[d]  7+d best x[d]  7+2d p_sigma[d]  7+3d p_c[d]  7+4d D[d] (sqrt of the eigenvalues of C)
 *   7+5d C[d*d]  7+5d+d^2 B[d*d] (eigenvectors in columns)  7+5d+2d^2 best-f history[L] (generation g at g % L)
 *   7+5d+2d^2+L z[lambda, d] (the last generation's standard normal draws)
 * Sampling: z ~ N(0, I) by Box-Muller (r = sqrt(-2 ln(1 - u0)), angle 2 pi u1) from Philox4x32-10, key = seed,
 * counter = (pair j, candidate c, generation, 2), u = the 53-bit uniforms of swm_philox_t; candidate
 * x_c = mean + sigma * B * (D .* z_c).  Update: rank by fitness ascending (+inf and NaN last, ties by lower
 * index), recombination, evolution paths, C and sigma, then C = B diag(D^2) B^T by cyclic Jacobi with a fixed
 * sweep count, best-ever tracking, and the stop tests (in this order): tolfun (range of the full best-f history
 * and this generation's fitness < tolfun), tolx (sigma sqrt(C_ii) < tolx and sigma |p_c,i| < tolx for all i),
 * condition (max D^2 / min D^2 > 1e14 or C not positive definite), max generations.  Once status != RUNNING
 * every kernel below is a no-op, so replaying past the stop point changes nothing. */
#define SWM_CMAES_MIN_POPSIZE 2
typedef enum {
  SWM_CMAES_RUNNING = 0,
  SWM_CMAES_STOP_MAXITER = 1,
  SWM_CMAES_STOP_TOLFUN = 2,
  SWM_CMAES_STOP_TOLX = 3,
  SWM_CMAES_STOP_CONDITIONCOV = 4
} swm_cmaes_status;
SWM_API int64_t swm_cmaes_state_doubles(int d, int lambda); /* 0 for d or lambda out of range */
/* mean = x0 (host [d]), sigma = sigma0, C = B = I, paths 0, generation 0; max_generations <= 0 picks
 * 100 + 150 (d+3)^2 / sqrt(lambda) (the cma package's default) */
SWM_API int swm_cmaes_init(double* state, int d, int lambda, const double* x0, double sigma0, double tolfun,
                           double tolx, int64_t max_generations, void* stream);
/* candidates[lambda, d] (and z in the state) of the current generation */
SWM_API int swm_cmaes_sample(double* state, int d, int lambda, uint64_t seed, double* candidates, void* stream);
/* one update from the candidates of swm_cmaes_sample and their fitness[lambda]; advances the generation */
SWM_API int swm_cmaes_update(double* state, int d, int lambda, const double* candidates, const double* fitness,
                             void* stream);
/* sample + prediction-error objective (data->d == d) + update: one generation, no host round trip */
SWM_API int swm_cmaes_generation(double* state, int d, int lambda, uint64_t seed, const swm_params_t* base,
                                 const swm_estimate_data_t* data, double* candidates, double* fitness,
                                 void* stream);

/* FP64 pipe probe: every thread runs `iters` x 8 independent DFMA chains; returns through
 * *flops_out (host) the number of floating-point operations executed (2 per DFMA).  Used by
 * bench.py to measure the FP64 roofline denominator on the box (MEASURED_PEAKS.json has none). */
SWM_API int swm_fp64_probe(int blocks, int threads, int iters, double* sink, double* flops_out,
                   void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SWIMMER_ARS_H */
