/* minppo_b200 -- C ABI of the B200-native PPO learner.
 *
 * Drop-in boundary for the learner hot path of kscalelabs/minppo:
 *   /root/reference/minppo/train.py:181-281  (GAE -> E epochs x M minibatches of
 *   shuffle/gather, ActorCritic forward/backward + PPO loss, global-norm clip + Adam).
 *
 * The reference has no FFI for this path -- it is a span of traced Python inside one
 * jax.jit (SURVEY.md section 8b).  These entry points are what an XLA-FFI custom call
 * (jax.ffi) or any other host binds: plain device pointers, explicit sizes, scalar
 * hyper-parameters and a cudaStream_t (passed as void*).  No torch / JAX types.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - the caller owns every buffer and the stream; the library owns only the context;
 *   - everything is enqueued on `stream`; no call synchronises the device or the host;
 *   - return value: 0 on success, negative MINPPO_ERR_* otherwise; minppo_last_error()
 *     returns a thread-local message.  Nothing throws, nothing exits.
 *   - trajectories are TIME-MAJOR [T, N, ...] exactly as jax.lax.scan stacks `Memory`
 *     (train.py:26-33, 179); flat transition index = t * N + n (train.py:260).
 */
#ifndef MINPPO_B200_H_
#define MINPPO_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MINPPO_OK 0
#define MINPPO_ERR_ARG (-1)        /* bad argument / shape / alignment            */
#define MINPPO_ERR_CUDA (-2)       /* a CUDA runtime or driver call failed        */
#define MINPPO_ERR_WORKSPACE (-3)  /* workspace too small                         */
#define MINPPO_ERR_UNSUPPORTED (-4)/* shape outside what the kernels implement    */
#define MINPPO_ERR_NCCL (-5)       /* a NCCL call failed                          */
#define MINPPO_ERR_BARRIER (-6)    /* device-side grid barrier timed out          */
#define MINPPO_ERR_NONFINITE (-7)  /* loss or gradient norm is not finite         */

#define MINPPO_PRNG_LEGACY 0        /* jax_threefry_partitionable = False (JAX < 0.5 default) */
#define MINPPO_PRNG_PARTITIONABLE 1 /* jax_threefry_partitionable = True  (JAX >= 0.5 default) */

#define MINPPO_MAX_LEAVES 32
#define MINPPO_MAX_RANKS 8

typedef struct minppo_ctx minppo_ctx;

/* Hyper-parameters: the rl.* / training.* / opt.* / model.* keys the learner reads
 * (/root/reference/minppo/config.py:50-84), plus the shapes the reference takes from
 * the environment (env.py:99, 245-261) and the sharding of this process. */
typedef struct minppo_config {
  int32_t num_envs;          /* training.num_envs   -- GLOBAL number of envs N        */
  int32_t num_steps;         /* training.num_steps == rl.num_env_steps -- T           */
  int32_t num_minibatches;   /* training.num_minibatches -- M                         */
  int32_t update_epochs;     /* training.update_epochs -- E                           */
  int64_t total_timesteps;   /* training.total_timesteps (LR schedule, train.py:93)   */
  int32_t anneal_lr;         /* training.anneal_lr                                    */
  int32_t hidden_size;       /* model.hidden_size  (multiple of 64, <= 512; > 256: num_layers <= 2) */
  int32_t num_layers;        /* model.num_layers   (>= 1)                             */
  int32_t use_tanh;          /* model.use_tanh     (actor only; critic is relu, train.py:82) */
  int32_t obs_dim;           /* D                                                     */
  int32_t act_dim;           /* A (<= 64; > 32: layer-wise kernels)                   */
  int32_t prng_mode;         /* MINPPO_PRNG_*                                         */
  int32_t world_size;        /* G: env-sharded ranks (1 = single GPU)                 */
  int32_t rank;              /* this rank owns envs [rank*N/G, (rank+1)*N/G)          */
  int32_t fast_tanh;         /* 1: tanh.approx.f32 (MUFU) in the GEMM epilogue        */
  int32_t dw_splits;         /* split-K factor of the weight-gradient GEMMs (0 = auto) */
  int32_t disable_fused;     /* 1: always use the layer-wise kernels (default 0: fused step kernel when L == 2,
                                hidden_size <= 256 and act_dim <= 32; wider layers or heads always run layer-wise) */
  double training_lr;        /* training.lr  (annealed path, train.py:101)            */
  double opt_lr;             /* opt.lr       (constant path, train.py:123)            */
  double max_grad_norm;      /* opt.max_grad_norm                                     */
  double gamma;              /* rl.gamma                                              */
  double gae_lambda;         /* rl.gae_lambda                                         */
  double clip_eps;           /* rl.clip_eps                                           */
  double ent_coef;           /* rl.ent_coef                                           */
  double vf_coef;            /* rl.vf_coef                                            */
  double adam_b1, adam_b2, adam_eps, adam_eps_root; /* optax.adam(eps=1e-5) train.py:118 */
} minppo_config;

/* Thread-local message for the last failing call on this thread. */
const char* minppo_last_error(void);
int minppo_version(void);

/* ---- (1) GAE: replaces _calculate_gae, train.py:185-207 ------------------------------
 * reward, value: f32 [T, N]; done: u8 [T, N] (the reference's bool); last_val: f32 [N];
 * adv_out, tgt_out: f32 [T, N].  17 algorithmic bytes per transition. */
int minppo_gae(const float* reward, const float* value, const uint8_t* done, const float* last_val,
               float* adv_out, float* tgt_out, int32_t T, int64_t N, double gamma, double gae_lambda,
               void* stream);
/* Same, forcing the number of T-segments (1 = the reference's sequential scan order). */
int minppo_gae_chunked(const float* reward, const float* value, const uint8_t* done, const float* last_val,
                       float* adv_out, float* tgt_out, int32_t T, int64_t N, double gamma, double gae_lambda,
                       int32_t chunks, void* stream);

/* ---- (2) minibatch permutations: replaces jax.random.split + jax.random.permutation,
 * train.py:252, 258, for all `epochs` epochs of one update at once.
 * key_in: u32[2]; key_out: u32[2] (rng after `epochs` splits; may be NULL);
 * perm_out: i32 [epochs, B]: row e is the permutation epoch e uses; minibatch k of epoch e
 * is perm_out[e, k*mb : (k+1)*mb] (train.py:262-265). */
size_t minppo_permutation_workspace_size(int32_t epochs, int64_t B);
int minppo_permutation(const uint32_t* key_in, uint32_t* key_out, int32_t prng_mode, int32_t epochs, int64_t B,
                       int32_t* perm_out, void* workspace, size_t workspace_bytes, void* stream);

/* ---- parameter arena -----------------------------------------------------------------
 * params / mu / nu are contiguous f32 arenas; leaves in JAX's sorted flatten order of the
 * checkpoint tree (train.py:86-89; SURVEY.md section 5):
 *   MLP_0/Dense_0/bias, MLP_0/Dense_0/kernel, ..., MLP_1/..., log_std.  kernel = [in, out].
 * Writes nleaves, offsets[i], rows[i], cols[i] (bias / log_std: rows = 1).  Returns P. */
int64_t minppo_param_layout(const minppo_config* cfg, int32_t* nleaves, int64_t* offsets, int64_t* rows,
                            int64_t* cols);

/* ---- kernel path ---------------------------------------------------------------------------
 * The kernels minppo_ctx_create and minppo_update pick for a config on a device with `sm_count` SMs (minppo_ctx_create
 * uses the device's).  Host only, no CUDA call: it answers without a GPU.  A config the context refuses is refused here
 * with the same code and message.  Named like `struct stat` / stat(): declare the result as `struct minppo_plan`.
 *   num_params     P
 *   fused          fused step kernel (num_layers == 2, hidden_size <= 256, act_dim <= 32, not disabled)
 *   ap, head_amax  head width of the fused step kernel (16 or 32) and template of the layer-wise heads (8, 16, 32, 64)
 *   hsplit         column groups of the forward, dX and policy GEMMs (2: hidden_size > 256)
 *   dw_nsplit, S   column groups per (net, layer) and split-K factor of the weight-gradient GEMM
 *   dw_gemm_ctas   CTAs of that GEMM; two_launch = dw_gemm_ctas > sm_count: it runs as a launch of its own
 *   maxu           4-element units per thread of the optimizer's register-resident path (1, 2 or 4); dwopt_fast: that
 *                  path holds the weight-gradient GEMM's leaves
 *   padded         row lists sized for a worst-case row count (world_size > 1), row counts read on the device
 *   row_cap        rows per minibatch row list (a multiple of 128)
 *   peer_exchange  world_size > 1: the peer-memory gradient exchange may replace NCCL once peers are set */
struct minppo_plan {
  int64_t num_params;
  int32_t fused, ap, head_amax, hsplit, dw_nsplit, S, dw_gemm_ctas, two_launch;
  int32_t maxu, dwopt_fast, padded, row_cap, peer_exchange;
};
int minppo_plan(const minppo_config* cfg, int32_t sm_count, struct minppo_plan* out);

/* ---- (3) context -----------------------------------------------------------------------
 * Owns workspace, TMA descriptors, weight images and (world_size > 1) a NCCL communicator
 * built from `nccl_unique_id_host` (128 bytes from minppo_nccl_unique_id on rank 0, broadcast
 * by the caller).  One context per (device, shape); calls on one context are not re-entrant. */
int minppo_nccl_unique_id(void* id128_host);
int minppo_ctx_create(const minppo_config* cfg, const void* nccl_unique_id_host, minppo_ctx** out);
int minppo_ctx_destroy(minppo_ctx* ctx);

/* ---- gradient exchange over NVLink peer memory (world_size > 1, optional) ----------------------
 * Default for sharded ranks is ncclAllReduce + a separate optimizer launch per minibatch.  With peer buffers set, the
 * all-reduce is fused INTO the weight-gradient/optimizer kernel: every rank stores its gradient sums straight into the
 * peers' staging buffers over NVLink and polls its own (the data is its own arrival flag: a sentinel value marks
 * "not yet written"), sums the contributions in rank order and applies the identical clip + Adam -- no NCCL call, no
 * extra launch on the per-minibatch path, parameters bit-identical on all ranks.  One-shot (every rank to every rank)
 * below 4 ranks, two-phase (reduce at one owner per unit, result pushed back) from 4 ranks on.
 * Every rank exports one CUDA-IPC handle (64 bytes); the host framework all-gathers them (rank order) and hands the
 * table back.  All ranks must then issue the same sequence of minppo_update calls. */
int minppo_ctx_ipc_handle(minppo_ctx* ctx, void* handle64_host);
int minppo_ctx_set_peers(minppo_ctx* ctx, const void* handles_host /* [world_size][64] */);

/* ---- (4) one learner update: replaces train.py:185-281 ---------------------------------
 * In place: params, mu, nu (f32 [P]), count (i32 [1], Adam step count == TrainState.step).
 * Read only: obs f32 [T, Nl, D], action f32 [T, Nl, A], value / reward / log_prob f32 [T, Nl],
 * done u8 [T, Nl], last_val f32 [Nl]  -- Nl = N / world_size, this rank's env shard.
 * key_in u32[2] -> key_out u32[2] (RunnerState.rng, train.py:280).
 * losses_out: f32 [E, M, 4] = (total, value_loss, actor_loss, entropy) per minibatch, may be NULL.
 * use_graph != 0: the step sequence is captured once into a CUDA graph per POINTER SET and replayed (the 4 most recently
 * used pointer sets are kept: present the same buffers every call -- ping-pong pairs are fine -- or every call re-captures);
 * use_graph == 0: kernels are enqueued directly (also valid inside a caller's capture: tests/test_gpu_capture.py).
 * A device-side failure of the update (a row list that overflowed its capacity on an env-sharded rank, a grid-barrier or
 * peer-exchange timeout) turns every value written to losses_out by the remaining steps into NaN; minppo_ctx_check names it. */
int minppo_update(minppo_ctx* ctx, float* params, float* mu, float* nu, int32_t* count, const float* obs,
                  const float* action, const float* value, const float* reward, const float* log_prob,
                  const uint8_t* done, const float* last_val, const uint32_t* key_in, uint32_t* key_out,
                  float* losses_out, int32_t use_graph, void* stream);

/* minppo_update plus per-minibatch PPO diagnostics (minppo_update is this call with stats_out == NULL).
 * stats_out: f32 [E, M, 4], may be NULL.  Row s = e * M + k describes minibatch step s over the rows of the GLOBAL
 * minibatch (all ranks, live rows only), evaluated in the forward pass of that step's loss, i.e. with the parameters
 * BEFORE that step's Adam update; r = exp(logp_new - logp_old) is the loss's probability ratio:
 *   [0] approx_kl            mean(expm1(log r) - log r)        (the "(r - 1) - log r" estimator)
 *   [1] clip_fraction        mean(|r - 1| > clip_eps)
 *   [2] value_clip_fraction  mean(|v - v_old| > clip_eps)
 *   [3] grad_norm            global gradient norm before clipping (clip_by_global_norm), bit-identical to
 *                            minppo_ctx_read buffer 4
 * The sums are always computed; stats_out only selects whether they are written.  Everything else the update computes
 * is bit-identical with and without stats_out.  stats_out is part of the graph cache's pointer set.  A device-side
 * failure turns all four columns of the remaining steps into NaN, as it does the losses. */
int minppo_update_with_stats(minppo_ctx* ctx, float* params, float* mu, float* nu, int32_t* count, const float* obs,
                             const float* action, const float* value, const float* reward, const float* log_prob,
                             const uint8_t* done, const float* last_val, const uint32_t* key_in, uint32_t* key_out,
                             float* losses_out, float* stats_out, int32_t use_graph, void* stream);

/* ---- (5) policy / value inference for the rollout: replaces train.py:157-160 and 182-183 ------------
 * One env step's network evaluation on this rank's Nl = N / world_size envs, forward only, on the same bf16 weight
 * images and with the same rounding points as the learner's forward pass:
 *   pi, value = network.apply(params, last_obs); rng, action_rng = split(rng);
 *   action = pi.sample(seed=action_rng); log_prob = pi.log_prob(action)
 * obs f32 [Nl, D] (read only).  Outputs (each may be NULL): action f32 [Nl, A], log_prob f32 [Nl], value f32 [Nl],
 * mean f32 [Nl, A] (the distribution's mode, for evaluation).  key_in u32[2] -> key_out u32[2] = rng after the
 * split (key_out may be NULL, must not alias key_in); key_in == NULL: no sampling, action = mean, log_prob of it.
 * action == log_prob == mean == NULL: critic only -- the bootstrap value `_, last_val = network.apply(params,
 * last_obs)` (train.py:182-183).
 * The normal draw is the GLOBAL jax.random.normal(action_rng, (N, A)): an env-sharded rank produces its rows of it.
 * flags: MINPPO_POLICY_WEIGHTS_CURRENT = the context's weight images already match `params` (true right after
 * minppo_update or a previous policy step with the same, unmodified arena) -> skips the image refresh launch.
 * Enqueues on `stream`, never synchronises; valid inside a caller's graph capture.  Two-hidden-layer nets: ONE launch
 * (observation conversion, both hidden layers, heads, sampler: policy_fused.cuh) after the optional image refresh. */
#define MINPPO_POLICY_WEIGHTS_CURRENT 1
int minppo_policy_step(minppo_ctx* ctx, const float* params, const float* obs, const uint32_t* key_in,
                       uint32_t* key_out, float* action, float* log_prob, float* value, float* mean,
                       int32_t flags, void* stream);

/* Device-side error flag of the last update (0 = ok); synchronises `stream`. */
int minppo_ctx_check(minppo_ctx* ctx, void* stream);

/* Number of kernel launches one update enqueues (for bench.py's gpu_launches). */
int64_t minppo_update_launch_count(const minppo_ctx* ctx);

/* ---- per-kernel-class timing (bench.py's roofline) -----------------------------------------
 * With profiling enabled, an update enqueued with use_graph == 0 records a CUDA-event pair on
 * `stream` around every kernel class; minppo_ctx_profile_read synchronises and returns, per
 * class, the summed milliseconds and the number of timed scopes of the LAST update.
 * Classes: 0 gae, 1 permutation sort, 2 row lists + advantage stats, 3 observation image,
 * 4 weight images, 5 forward GEMMs, 6 heads + loss, 7 backward (dX) GEMMs, 8 weight-gradient
 * GEMMs, 9 optimizer, 10 all-reduce. */
#define MINPPO_PROFILE_CLASSES 11
int minppo_ctx_profile(minppo_ctx* ctx, int32_t enable);
int minppo_ctx_profile_read(minppo_ctx* ctx, float* ms_per_class_host, int32_t* scopes_per_class_host,
                            int32_t nclasses);

/* ---- introspection for tests: copy an internal buffer (device -> device, on `stream`) ----
 * what: 0 advantages f32 [T,Nl]; 1 targets f32 [T,Nl]; 2 perms i32 [E,B]; 3 last gradient f32 [P+4];
 *       4 grad norms f32 [E*M]; 5 row counts i32 [E*M]; 6 adv stats f32 [E*M,2] */
int minppo_ctx_read(minppo_ctx* ctx, int32_t what, void* dst, size_t bytes, void* stream);

/* ---- unit-test hook for the tcgen05 GEMM engine ----------------------------------------
 * C[M,N] (f32) = A * B with bf16 operands, through the same kernel the learner uses.
 *  mode 0: A [M,K] row-major, B [N,K] row-major            (K-major / K-major, TMA)
 *  mode 1: A = At^T with At [K,M], B = Bt^T with Bt [K,N]  (MN-major / MN-major, TMA)
 *  mode 2: A rows gathered: A[m,:] = img[rowidx[m],:K], B [N,K]          (gather K-major)
 *  mode 3: A[m,k] = img[rowidx[k], m], B = Bt^T with Bt [K,N]            (gather MN-major)
 * M multiple of 128, K multiple of 64, N multiple of 64 and <= 256; splits >= 1 partial sums
 * are written to C as [splits, M, N]. */
int minppo_debug_gemm(int32_t mode, const void* a_bf16, const void* b_bf16, const int32_t* rowidx, float* c,
                      int32_t M, int32_t N, int32_t K, int32_t lda, int32_t splits, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MINPPO_B200_H_ */
