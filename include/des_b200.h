/*
 * des_b200.h — C ABI of the B200-native Evolution-Strategies hot path.
 *
 * Drop-in boundary for the per-generation hot path of ShangtongZhang/DistributedES
 * (reference @ c4de970; the reference is pure Python and has no FFI of its own — each entry point
 * below names the reference lines it replaces; INTEGRATION.md shows the ctypes stub a maintainer
 * would add to natural_es.py / cma_es.py).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; no torch / C++ types cross this boundary.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 *   - Pointers named *_dev are device pointers on the current CUDA device, caller-owned,
 *     contiguous, naturally aligned; nothing is retained past the return of a call.
 *   - Device-pointer entry points only enqueue work: no host synchronisation, no allocation —
 *     they are CUDA-graph capturable.  Scratch memory is an explicit caller-owned workspace.
 *   - Every function returns DES_OK (0) or a negative des_status; des_last_error() returns a
 *     thread-local message.  There is no CPU fallback anywhere: without a CUDA device the calls fail.
 *   - Flat parameter layout (model.py:8-25 with StandardFCNet model.py:30-32), P floats:
 *       [fc1.weight (H x d0 row-major) | fc1.bias (H) | fc2.weight (H x H) | fc2.bias (H)
 *        | fc3.weight (A x H) | fc3.bias (A)]
 *   - Noise contract: eps[member][j] is a pure function of (seed, generation, GLOBAL member index,
 *     j): Philox4x32-7 (Random123 constants, 7 rounds), counter = (j/4, member, generation, stream_tag), key = (seed_lo, seed_hi);
 *     words (x0,x1) -> Box-Muller -> (eps[4q], eps[4q+1]); (x2,x3) -> (eps[4q+2], eps[4q+3]).
 *     Box-Muller on the LOW 23 bits k of each word, f = 1 + k*2^-23:  u1 = f1 - (1 - 2^-24) in (0,1),
 *     ang = fl32(f2*fl32(2 pi) - fl32(3 pi - pi 2^-23)) ~ 2 pi u2 - pi,
 *     z_first = -sqrt(-2 ln u1) cos(ang), z_second = -sqrt(-2 ln u1) sin(ang).
 *     (oracle/nes_oracle.py restates it bit-exactly for the uint32 words.)  It replaces
 *     np.random.randn at natural_es.py:29; eps never crosses a process/GPU boundary.
 */
#ifndef DES_B200_H
#define DES_B200_H

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define DES_API __attribute__((visibility("default")))
#else
#define DES_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef enum des_status {
    DES_OK = 0,
    DES_ERR_INVALID_ARGUMENT = -1,   /* bad shape / null pointer / misaligned / unsupported size */
    DES_ERR_CUDA = -2,               /* a CUDA runtime call failed (message has the CUDA error)   */
    DES_ERR_NO_DEVICE = -3,          /* no usable CUDA device — there is no CPU fallback           */
    DES_ERR_WORKSPACE = -4,          /* workspace too small (see *_workspace_bytes)               */
    DES_ERR_UNSUPPORTED = -5         /* valid request this build/device cannot run                */
} des_status;

/* Policy-forward arithmetic (StandardFCNet.forward model.py:34-39). */
typedef enum des_precision {
    DES_FWD_FP32 = 0,     /* CUDA-core FFMA, fp32 everywhere: the parity-grade path              */
    DES_FWD_F16 = 1,      /* tcgen05 kind::f16: operands rounded to fp16 (11 significant bits,     */
                          /* like TF32), fp32 accumulate in TMEM, MUFU tanh                        */
    DES_FWD_F16X3 = 2     /* tcgen05 kind::f16 with hi/lo split operands (3 MMAs), ~fp32 accuracy */
} des_precision;

/* MLP shape (config.py:10-13: state_dim, action_dim, hidden_size) + the tape length. */
typedef struct des_dims {
    int32_t state_dim;    /* d0 */
    int32_t hidden;       /* H  */
    int32_t action_dim;   /* A  */
    int32_t tape_len;     /* T: observations evaluated per member per generation */
} des_dims;

/* Adam hyper-parameters (utils.py:151-154) + the NES step (natural_es.py:92-96). */
typedef struct des_opt {
    double sigma;          /* config.sigma          natural_es.py:30,92 */
    double learning_rate;  /* config.learning_rate  natural_es.py:96    */
    double weight_decay;   /* config.weight_decay   natural_es.py:93    */
    double beta1, beta2, epsilon;   /* utils.py:151 */
} des_opt;

/* Per-run counters living in DEVICE memory so a captured CUDA graph can be replayed:
 * generation (RNG counter word), Adam step count and the running beta^t products
 * (utils.py:160-161 keeps them as repeated products, not pow()). */
typedef struct des_state {
    uint64_t generation;
    uint64_t adam_t;
    double beta1_t;
    double beta2_t;
} des_state;

DES_API const char *des_last_error(void);
DES_API const char *des_version(void);
/* Number of CUDA devices usable by this build (0 if none); never falls back to CPU. */
DES_API int des_device_count(void);

/* P = d0*H + H + H*H + H + H*A + A  (model.py:30-32).  Negative on invalid dims. */
DES_API int64_t des_param_count(int32_t state_dim, int32_t hidden, int32_t action_dim);

/* ---- noise ------------------------------------------------------------------------------- */

/* eps_out_dev[n_members][P] fp32 = the noise rows of members [member_offset, member_offset+n).
 * Debug / parity op (the hot path never materialises eps).  Replaces natural_es.py:29. */
DES_API int des_noise_fill(float *eps_out_dev, int64_t n_members, int64_t P, uint64_t seed,
                   uint64_t generation, int64_t member_offset, uint32_t stream_tag, void *stream);

/* theta_out_dev[n_members][P] = fp32(theta + sigma*eps_i)  (natural_es.py:28-30).  Debug / parity op. */
DES_API int des_nes_perturb(float *theta_out_dev, const float *theta_dev, int64_t n_members, int64_t P,
                    double sigma, uint64_t seed, uint64_t generation, int64_t member_offset,
                    void *stream);

/* ---- observation normaliser (StaticNormalizer / SharedStats, utils.py:37-106) -------------------------- */

/* stats_dev: fp32 [m (d0) | v (d0) | n (1)], zero-initialised = "no statistics" (utils.py:61-63).
 * des_obs_stats_merge: Chan-merge (utils.py:85-96) the statistics of the tape obs_dev[T][d0], fed n_feed times
 * (n_feed = members * T * repetitions: what the workers' online stats hold after one generation on the tape env),
 * into stats_dev.  des_obs_normalize: obs_out = (obs - m)/sqrt(v + 1e-6), or obs unchanged while n == 0
 * (utils.py:48-51).  obs_out_dev may alias obs_dev. */
DES_API int des_obs_stats_merge(float *stats_dev, const float *obs_dev, int32_t tape_len, int32_t state_dim,
                        double n_feed, void *stream);
DES_API int des_obs_normalize(float *obs_out_dev, const float *obs_dev, const float *stats_dev, int32_t tape_len,
                      int32_t state_dim, void *stream);

/* ---- closed-loop rollouts: environment stepped on the device (SURVEY 8f row 3) ------------------------------- */

#define DES_ENV_PENDULUM 0 /* 'Pendulum-v0' of PendulumConfig config.py:26-31: state_dim 3, action_dim 1, clip 2, 200 steps */

/* fitness_out_dev[i] (i < n_local) = mean over `repetitions` episodes of sum_t reward_t for the policy
 * theta + sigma*eps_m, m = member_offset + i, each episode stepped in closed loop for dims.tape_len steps:
 * Worker.run natural_es.py:27-32 -> Evaluator.eval utils.py:116-124 -> single_run utils.py:126-139 (normalise the
 * observation with obs_stats_dev [m|v|n] or pass it through while n == 0 / NULL, forward, + action_noise_std * N(0,1),
 * clip, env.step).  Episode (m, r) of generation g resets from counter stream 2: Philox(r, m, g, 2) (see
 * oracle/pendulum_oracle.py); noiseless != 0 evaluates theta itself over `repetitions` test episodes
 * (test() natural_es.py:101-110; n_local must be 1, reset member 0x40000000).
 * episode_returns_out_dev (optional, [n_local][repetitions]) receives the individual episode returns.
 * obs_totals_out_dev (optional, fp64 [2*state_dim + 1]) receives sum, sum of squares and count of the RAW observations
 * fed to the normaliser by these members — what the workers' online stats hold (utils.py:68-73) — to be summed over
 * ranks and merged with des_obs_stats_merge_totals; it needs workspace_dev of n_local * (2*state_dim+1) * 8 bytes.
 * hidden must be a multiple of 32 (<= 128), repetitions <= 10.  Arithmetic: policy in fp32 (FFMA, accurate tanh),
 * dynamics in fp64 like gym's float64 state. */
DES_API int des_rollout_eval(float *fitness_out_dev, float *episode_returns_out_dev, double *obs_totals_out_dev,
                             const float *theta_dev, const float *obs_stats_dev, int env, des_dims dims, int32_t repetitions, double sigma,
                             double clip, double action_noise_std, uint64_t seed, uint64_t generation,
                             const des_state *state_dev, int64_t member_offset, int64_t n_local, int noiseless,
                             void *workspace_dev, size_t workspace_bytes, void *stream);

/* Chan merge (utils.py:85-96) of a batch given by obs_totals_dev = [sum (d0) | sum of squares (d0) | count] into
 * stats_dev [m|v|n]  (natural_es.py:85-89 after the cross-rank sum of the totals). */
DES_API int des_obs_stats_merge_totals(float *stats_dev, const double *obs_totals_dev, int32_t state_dim, void *stream);

/* ---- fused sample + forward + fitness ------------------------------------------------------ */

/* fitness_out_dev[i] (i < n_local) = sum_t -|| clip(pi_{theta+sigma*eps_m}(obs_t), -clip, clip) - target_t ||^2
 * for global member m = member_offset + i.  Replaces, per member, Worker.run natural_es.py:27-32 ->
 * Evaluator.eval utils.py:116-124 -> single_run utils.py:126-139 -> StandardFCNet.forward
 * model.py:34-39 over the synthetic tape env (obs_dev [T][d0], target_dev [T][A], both fp32).
 * `state_dev` may be NULL (then `generation` is used); if non-NULL, state_dev->generation wins
 * (graph replay).  precision: see des_precision; DES_FWD_F16 / F16X3 need H in {64,128,256},
 * d0 <= 32, A <= 8, T a multiple of 128 and |values| < 65504 — otherwise DES_ERR_UNSUPPORTED (never a silent fallback).
 * workspace (optional, may be NULL): des_nes_eval_workspace_bytes() bytes, 16-byte aligned; shapes whose tape does not
 * fit the tensor memory in one pass use it to keep a member's generated weight tiles between passes instead of
 * regenerating them (same results either way). */
DES_API size_t des_nes_eval_workspace_bytes(des_dims dims, int precision);
DES_API int des_nes_eval(float *fitness_out_dev, const float *theta_dev, const float *obs_dev,
                 const float *target_dev, des_dims dims, double sigma, double clip, uint64_t seed,
                 uint64_t generation, const des_state *state_dev, int64_t member_offset,
                 int64_t n_local, int precision, void *workspace_dev, size_t workspace_bytes,
                 void *stream);

/* fitness_out_dev[i] = the same tape fitness for EXPLICIT weight vectors solutions_dev[n_solutions][P] (no noise):
 * the evaluation CMA-ES needs, where the master ships sampled solutions to the workers (cma_es.py:62-64,
 * Worker.run cma_es.py:22-29 -> Evaluator.eval utils.py:116-124).  fp32 CUDA-core path, any shape. */
DES_API int des_pop_eval(float *fitness_out_dev, const float *solutions_dev, const float *obs_dev,
                 const float *target_dev, des_dims dims, double clip, int64_t n_solutions, void *stream);

/* ---- centered-rank shaping ------------------------------------------------------------------ */

/* For the n_local members starting at member_offset of the GLOBAL fitness vector fitness_all_dev[N]:
 * rank_out_dev[i] = #{j : f_j < f_i} + #{j < i : f_j == f_i}  (ascending, ties by index; -0 == +0,
 * NaN ranks last) and shaped_out_dev[i] = fp32(rank/(N-1) - 0.5).  Replaces fitness_shift
 * utils.py:142-148 (whose argsort is unstable on ties; identical on tie-free input).
 * rank_out_dev may be NULL.  N >= 2.  workspace: at least des_rank_workspace_bytes(n_local); with
 * des_rank_workspace_bytes_n(N, n_local) bytes, populations above 2048 use the bucketed (sample-sort style)
 * path whose cost is ~N*N/1024 instead of n_local*N compares.  Results are identical either way. */
DES_API size_t des_rank_workspace_bytes(int64_t n_local);
DES_API size_t des_rank_workspace_bytes_n(int64_t N, int64_t n_local);
DES_API int des_centered_rank(float *shaped_out_dev, int32_t *rank_out_dev, const float *fitness_all_dev,
                      int64_t N, int64_t member_offset, int64_t n_local, void *workspace_dev,
                      size_t workspace_bytes, void *stream);

/* ---- fitness x noise reduction -------------------------------------------------------------- */

/* partial_out_dev[j] (j < P) = sum_{i < n_local} shaped_local_dev[i] * eps[member_offset+i][j]
 * (eps regenerated, fp32 FFMA per chunk, fp64 across chunks, stored fp32).  This is the per-shard
 * term of natural_es.py:91 before the mean and the 1/sigma; shards are summed by ONE all-reduce.
 * workspace: des_grad_workspace_bytes(n_local, P). */
DES_API size_t des_grad_workspace_bytes(int64_t n_local, int64_t P);
DES_API int des_nes_grad_partial(float *partial_out_dev, const float *shaped_local_dev, int64_t n_local,
                         int64_t P, uint64_t seed, uint64_t generation, const des_state *state_dev,
                         int64_t member_offset, void *workspace_dev, size_t workspace_bytes,
                         void *stream);

/* ---- (1-wd) scale + Adam + step ------------------------------------------------------------- */

/* g = (partial_sum/N)/sigma; g -= wd*g (natural_es.py:92-93); Adam (utils.py:159-166, fp64 state
 * adam_m_dev/adam_v_dev[P]); update = lr * fp32(step); theta += update (natural_es.py:95-96).
 * update_out_dev (may be NULL) receives the 'parameter-update vector'; grad_out_dev (may be NULL)
 * receives g before weight decay as fp64.  Adam's t / beta^t come from state_dev (required) and are
 * NOT advanced here: call des_state_advance once per generation after this. */
DES_API int des_nes_apply(float *theta_dev, double *adam_m_dev, double *adam_v_dev, float *update_out_dev,
                  double *grad_out_dev, const float *partial_sum_dev, int64_t P, int64_t N,
                  des_opt opt, const des_state *state_dev, void *stream);

/* state <- {generation+1, adam_t+1, beta1_t*beta1, beta2_t*beta2}.  des_state_init writes
 * {generation, 0, 1.0, 1.0}. */
DES_API int des_state_init(des_state *state_dev, uint64_t generation, void *stream);
DES_API int des_state_advance(des_state *state_dev, double beta1, double beta2, void *stream);

/* ---- CMA-ES rank-mu covariance update (inside es.tell, cma_es.py:90) ------------------------- */

/* dC_out_dev[n][n] = sum_{i < lambda_local} w_dev[i] * y_i y_i^T with Y_dev[lambda_local][n]
 * row-major (y_i = (x_i - m_old)/sigma, already sorted/weighted by the caller).  Full symmetric
 * matrix is written.  fp32 FFMA with fp32 accumulation per k-panel. */
DES_API int des_cma_rank_mu(float *dC_out_dev, const float *Y_dev, const float *w_dev, int64_t lambda_local,
                    int64_t n, void *stream);

/* C <- decay*C + c1 * pc pc^T + cmu * dC   (decay = 1 - c1 - cmu*sum(w) [+ (1-hsig) term folded in by
 * the caller]).  pc_dev may be NULL (then no rank-one term).  In place on C_dev[n][n]. */
DES_API int des_cma_cov_apply(float *C_dev, const float *dC_dev, const float *pc_dev, int64_t n, double decay,
                      double c1, double cmu, void *stream);

/* The same two steps with the rank-mu partial kept as PACKED upper-triangular tiles — the payload to all-reduce across
 * ranks when lambda is sharded (half the bytes of the [n][n] matrix; SURVEY 8e).  Layout: tiles (bi <= bj) in row-major
 * order of (bi, bj), each [tile][tile] row-major with tile = 64 (n <= 2048) or 128; entries beyond n are zero.
 * des_cma_packed_elems(n) floats.  des_cma_cov_apply_packed mirrors the tiles while applying them (diagonal tiles take the
 * j >= i entry for both sides: C stays exactly symmetric). */
DES_API int64_t des_cma_packed_elems(int64_t n);
DES_API int des_cma_rank_mu_packed(float *tiles_out_dev, const float *Y_dev, const float *w_dev, int64_t lambda_local,
                                   int64_t n, void *stream);
DES_API int des_cma_cov_apply_packed(float *C_dev, const float *tiles_dev, const float *pc_dev, int64_t n, double decay,
                                     double c1, double cmu, void *stream);

/* The rank-mu term on the tensor cores (csrc/des_cma_tc.cu): dC = Zs^T Z with Z = diag(sqrt|w|) Y, each coordinate j of Z
 * scaled by a power of two 2^e_j (undone exactly on the output) so that its largest |entry| lies in [2^14, 2^15), then
 * split into fp16 hi + lo (three tcgen05 MMAs per k-step, fp32 accumulation, TMA-fed) — same result contract as
 * des_cma_rank_mu (packed == 0: full symmetric [n][n]) / des_cma_rank_mu_packed (packed != 0), within 1e-5 of the fp64
 * restatement in both norms and entry by entry within 1e-5 sqrt(A_ii A_jj), A = sum_k |w_k| y_k y_k^T, at any scale of
 * the coordinates.  An inf or NaN in coordinate j of Y reaches only row and column j.  Needs
 * des_cma_tc_workspace_bytes(n, lambda_local) bytes of workspace. */
DES_API size_t des_cma_tc_workspace_bytes(int64_t n, int64_t lambda_local);
DES_API int des_cma_rank_mu_tc(float *out_dev, const float *Y_dev, const float *w_dev, int64_t lambda_local, int64_t n,
                               int packed, void *workspace_dev, size_t workspace_bytes, void *stream);

/* ---- exchange steps of a sharded generation over peer memory (NVLink) ------------------------- */

/* One process per GPU on one node.  Replaces the reference's result pipe (natural_es.py:62-75: every worker ships
 * (epsilon, fitness, steps) to the master) for the two things a shard must exchange: its fitness values (ranks are
 * global, utils.py:142-148) and its partial sum_i s_i eps_i (natural_es.py:91).  Each rank owns one device block
 * [fitness_all[N] | slots[world][P]] exported with cudaIpc; the kernels store straight into the peers' blocks and
 * synchronise with epoch flags kept in device memory (CUDA-graph capturable, no host involvement).
 *   des_comm_create     allocates the local block on the current device; ipc_handle_out receives 64 bytes to hand to
 *                       every peer (any transport: torch.distributed all_gather, a file, MPI ...)
 *   des_comm_connect    all_handles = world x 64 bytes in rank order; maps the peers' blocks (enables P2P access)
 *   des_comm_fitness_all_dev   the local fitness_all[N]: des_nes_eval writes the shard here.  Peers store into it: a host
 *                       that reads it after a generation must take a stream-ordered copy right after the all-gather
 *                       (a peer that runs ahead may already be storing its next shard)
 *   des_comm_allgather_fitness stores the local shard [member_offset, +n_local) into every peer's fitness_all and
 *                       returns (on the stream) when every peer's shard has landed here: all ranks then hold the same N values
 *   des_comm_allreduce_partial  partial_sum_out[j] = sum over ranks r = 0..world-1, in that order, of rank r's
 *                       partial_dev[j]: bit-identical on every rank (fixed order), so theta needs no broadcast. */
typedef struct des_comm des_comm;
DES_API int des_comm_create(des_comm **out, int rank, int world, int64_t N, int64_t P, void *ipc_handle_out);
DES_API int des_comm_connect(des_comm *c, const void *all_handles);
DES_API void des_comm_destroy(des_comm *c);
DES_API float *des_comm_fitness_all_dev(des_comm *c);
DES_API int des_comm_allgather_fitness(des_comm *c, int64_t member_offset, int64_t n_local, void *stream);
DES_API int des_comm_allreduce_partial(des_comm *c, float *partial_sum_out_dev, const float *partial_dev, int64_t P,
                                       void *stream);

/* ---- host-buffer session: the call a reference-side binding makes --------------------------- */

typedef struct des_session des_session;   /* opaque; owns device buffers + a stream */

/* One NES population shard on `device`: members [member_offset, member_offset + n_local) of a
 * population of N.  theta0_host[P] initialises theta (config.initial_weight, natural_es.py:38). */
DES_API int des_session_create(des_session **out, int device, des_dims dims, int64_t N, int64_t member_offset,
                       int64_t n_local, des_opt opt, double clip, uint64_t seed, int precision,
                       const float *theta0_host);
DES_API void des_session_destroy(des_session *s);

/* One whole generation with HOST buffers (single-shard populations: n_local == N):
 * H2D obs/target(/theta if theta_in_host != NULL) -> eval -> rank -> grad -> apply -> D2H.
 * Outputs (any may be NULL): fitness_out_host[N] (the rewards list natural_es.py:64-73),
 * update_out_host[P], theta_out_host[P] (param after natural_es.py:96).  Synchronous. */
DES_API int des_session_generation_host(des_session *s, const float *obs_host, const float *target_host,
                                const float *theta_in_host, float *fitness_out_host,
                                float *update_out_host, float *theta_out_host);

/* Multi-shard use: the three phases around the two collectives (fitness gather, partial all-reduce)
 * operating on the session's device buffers; pointers are returned so the caller's communication
 * library (NCCL via torch.distributed) can reduce them in place. */
DES_API int des_session_upload_tape(des_session *s, const float *obs_host, const float *target_host);
DES_API int des_session_eval(des_session *s);                           /* fills fitness_all[offset:offset+n_local] */
DES_API int des_session_rank_and_grad(des_session *s);                  /* fitness_all -> partial[P]              */
DES_API int des_session_apply(des_session *s);                          /* partial (summed) -> theta, advance state */
DES_API float *des_session_fitness_all_dev(des_session *s);             /* [N], zero outside the local range      */
DES_API float *des_session_partial_dev(des_session *s);                 /* [P]                                   */
DES_API float *des_session_theta_dev(des_session *s);                   /* [P]                                   */
DES_API void *des_session_stream(des_session *s);                       /* cudaStream_t                           */
DES_API int des_session_sync(des_session *s);

#ifdef __cplusplus
}
#endif
#endif /* DES_B200_H */
