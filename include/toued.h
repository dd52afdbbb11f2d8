/* toued.h — C ABI of the B200-native TO-UED / GROOVE meta-training hot path.
 *
 * The reference (nmonette/TO-UED) is a pure-JAX program with no plugin / operator / FFI layer
 * (SURVEY.md §8b); the de-facto boundary is its Python call signatures.  Each entry point below is
 * the device-side operation one of those Python functions performs; the Python mirror in
 * to_ued_b200/ keeps the reference names and argument meaning and binds these with ctypes
 * (INTEGRATION.md shows the stub a reference maintainer would add).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in _host; plain C types only;
 *   - `stream` is the caller's cudaStream_t passed as void* (NULL = legacy default stream);
 *   - no entry point allocates device memory or synchronises; all work is enqueued on `stream`;
 *   - return 0 on success, non-zero on error; toued_last_error() gives the message (thread-local);
 *   - layouts: "agent" axis N, "worker" axis W, time axis L.  Trajectories are [N][L][W]
 *     (obs: [N][L+1][W]); tables are [N][D][8] floats (actor rows padded 5 -> 8, critic rows = 8).
 */
#ifndef TOUED_H
#define TOUED_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define TOUED_LEVEL_BYTES 192   /* sizeof(LevelRec), see to_ued_b200/csrc/common.cuh */

const char* toued_last_error(void);
int toued_version(void);

/* environments/rollout.py:45-102 RolloutWrapper.batch_rollout (+ :38-42 batch_reset when
 * reset_first != 0) fused with environments/gridworld/gridworld.py:72-211 and the tabular Actor
 * of models/agent.py:7-17.
 *   levels          LevelRec[N]           packed EnvParams (+ lifetime, buffer_id)
 *   keys            u32[N][2]             the per-agent key passed to batch_rollout
 *   actor           f32[N][D][8]          actor tables
 *   forced_actions  u8[N][L][W] or NULL   replay a given action stream instead of sampling
 *   state           i32[N][W] in/out      packed EnvState (pos | exists<<8 | time<<16); may be NULL
 *                                         when reset_first != 0 and the end state is not wanted
 *   obs             i32[N][L+1][W] out    packed observations (row | time<<16); NULL = no trajectory
 *   action,done     u8[N][L][W] out ; reward f32[N][L][W] out
 *   ep_return       f32[N][W] out or NULL first-episode return (rollout.py:68-69)               */
int toued_rollout(const void* levels, const uint32_t* keys, const float* actor,
                  const uint8_t* forced_actions, int32_t* state, int32_t* obs, uint8_t* action,
                  float* reward, uint8_t* done, float* ep_return, int n_agents, int n_workers,
                  int rollout_len, int obs_dim, int max_grid_size, int max_n_objs, int reset_first,
                  void* stream);

/* gymnax-style single transitions: environments/gridworld/gridworld.py:72-182 behind
 * gymnax==0.0.6 Environment.step (key split + auto-reset) / Environment.reset.
 *   keys u32[N][W][2] per-env step keys ; actions i32[N][W] ; state i32[N][W] in/out ;
 *   obs i32[N][W] out ; reward f32[N][W] out ; done u8[N][W] out                                */
int toued_env_step(const void* levels, const uint32_t* keys, const int32_t* actions, int32_t* state,
                   int32_t* obs, float* reward, uint8_t* done, int n_agents, int n_workers,
                   int max_grid_size, int max_n_objs, void* stream);
int toued_env_reset(const void* levels, int32_t* state, int32_t* obs, int n_agents, int n_workers,
                    int max_grid_size, void* stream);

/* ---- LPG-driven agent update (agents/lpg_agent.py:31-140, models/lpg.py:11-85) ----------------
 * LPG tensors are time-major [L][R] with R = N*W, row = n*W + w.
 * lpg_params: the flat parameter vector, layout in to_ued_b200/csrc/lpg_common.cuh.              */

/* Stable per-agent sort of the W*L tokens by observation row; sorted_tok u16[N][W*L] holds token
 * ids t*W+w.  Makes every later row scatter a deterministic segmented sum.                      */
int toued_sort_tokens(const int32_t* obs, uint16_t* sorted_tok, int n_agents, int n_workers,
                      int rollout_len, void* stream);

/* lpg_agent.py:46-58 + lpg.py:64-76: actor/critic forward on obs & next_obs, embedding MLP, LPG
 * input rows x f32[L][R][8] = [r, d, pi+1e-8, pyt, pyt1*(1-d), step|0, lifetime|0, 1].
 * ximg (or NULL): the same rows as a bf16 token-tile image [L*Rp/64][1][64][64] (zero-initialised by the
 * caller; columns 8..63 stay zero) for the tensor-core weight-gradient GEMM.                        */
int toued_lpg_prepare(const int32_t* obs, const uint8_t* action, const float* reward,
                      const uint8_t* done, const float* actor, const float* critic,
                      const float* lpg_params, const int32_t* step, const void* levels, float* x,
                      void* ximg, int n_agents, int n_workers, int rollout_len, int obs_dim,
                      int lifetime_conditioning, int lpg_stride, void* stream);

/* lpg.py:11-30,77-84: reverse GRU with done-reset, relu, heads.  Exact-fp32 SIMT path.
 *   h_out f32[L][R][256]; gates f32[4][L][R][256] (r, z, n, Whn h + bhn) or NULL;
 *   pi_hat f32[L][R]; y_hat f32[L][R][8]
 * lpg_stride (here and in toued_lpg_prepare): 0 = one shared parameter vector; otherwise agent n uses
 * lpg_params + n * lpg_stride (per-candidate parameters of the ES path, meta/train.py:167-176).    */
int toued_gru_forward(const float* x, const uint8_t* done, const float* lpg_params, float* h_out,
                      float* gates, float* pi_hat, float* y_hat, int n_agents, int n_workers,
                      int rollout_len, int lifetime_conditioning, int lpg_stride, void* stream);

/* lpg_agent.py:60-85,119-120 + optim.py:6-11: closed-form actor/critic gradients, clip-by-global-
 * norm SGD, lifetime mask, step += keep, entropies of the updated nets.
 *   scalars f32[N][8] = {|g_actor|, |g_critic|, keep, critic_loss, pi_l2, y_l2, policy_entropy,
 *                        critic_entropy}
 * toued_agent_update / toued_agent_backward need a temporary of 52 B x min(W*L, D) per agent for the duration of the
 * launch: run_scratch, f32[toued_agent_scratch_floats(N, W, L, D)], provided by the caller like every other buffer
 * (calls that may run concurrently on different streams need distinct scratch buffers).
 * tables_precopied != 0: actor_out / critic_out already hold a copy of actor_in / critic_in (made by the caller, e.g. on
 * a side stream next to the LPG forward); the kernel then writes the touched rows only.                  */
int toued_agent_scratch_floats(int n_agents, int n_workers, int rollout_len, int obs_dim);
int toued_agent_update(const int32_t* obs, const uint8_t* action, const uint16_t* sorted_tok,
                       const float* pi_hat, const float* y_hat, const float* actor_in,
                       const float* critic_in, float* actor_out, float* critic_out,
                       const void* levels, int32_t* step, float* scalars, int n_agents,
                       int n_workers, int rollout_len, int obs_dim, float lr_actor, float lr_critic,
                       float max_grad_norm, float agent_target_coeff, int tables_precopied, float* run_scratch,
                       void* stream);

/* ---- meta-gradient (meta/train.py:14-130): what the reference gets from jax.grad ---------------- */

/* meta/train.py:60-100 on the eval rollout: GAE with the (frozen, Q2) value critic, advantage
 * normalisation, LPG loss (outer_product_quirk != 0 reproduces Q16), and the adjoint of theta_K.
 *   value_table f32[N][D][value_stride] (column 0 used) ; lam, mu f32[N][D][8] out (mu zeroed)
 *   scalars f32[N][2] = {lpg_loss, value_loss} ; grad_scale = 1 / (global number of agents)        */
int toued_meta_loss(const int32_t* obs, const uint8_t* action, const float* reward,
                    const uint8_t* done, const uint16_t* sorted_tok, const float* value_table,
                    const float* actor, float* lam, float* mu, float* scalars, int n_agents,
                    int n_workers, int rollout_len, int obs_dim, int value_stride, float gamma,
                    float gae_lambda, float grad_scale, int outer_product_quirk, void* stream);

/* Adjoint of agent update k (lpg_agent.py:60-82 under jax.grad): entropy regularisers at the updated
 * tables, Hessian-vector products through grad/clip/SGD/lifetime-mask, cotangents of pi_hat, y_hat.
 * The four regulariser coefficients are passed already divided by K (mean over the K updates).
 *   update_scalars: the f32[N][8] written by toued_agent_update for this k ; lam, mu in/out        */
int toued_agent_backward(const int32_t* obs, const uint8_t* action, const uint16_t* sorted_tok,
                         const float* pi_hat, const float* y_hat, const float* actor_k,
                         const float* critic_k, const float* actor_k1, const float* critic_k1,
                         const float* update_scalars, float* lam, float* mu, float* d_pi_hat,
                         float* d_y_hat, int n_agents, int n_workers, int rollout_len, int obs_dim,
                         float lr_actor, float lr_critic, float max_grad_norm,
                         float agent_target_coeff, float policy_entropy_coeff,
                         float target_entropy_coeff, float policy_l2_coeff, float target_l2_coeff,
                         float grad_scale, float* run_scratch, void* stream);

/* whT f32[768][256] = transpose of the recurrent matrix Wh (once per meta-step).                 */
int toued_transpose_wh(const float* lpg_params, float* whT, void* stream);

/* BPTT through heads + reverse GRU (models/lpg.py:11-30,77-84).  gates f32[4][L][R][256] is
 * overwritten in place with (dar, daz, dan, dhn); dl f32[L][R][8] (head logit cotangents) and
 * dx f32[L][R][2] (d pyt, d pyt1) are outputs.                                                    */
int toued_gru_backward(const uint8_t* done, const float* lpg_params, const float* whT,
                       const float* h, float* gates, const float* y_hat, const float* d_pi_hat,
                       const float* d_y_hat, float* dl, float* dx, int n_agents, int n_workers,
                       int rollout_len, int lifetime_conditioning, void* stream);

/* Parameter gradients of one update as deterministic token-split partial sums in `workspace`
 * (toued_lpg_wgrad_workspace_floats() floats); accumulate != 0 adds to the partials of earlier
 * updates.  toued_reduce_partials then writes the flat gradient f32[P].                            */
int toued_lpg_wgrad_workspace_floats(void);
int toued_lpg_wgrad(const int32_t* obs, const uint8_t* done, const float* critic,
                    const float* lpg_params, const float* x, const float* h, const float* dgates,
                    const float* d_pi_hat, const float* dl, const float* dx, float* workspace,
                    int n_agents, int n_workers, int rollout_len, int obs_dim,
                    int lifetime_conditioning, int accumulate, void* stream);
int toued_lpg_wgrad_workspace_offset(int which);   /* float offset of the {0: Wh, 1: small, 2: embed} partial area */
int toued_lpg_wgrad_embed(const int32_t* obs, const uint8_t* done, const float* critic, const float* lpg_params,
                          const float* dx, float* workspace, const uint32_t* cotangent_max, int n_agents, int n_workers,
                          int rollout_len, int obs_dim, int lifetime_conditioning, int accumulate, void* stream);
/* wh_splits / sm_splits: how many dWh and small-parameter partial areas the producer filled --
 * toued_lpg_wgrad_splits(0) / (1) after toued_lpg_wgrad, toued_wgrad_tc_splits() / toued_wgrad_tc_small_splits() after
 * toued_lpg_wgrad_tc.  Areas beyond these counts are never read.                                         */
int toued_lpg_wgrad_splits(int which);
int toued_reduce_partials(const float* workspace, float* grad, int lifetime_conditioning, int wh_splits,
                          int sm_splits, void* stream);

/* models/optim.py:12-17: optax.scale_by_adam -> scale(lr) -> scale(-1); count is 1-based.          */
int toued_adam(float* params, const float* grad, float* mu, float* nu, int n, int count, float lr,
               float b1, float b2, float eps, void* stream);
/* the same step with the number of updates done so far in device memory (count_dev i32[1], incremented by the call):
 * no host-side state, so the call can be part of a captured CUDA graph (meta/graph.py).               */
int toued_adam_dev(float* params, const float* grad, float* mu, float* nu, int* count_dev, int n, float lr,
                   float b1, float b2, float eps, void* stream);
/* models/optim.py:6-11 (--lpg_opt SGD): optax.clip_by_global_norm(max_norm) -> scale(lr) -> scale(-1) on the flat LPG
 * parameter vector.  sqnorm_scratch f32[1] receives |grad|^2 (fixed-order reduction).                       */
int toued_sgd_clip(float* params, const float* grad, float* sqnorm_scratch, int n, float lr, float max_norm,
                   void* stream);

/* ---- A2C antagonist (agents/a2c.py:19-76), used by the algorithmic-regret level score ---------- */
/* critic_in/out: value tables f32[N][D][8] (column 0).  scalars f32[N][4] = {actor_loss, critic_loss,
 * |g_actor|, |g_critic|}.  outer_product_quirk != 0 reproduces Q16 (a2c.py:60 broadcast).           */
int toued_a2c_update(const int32_t* obs, const uint8_t* action, const float* reward, const uint8_t* done,
                     const uint16_t* sorted_tok, const float* actor_in, const float* critic_in,
                     float* actor_out, float* critic_out, const void* levels, int32_t* step,
                     float* scalars, int n_agents, int n_workers, int rollout_len, int obs_dim,
                     float lr_actor, float lr_critic, float max_grad_norm, float gamma, float gae_lambda,
                     float entropy_coeff, int outer_product_quirk, void* stream);

/* agents/a2c.py:79-125, the whole training loop in one call: num_updates x [toued_rollout -> toued_sort_tokens ->
 * toued_a2c_update], tables ping-ponging between (actor0, critic0) and (actor1, critic1) -- the result is in buffer
 * (num_updates & 1); keys u32[num_updates][N][2] (toued_key_chain); loss_sums f32[N][2] += {actor_loss, critic_loss}
 * of every update.  Keeps the 2500-update lifetime of the algorithmic-regret antagonist off the Python interpreter.  */
int toued_a2c_train(const void* levels, const uint32_t* keys, float* actor0, float* actor1, float* critic0,
                    float* critic1, int32_t* state, int32_t* obs, uint8_t* action, float* reward, uint8_t* done,
                    uint16_t* sorted_tok, int32_t* step, float* scalars, float* loss_sums, int num_updates,
                    int n_agents, int n_workers, int rollout_len, int obs_dim, int max_grid_size, int max_n_objs,
                    float lr_actor, float lr_critic, float max_grad_norm, float gamma, float gae_lambda,
                    float entropy_coeff, int outer_product_quirk, void* stream);

/* ---- OpenES ask / tell (evosax==0.1.4, meta/train.py:133-227) ----------------------------------- */
/* candidates f32[popsize][cand_stride] (first P of each row used; cand_stride a multiple of 4 floats so
 * every candidate is 16-byte aligned) in pair-adjacent order (2i = mean + sigma z_i, 2i+1 = mean - sigma z_i). */
int toued_es_ask(const uint32_t* key, const float* mean, float sigma, float* candidates, int popsize,
                 int n_params, int cand_stride, void* stream);
/* fitness f32[popsize] (higher is better; negated internally like evosax maximize=True); in-place Adam
 * step on `mean` with state m, v; gen_counter is 0-based.                                            */
int toued_es_tell(const float* candidates, const float* fitness, float* mean, float* m, float* v,
                  int popsize, int n_params, int cand_stride, float sigma, float lrate, float beta1,
                  float beta2, float eps, int gen_counter, float mean_decay, void* stream);

/* Multi-GPU ES (agents sharded over ranks, antithetic pairs kept on one rank; SURVEY.md section 8e, reference
 * meta/train.py:203-216): ask_shard writes the candidates of the pairs [pair_offset, pair_offset + n_pairs) of a global
 * population exactly as toued_es_ask would (candidates f32[2 * n_pairs][cand_stride]); grad_partial writes this rank's
 * sum_i noise_i * (-fitness_i) into grad_sum f32[n_params] (the caller all-reduces it over the ranks); es_adam is the
 * second half of toued_es_tell on the reduced sum.                                                        */
int toued_es_ask_shard(const uint32_t* key, const float* mean, float sigma, float* candidates, int popsize_global,
                       int n_params, int cand_stride, int pair_offset, int n_pairs, void* stream);
int toued_es_grad_partial(const float* candidates, const float* fitness, const float* mean, float* grad_sum,
                          int n_members, int n_params, int cand_stride, float sigma, void* stream);
int toued_es_adam(const float* grad_sum, float* mean, float* m, float* v, int popsize_global, int n_params,
                  float sigma, float lrate, float beta1, float beta2, float eps, int gen_counter, float mean_decay,
                  void* stream);

/* ---- device level generator (environments/gridworld/configs.py:12-57, environments.py:23-38) -------- */
/* Prioritised Level Replay index work on the device (environments/level_sampler.py:183-234, 331-408), one CTA.
 * The level buffer is score f32[B], active u8[B], is_new u8[B] (B <= 8192), updated in place.
 * toued_plr_reset_lowest = _reset_lowest_scoring (:331-353, quirk Q3 reproduced): writes the minimum_new ids of the
 *   lowest-scoring levels to reset_ids i32[minimum_new] and resets their score / flags; the caller regenerates those
 *   level records (toued_generate_levels with buffer_ids = reset_ids).
 * toued_plr_select = the buffer update with the regret scores of the terminated agents, _replay_from_buffer with
 *   score_transform "rank", _sample_random_from_buffer, the Bernoulli(p_replay) replay count, the permutation and the
 *   final choice (:183-234).  (key0, key1) = the sampler's rng right before split(rng, 3) at :201; old_ids /
 *   terminated / new_scores are those of the GLOBAL batch (n_agents <= B); shuffle_rounds =
 *   ceil(3 ln n / ln(2^32 - 1)) (jax _shuffle).  Writes new_ids i32[n_agents] and marks them active.
 * Float contract of the rank transform: exp_portable(clamp(score / temperature, -80, 80)), left-to-right fp32 sum.  */
int toued_plr_reset_lowest(float* score, uint8_t* active, uint8_t* is_new, int buffer_size, int minimum_new,
                           int* reset_ids, void* stream);
int toued_plr_select(uint32_t key0, uint32_t key1, float* score, uint8_t* active, uint8_t* is_new, int buffer_size,
                     const int* old_ids, const uint8_t* terminated, const float* new_scores, int n_agents,
                     float p_replay, float temperature, int shuffle_rounds, int* new_ids, void* stream);

/* One LevelRec per key: keys u32[n][2] are the per-level keys the reference passes to reset_env_params
 * (split(rng, n)); gen_desc is the mode description built by the host (to_ued_b200/environments/gridworld/levelgen.py,
 * toued_generate_levels_desc_bytes() bytes); buffer_ids i32[n] or NULL (0); lifetimes_out i32[n] or NULL.
 * Bit-exact with oracle/configs.py under the RNG / float contract of DESIGN.md section 2.            */
int toued_generate_levels_desc_bytes(void);
int toued_generate_levels(const void* gen_desc, const uint32_t* keys, const int32_t* buffer_ids, void* levels_out,
                          int32_t* lifetimes_out, int n_levels, void* stream);

/* ---- optimal return (environments/gridworld/gridworld.py:253-323 optimal_return) ------------------- */
/* out f64[n_levels] = the optimal expected undiscounted first-episode return of each LevelRec over `horizon` steps
 * (the level's max_steps caps the episode): exact finite-horizon DP over (cell, exists mask) in fp64 with a fixed
 * operation order, bitwise reproducible and independent of the batch.  max_n_objs <= 5, max_grid_size^2 <= 255;
 * a record outside those bounds gives NaN.                                                                  */
int toued_optimal_return(const void* levels, int n_levels, int horizon, int max_grid_size, int max_n_objs,
                         double* out, void* stream);

/* ---- double-oracle Nash solver (environments/nash_sampler.py:24-58, util/projection.py:9-38) ------ */
/* game f32[n][n] (row player x minimises x^T G y), supports = first x_nz / y_nz coordinates, n <= 1024.
 * Averaged iterates of num_iters projected-gradient steps (reference: 10,000 steps, lr 0.01).        */
int toued_get_nash(const float* game, const float* x0, const float* y0, float* x_out, float* y_out,
                   int n, int x_nz, int y_nz, int num_iters, float lr, void* stream);
int toued_projection_simplex(float* v, int n, int max_nz, void* stream);

/* ---- agent (re-)creation (agents/agents.py:31-95, level_sampler.py:273-291) --------------------- */

/* lecun-normal tables from threefry keys: keys u32[N][2], mask u8[N] or NULL (only masked agents are
 * written), tables f32[N][D][8] (columns >= n_out zeroed).                                          */
int toued_init_tables(const uint32_t* keys, const uint8_t* mask, float* tables, int n_agents,
                      int obs_dim, int n_out, void* stream);
/* reset the W environments (and the step counter, if given) of every masked agent.                  */
int toued_masked_reset(const void* levels, const uint8_t* mask, int32_t* state, int32_t* obs,
                       int32_t* step, int n_agents, int n_workers, int max_grid_size, void* stream);

/* Host helper (plain C loop, no GPU): out u32[n_keys][n] = threefry_2x32(keys[i], iota(n)), jax 0.4.13 rule
 * (jax/_src/prng.py threefry_random_bits): the host-side level generator / level sampler key plumbing.   */
int toued_host_iota_bits(const uint32_t* keys, int n_keys, int n, uint32_t* out);

/* ---- key derivation on the device (jax 0.4.13 threefry2x32 split, bit-exact) ---------------------- */

/* out u32[n_keys][count][2] = jax.random.split(keys_in[i], num)[offset : offset + count]
 * (meta/train.py:38 ``jax.random.split(rng, num_agents)``, restricted to a rank's agents).          */
int toued_key_split(const uint32_t* keys_in, int n_keys, int num, int offset, int count, uint32_t* out,
                    void* stream);
/* The ``rng, _rng = jax.random.split(rng)`` chain (lpg_agent.py:104-105, meta/train.py:40-42,109,
 * agents.py:99-103): keys_out u32[chain_len][n_keys][2] = the _rng of every link, carry_out
 * u32[n_keys][2] (or NULL) = the final rng.                                                          */
int toued_key_chain(const uint32_t* keys_in, int n_keys, int chain_len, uint32_t* keys_out,
                    uint32_t* carry_out, void* stream);

/* ---- tensor-core (tcgen05 / TMEM) path -------------------------------------------------------- */

/* Unit check of the tcgen05 building blocks: D f32[128][48] = A f32[128][256] * B f32[48][256]^T with
 * fp16 operands / fp32 accumulation in TMEM.  scratch_img: 24 KiB device scratch.                  */
int toued_tc_gemm_test(const float* A, const float* B, void* scratch_img, float* D, void* stream);
/* Same with K = 256 + 16: the last 16 K-columns live in no-swizzle K-major tiles (the layout of the
 * input-projection block of the GRU forward).  A f32[128][272], B f32[48][272]; scratch_img 32 KiB.   */
int toued_tc_gemm_mixed_test(const float* A, const float* B, void* scratch_img, float* D, void* stream);
/* Same for MN-major bf16 operands from token tile images: D f32[128][128] = A f32[128 k][128]^T * B f32[128 k][128]
 * (the weight-gradient GEMM shape).  scratch_img: 64 KiB.                                           */
int toued_tc_gemm_mn_test(const float* A, const float* B, void* scratch_img, float* D, int lbo, int sbo,
                          int kadv, void* stream);
/* the same contraction on a CTA pair (cta_group::2, M = 256 over a 2-cluster): D f32[256][256] = A[128 k][256 m]^T B[128 k][256 n];
 * scratch_img >= 128 KiB                                                                              */
int toued_tc_gemm_mn2_test(const float* A, const float* B, void* scratch_img, float* D, void* stream);
/* the weight-gradient GEMM's operand roles, fp16 (csrc/wgrad_tc.cu): D f32[128][256 + 16] = A[128 k][128 m]^T [B[128 k][256 n] |
 * X[128 k][0:16]] with X f32[128 k][64]; the X operand is the first 16 columns of one 64-column SW128 group (N = 16).
 * scratch_img >= 112 KiB                                                                              */
int toued_tc_gemm_mn_x16_test(const float* A, const float* B, const float* X, void* scratch_img, float* D, void* stream);

/* Pack the recurrent matrix Wh (+ input projection Wi, b_i) into the fp16 pass images the tensor-core
 * forward streams (wh_img: 16 x 26 KiB = 416 KiB, once per meta-step).                              */
int toued_pack_wh_forward(const float* lpg_params, void* wh_img, int lifetime_conditioning, void* stream);
/* Tensor-core version of toued_gru_forward (models/lpg.py:11-30,77-84): fp16 operands, fp32
 * accumulation in TMEM.  Saved for the reverse pass (NULL to skip; h16 may be NULL only when fac and hpimg are):
 *   h16   f16, RB32 layout [L][ceil(R/32)][32 chunks][32 rows][8 units] (csrc/tc.cuh::rb32_index)   h_t
 *   fac   f16 [L][R/32][4 planes][32 chunks][32 rows][8]: the gates r, z, n and hn = Whn h' + bhn as RB32 blocks with
 *         the planes interleaved per (t, 32-row block); the sign bits of the z plane carry relu'(h_t) (set: h_t <= 0).
 *         The reverse pass rebuilds its factors from them and takes h' from h16 of step t+1.
 *   hpimg bf16 token-tile image [L*Rp/64][4][64][64] of the masked carry h' used at each step
 * pi_hat / y_hat stay fp32.                                                                        */
int toued_gru_forward_tc(const float* x, const uint8_t* done, const float* lpg_params, const void* wh_img,
                         void* h16, void* fac, void* hpimg, float* pi_hat, float* y_hat, int n_agents,
                         int n_workers, int rollout_len, int lifetime_conditioning, void* stream);
/* Per-candidate variants for the ES path (meta/train.py:167-176: every agent runs its own LPG parameter vector):
 * agent n uses lpg_params + n * lpg_stride and the pass images wh_img + n * 425,984 bytes; one CTA per agent
 * (n_workers <= 128 sequences); inference only (no saved activations).                                   */
int toued_pack_wh_forward_multi(const float* lpg_params, void* wh_img, int lifetime_conditioning, int n_sets,
                                int lpg_stride, void* stream);
int toued_gru_forward_tc_multi(const float* x, const uint8_t* done, const float* lpg_params, const void* wh_img,
                               float* pi_hat, float* y_hat, int n_agents, int n_workers, int rollout_len,
                               int lifetime_conditioning, int lpg_stride, void* stream);

/* Pack Wh into the bf16 SW128 chunk images of the tensor-core reverse pass (384 KiB).               */
int toued_pack_wh_backward(const float* lpg_params, void* whb_img, void* stream);
/* Scaled fp16 reverse pass.  The reverse pass is linear in the cotangents (d_pi_hat, d_y_hat), which are far below
 * fp16's range: the tensor-core reverse kernels derive a power of two S from max |cotangent|, run on S x cotangents
 * with fp16 operands (saturating conversions) and fp32 accumulation, and the consumers divide S back out.
 * cotangent_max u32[2] of one launch = {max, status}:
 *   [0] max |cotangent| as the bit pattern of a float, +inf if any cotangent is inf or NaN (then S = 1);
 *       written by toued_cotangent_max, which resets this word only;
 *   [1] status bits, OR-ed in and never cleared by a kernel (the caller zeroes the word): a set bit means the result of
 *       the launch may be wrong.  TOUED_STATUS_NONFINITE_COT: toued_cotangent_max saw an inf / NaN cotangent.
 *       TOUED_STATUS_FP16_RANGE: toued_gru_backward_tc or toued_lpg_wgrad_tc met an fp16 operand with |S v| > 65504
 *       (saturated: the carry grew past ~2^12 x max |cotangent| along the chain) or non-finite.
 * cotangent_max == NULL means S = 1 and no status.                                                            */
#define TOUED_STATUS_NONFINITE_COT 1u
#define TOUED_STATUS_FP16_RANGE 2u
int toued_cotangent_max(const float* d_pi_hat, const float* d_y_hat, int n_agents, int n_workers, int rollout_len,
                        uint32_t* cotangent_max, void* stream);
/* Tensor-core BPTT (reverse of toued_gru_forward_tc).  Reads h16 / fac saved by the forward; writes, in units of S,
 *   dgimg fp16 token-tile image [L*Rp/64][16][64][64]: column groups 0-3 dar, 4-7 daz, 8-11 dhn, 12-15 dan
 *   dl f32[L][R][8] head-logit cotangents, dx f32[L][R][2] (d pyt, d pyt1)                          */
int toued_gru_backward_tc(const uint8_t* done, const float* lpg_params, const void* whb_img,
                          const void* h16, const void* fac, const float* y_hat, const float* d_pi_hat,
                          const float* d_y_hat, void* dgimg, float* dl, float* dx, uint32_t* cotangent_max,
                          int n_agents, int n_workers, int rollout_len, int lifetime_conditioning, void* stream);
/* Tensor-core weight gradients from the token tile images (hpimg from the forward, dgimg from the
 * backward) + streaming small gradients; partial areas of the toued_lpg_wgrad workspace.             */
int toued_wgrad_tc_splits(void);
int toued_wgrad_tc_small_splits(void);
int toued_lpg_wgrad_tc(const void* hpimg, const void* dgimg, const void* ximg, const void* h16,
                       const float* d_pi_hat, const float* dl, float* wh_partials, float* small_partials,
                       uint32_t* cotangent_max, int n_agents, int n_workers, int rollout_len, int accumulate,
                       void* stream);

#ifdef __cplusplus
}
#endif
#endif
