/*
 * lzb200.h -- C ABI of the B200-native batched MuZero MCTS + inference engine.
 *
 * This is the drop-in boundary for ONE hot path of opendilab/LightZero (file:line relative to the
 * reference repository root):
 *
 *   lzero/mcts/ctree/ctree_muzero/mz_tree.pyx:5-107   (the Cython surface: Roots, MinMaxStatsList,
 *        ResultsWrapper, batch_traverse, batch_backpropagate)  -> lz_tree_*
 *   lzero/mcts/ctree/ctree_muzero/lib/cnode.cpp:83-147,169-203,301-358,387-500,551-595,654-698,754-825
 *        (expand / compute_mean_q / prepare / results / backpropagate / select / ucb / traverse)
 *   lzero/mcts/ctree/common_lib/cminimax.cpp:7-66      (MinMaxStats)          -> folded into lz_tree
 *   lzero/model/muzero_model.py:210-272                (initial/recurrent_inference) -> lz_model_*
 *   lzero/policy/scaling_transform.py:64-92            (InverseScalarTransform) -> fused in lz_model_*
 *   lzero/mcts/tree_search/mcts_ctree.py:267-368       (MuZeroMCTSCtree.search loop) -> lz_search_*
 *   lzero/policy/muzero.py:749-779                     (_forward_collect inner part) -> lz_search_collect
 *
 * Conventions
 *   - every function returns 0 on success or a negative LZ_E* code; lz_last_error() gives the
 *     message of the last failure on the calling thread.  No C++ exception crosses this boundary.
 *   - pointers named d_* are DEVICE pointers, h_* are HOST pointers.  Plain pointers and sizes only.
 *   - every compute call takes the cudaStream_t (passed as void*) it is enqueued on and performs
 *     NO host<->device synchronisation; results are valid once the stream reaches that point.
 *   - a handle must be used from one stream at a time (thread-compatible, no global state).
 *   - there is no CPU fallback: without a CUDA device every create call fails with LZ_ECUDA.
 *   - tie-breaking: `deterministic != 0` picks the first legal action attaining the exact maximum
 *     (cnode.cpp:592 front()); 0 draws uniformly among the reference's epsilon-tie list with a
 *     counter-based device RNG (the reference reseeds rand() from the wall clock, cnode.cpp:770).
 */
#ifndef LZB200_H
#define LZB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LZ_OK 0
#define LZ_EINVAL (-1)   /* bad argument */
#define LZ_ECUDA (-2)    /* CUDA runtime error (message has the cudaError string) */
#define LZ_ESTATE (-3)   /* call order violated (e.g. search before prepare) */
#define LZ_ENOMEM (-4)

typedef struct lz_tree lz_tree;
typedef struct lz_model lz_model;
typedef struct lz_search lz_search;
typedef struct lz_frames lz_frames;       /* device-resident observation frame stacks of B environments */
typedef struct lz_segments lz_segments;   /* device-resident search statistics of B game segments */
typedef void *lz_stream;   /* cudaStream_t */

int lz_version(void);
/* Launch accounting: kernels this library has enqueued since load (kernel nodes of launched graphs included). */
unsigned long long lz_debug_launch_count(void);
const char *lz_last_error(void);

/* ------------------------------------------------------------------ tree (mz_tree / cnode.cpp) */

/* B trees, A actions, room for max_sims expansions per tree (node slot k == latent index k). */
int lz_tree_create(int B, int A, int max_sims, lz_tree **out);
int lz_tree_destroy(lz_tree *t);

/* Search constants (mcts_ctree.py:286,292): PUCT constants, discount, MinMax value_delta_max.
 * Precomputes the per-visit-count exploration table on the host with libm logf (cnode.cpp:672). */
int lz_tree_set_params(lz_tree *t, int pb_c_base, float pb_c_init, float discount, float value_delta_max);

/* CRoots::CRoots (cnode.cpp:301-317).  d_legal: int32 [B,A] legal action ids in the caller's order,
 * -1 padded; d_nlegal: int32 [B] (0 == all actions, cnode.cpp:101-107).  Both NULL == all legal.
 * Also resets MinMax stats (a fresh MinMaxStatsList per search, mcts_ctree.py:291-292). */
int lz_tree_reset(lz_tree *t, const int32_t *d_legal, const int32_t *d_nlegal, lz_stream s);
/* Same from a mask uint8 [B,A] (legal ids ascending == np.nonzero order, policy/muzero.py:760). */
int lz_tree_reset_mask(lz_tree *t, const uint8_t *d_mask, lz_stream s);

/* CRoots::prepare / prepare_no_noise (cnode.cpp:321-358).  d_logits f32 [B,A] by action id;
 * d_noise f32 [B,A] rows in LEGAL ORDER (first nlegal[b] used) or NULL for prepare_no_noise;
 * d_rewards f32 [B] or NULL (zeros); d_to_play int32 [B] (-1 == single player). */
int lz_tree_prepare(lz_tree *t, const float *d_logits, const float *d_noise, float noise_weight,
                    const float *d_rewards, const int32_t *d_to_play, lz_stream s);

/* cbatch_traverse (cnode.cpp:754-825): one PUCT descent per tree.  Outputs (each int32 [B], may be
 * NULL): latent-pool slot of the leaf's parent (== its current_latent_state_index), batch index
 * (== tree index), last action, search length, virtual to_play after the descent. */
int lz_tree_traverse(lz_tree *t, int deterministic, int32_t *d_ix, int32_t *d_iy,
                     int32_t *d_last_action, int32_t *d_search_len, int32_t *d_virtual_to_play,
                     lz_stream s);

/* cbatch_backpropagate (cnode.cpp:480-500): expand the leaves found by the last traverse into slot
 * `latent_index` (simulation_index + 1) and back up.  d_reward/d_value f32 [B] (scalars, after the
 * inverse transform), d_logits f32 [B,A]; d_to_play int32 [B] or NULL (use the virtual to_play the
 * last traverse produced, which is what mcts_ctree.py:365-368 passes). */
int lz_tree_backpropagate(lz_tree *t, int latent_index, const float *d_reward, const float *d_value,
                          const float *d_logits, const int32_t *d_to_play, lz_stream s);

/* ---- EfficientZero tree (lzero/mcts/ctree/ctree_efficientzero/lib/cnode.cpp, ez_tree.pyx) ----
 * lz_tree_set_ez switches a tree to value-prefix semantics before lz_tree_prepare: the reward slot carries the child's
 * value prefix, every expanded node carries is_reset, the reward of a step is the prefix difference unless the parent
 * was reset (cnode.cpp:185-195, 496-573, 786-790).  lstm_horizon_len (mcts_ctree.py:857) is used by the fused search
 * and by lz_tree_traverse_ez to derive is_reset = (search_len % lstm_horizon_len == 0).
 * The reference tie-break is rand() % len(ties) with no deterministic switch (cnode.cpp:691); these entry points use
 * the first-maximum rule, which is that draw with rand() == 0 (how the parity oracle builds the reference). */
int lz_tree_set_ez(lz_tree *t, int efficientzero, int lstm_horizon_len);
/* Tie-breaking of the EfficientZero and *_with_reuse descents, which have no deterministic switch in the reference (they draw
 * rand() % len(ties) after reseeding from the wall clock, ctree_efficientzero/lib/cnode.cpp:691, ctree_muzero cnode.cpp:610-640):
 * first_maximum = 1 (default; the reference's draw with rand() == 0, what the parity tests pin) or 0 = a uniform draw from the same tie
 * list with the counter-based device RNG of lz_tree_traverse(deterministic = 0). */
int lz_tree_set_tiebreak(lz_tree *t, int first_maximum);
/* cbatch_traverse (ctree_efficientzero cnode.cpp:876-958); d_is_reset int32 [B] out (may be NULL). */
int lz_tree_traverse_ez(lz_tree *t, int32_t *d_ix, int32_t *d_iy, int32_t *d_last_action, int32_t *d_search_len,
                        int32_t *d_virtual_to_play, int32_t *d_is_reset, lz_stream s);
/* cbatch_backpropagate (ctree_efficientzero cnode.cpp:577-601): value prefixes instead of rewards + is_reset_list. */
int lz_tree_backpropagate_ez(lz_tree *t, int latent_index, const float *d_value_prefix, const float *d_value,
                             const float *d_logits, const int32_t *d_is_reset, const int32_t *d_to_play, lz_stream s);

/* get_distributions / get_values / get_trajectories (cnode.cpp:237-277,369-417).
 * d_visits int32 [B,A] in legal order, -1 padded; d_values f32 [B]; d_nlegal int32 [B];
 * d_traj int32 [B, max_sims+1] -1 padded.  Any pointer may be NULL. */
int lz_tree_results(lz_tree *t, int32_t *d_visits, float *d_values, int32_t *d_nlegal,
                    int32_t *d_traj, lz_stream s);

/* ---- ReZero search_with_reuse (cnode.cpp:502-549, 597-652, 701-752, 828-932; SURVEY 8(f) row f-4); works on MuZero trees and,
 * with value-prefix semantics, on EfficientZero trees (ctree_efficientzero/lib/cnode.cpp:603-650, 699-754, 816-874, 960-1072) ----
 * d_true_action int32 [B] / d_reuse_value f32 [B]: the action taken in the stored trajectory and the value to reuse for it.
 * The root scores that child with carm_score and the descent stops right after the root when it is selected.  d_ix reports -1
 * for trees that stopped on an already expanded child ("no inference"); d_iy is the batch_index recorded when the parent was
 * expanded (the compact inference row under reuse).  Ties: first maximum (= the reference's rand() % len(ties) with rand()
 * == 0; these reference routines have no deterministic switch). */
int lz_tree_traverse_with_reuse(lz_tree *t, const int32_t *d_true_action, const float *d_reuse_value, int32_t *d_ix, int32_t *d_iy,
                                int32_t *d_last_action, int32_t *d_search_len, int32_t *d_virtual_to_play, lz_stream s);
/* cbatch_backpropagate_with_reuse: rows are indexed BY TREE (not compacted; rows of "no inference" trees are ignored).
 * d_batch_rank int32 [B] or NULL: compact row of each tree in the caller's inference batch, stored as the batch_index of the
 * node it expands.  d_is_reset int32 [B]: EfficientZero trees only (NULL otherwise).  Which trees skip the expansion / back up
 * the reuse value is the state the last traverse left. */
int lz_tree_backpropagate_with_reuse(lz_tree *t, int latent_index, const float *d_reward, const float *d_value, const float *d_logits,
                                     const float *d_reuse_value, const int32_t *d_batch_rank, const int32_t *d_is_reset,
                                     const int32_t *d_to_play, lz_stream s);

/* select_action (lzero/policy/utils.py:637-661) on the device, from the root visit counts of the finished search:
 * p = visit ** (1 / temperature) / sum (fp64), d_entropy = -sum p log2 p (scipy.stats.entropy(p, base=2)), d_action_pos = arg-max (deterministic != 0; the
 * eval path, policy/muzero.py:935) or one draw from p (inverse CDF of a counter-based uniform keyed by seed and tree index;
 * the reference draws with np.random.choice), d_action = the action id at that legal position (policy/muzero.py:800).
 * Outputs int32 [B] / f32 [B], any may be NULL.  SURVEY 8(f) row f-3: keeps the collector's action choice on the GPU. */
int lz_tree_select_action(lz_tree *t, float temperature, int deterministic, uint64_t seed, int32_t *d_action,
                          int32_t *d_action_pos, float *d_entropy, lz_stream s);

/* ---- Gumbel MuZero tree (lzero/mcts/ctree/ctree_gumbel_muzero/lib/cnode.cpp, gmz_tree.pyx) ----
 * lz_tree_set_gumbel switches a tree to Gumbel mode (before lz_tree_prepare_gumbel) and precomputes on the host the fixed
 * Gumbel draw (std::mt19937(0), 10 * extreme_value(0, 1), cnode.cpp:1133-1151; every root uses the prefix of its legal-list
 * length) and the considered-visit row get_sequence_of_considered_visits(min(m, S), S) (:1041-1094).  Root choice is
 * sequential halving (cselect_root_child, :701-745), interior choice the completed-Q improved policy (cselect_interior_child,
 * :747-790).  Nothing on the search path draws random numbers: every call reproduces the reference bit for bit.
 * LZ_EINVAL when num_simulations exceeds the tree's max_sims. */
int lz_tree_set_gumbel(lz_tree *t, int num_simulations, int max_num_considered_actions);
/* CRoots::prepare / prepare_no_noise (cnode.cpp:418-455): lz_tree_prepare plus the root's raw value d_values f32 [B] (NULL: 0). */
int lz_tree_prepare_gumbel(lz_tree *t, const float *d_logits, const float *d_noise, float noise_weight,
                           const float *d_rewards, const float *d_values, const int32_t *d_to_play, lz_stream s);
/* cbatch_traverse (cnode.cpp:834-897); outputs as lz_tree_traverse, d_virtual_to_play = the root to_play unchanged.
 * LZ_ESTATE for more than num_simulations traverses since the last prepare (the reference indexes past its table). */
int lz_tree_traverse_gumbel(lz_tree *t, float discount, int32_t *d_ix, int32_t *d_iy, int32_t *d_last_action,
                            int32_t *d_search_len, int32_t *d_virtual_to_play, lz_stream s);
/* cbatch_back_propagate (cnode.cpp:605-652): expand the leaves into slot latent_index, store d_value as their raw value, back up
 * (single-player recurrence for every to_play: the reference asserts to_play == -1 and is built with NDEBUG). */
int lz_tree_backpropagate_gumbel(lz_tree *t, int latent_index, float discount, const float *d_reward,
                                 const float *d_value, const float *d_logits, lz_stream s);
/* get_children_values (cnode.cpp:309-338) -> d_children_values f32 [B,A] by action id, -inf for illegal actions;
 * get_policies (:355-385) -> d_improved_policy f32 [B,A] by action id, illegal entries 0;
 * d_action int32 [B]: np.argmax of the improved policy with illegal entries 0 (gumbel_muzero.py:591-592).  Any may be NULL.
 * Visit counts, root values and trajectories come from lz_tree_results. */
int lz_tree_results_gumbel(lz_tree *t, float discount, float *d_children_values, float *d_improved_policy,
                           int32_t *d_action, lz_stream s);

/* ------------------------------------------------------------------ model (muzero_model.py, efficientzero_model.py) */

typedef struct lz_model_config {
    int obs_c, obs_h, obs_w;       /* observation planes and size: (4|12, 64|84|96, same) */
    int action_space_size;
    int num_res_blocks;            /* per network (reference default 1) */
    int num_channels;              /* 64 */
    int reward_head_channels, value_head_channels, policy_head_channels;   /* 16 */
    int reward_hidden, value_hidden, policy_hidden;                         /* one hidden layer: 32 */
    float support_min, support_max, support_step;                           /* -300, 301, 1 (value == reward) */
    /* EfficientZeroModel (lzero/model/efficientzero_model.py:20-272): the reward head becomes conv1x1 -> BN -> ReLU ->
     * LSTM(hc*36 -> lstm_hidden_size) -> BN1d -> ReLU -> MLP and predicts a VALUE PREFIX; 0 = MuZeroModel */
    int efficientzero;
    int lstm_hidden_size;          /* 512 (must be a multiple of 16, <= 512) */
} lz_model_config;

int lz_model_create(const lz_model_config *cfg, lz_model **out);

/* MuZeroModelMLP (lzero/model/muzero_model_mlp.py:21-295; vector observations, BASELINE config 1).  The
 * handle is used with the same lz_model_* / lz_search_* calls: d_obs is f32 [B, obs_dim], latents are
 * f32 [B, latent_dim].  State-dict names follow muzero_model_mlp.py / common.py:790-850,1218-1292. */
typedef struct lz_mlp_config {
    int obs_dim, action_space_size, latent_dim;         /* 4, 2, 128 for CartPole */
    int reward_hidden, value_hidden, policy_hidden;     /* one hidden layer each: 32 */
    int res_connection_in_dynamics;                     /* policy default True (policy/muzero.py:68) */
    float support_min, support_max, support_step;
} lz_mlp_config;
int lz_model_create_mlp(const lz_mlp_config *cfg, lz_model **out);
int lz_model_destroy(lz_model *m);
/* Feed one tensor of the reference state_dict (names as produced by MuZeroModel.state_dict(),
 * SURVEY.md App. B.4; fp32, contiguous, HOST memory).  Unknown names are ignored (returns 1). */
int lz_model_set_tensor(lz_model *m, const char *name, const float *h_data, int64_t numel);
/* Folds eval-mode BatchNorm into per-channel scale/shift, packs weights for the kernels, uploads. */
int lz_model_finalize(lz_model *m);
/* Arithmetic of the latent-grid networks (recurrent_inference and the tail of initial_inference):
 *   0 = fp32 FFMA on the CUDA cores;
 *   1 = tcgen05 tensor cores with fp16 hi/lo operand splitting (3 MMAs per product, fp32 accumulate in
 *       TMEM): fp32-accurate, the mode parity is stated for;
 *   2 = tcgen05 single fp16 pass (fp32 accumulate): ~3x fewer MMAs, logits accurate to ~1e-3. */
int lz_model_set_math(lz_model *m, int mode);
/* Test hook: overrides the layer program of the tcgen05 kernels (see net_tc.cuh LF_* flags). */
int lz_model_debug_tc_program(lz_model *m, int which, int nlayers, const int *layer_w, const int *layer_flags,
                              int has_reward);
/* Test hook: 64 clock64 stamps of CTA 0 of the last tcgen05 launch made with env LZ_TC_DEBUG=1. */
int lz_debug_tc_stamps(unsigned long long *h_out);
int lz_model_latent_hw(const lz_model *m);   /* 6 for 84/96, 8 for 64 */
int lz_model_support_size(const lz_model *m);

/* initial_inference (muzero_model.py:210-240).  d_obs f32 [B,obs_c,H,W].  Outputs (NULL to skip):
 * d_latent f32 [B,C,h,w] (NCHW, as the reference returns), d_policy_logits f32 [B,A],
 * d_value_logits f32 [B,support], d_value f32 [B] (inverse-transformed scalar). */
int lz_model_initial_inference(lz_model *m, int B, const float *d_obs, float *d_latent,
                               float *d_policy_logits, float *d_value_logits, float *d_value,
                               lz_stream s);
/* recurrent_inference (muzero_model.py:242-272).  d_latent f32 [B,C,h,w], d_action int32 [B].
 * Outputs (NULL to skip): d_next_latent [B,C,h,w], d_reward_logits/d_value_logits [B,support],
 * d_policy_logits [B,A], d_reward/d_value f32 [B] scalars after the inverse transform. */
int lz_model_recurrent_inference(lz_model *m, int B, const float *d_latent, const int32_t *d_action,
                                 float *d_next_latent, float *d_reward_logits, float *d_value_logits,
                                 float *d_policy_logits, float *d_reward, float *d_value, lz_stream s);
/* EfficientZeroModel.recurrent_inference (efficientzero_model.py:240-272).  The reward hidden state is the tuple the
 * reference passes to nn.LSTM: d_hidden0 = element 0 (LSTM h), d_hidden1 = element 1 (LSTM c), each f32 [B, lstm_hidden_size]
 * (the leading sequence dimension of 1 dropped).  Outputs as lz_model_recurrent_inference with the value prefix in place of
 * the reward, plus the next hidden state (un-reset: resetting every lstm_horizon_len steps is the search driver's job,
 * mcts_ctree.py:856-861).  initial_inference is lz_model_initial_inference (the hidden state starts as zeros). */
int lz_model_recurrent_inference_ez(lz_model *m, int B, const float *d_latent, const float *d_hidden0, const float *d_hidden1,
                                    const int32_t *d_action, float *d_next_latent, float *d_next_hidden0, float *d_next_hidden1,
                                    float *d_value_prefix_logits, float *d_value_logits, float *d_policy_logits,
                                    float *d_value_prefix, float *d_value, lz_stream s);
int lz_model_lstm_hidden_size(const lz_model *m);   /* 0 for a MuZero model */

/* InverseScalarTransform (scaling_transform.py:82-92) on its own: logits f32 [B,support] -> f32 [B]. */
int lz_inverse_scalar_transform(lz_model *m, int B, const float *d_logits, float *d_out, lz_stream s);

/* ------------------------------------------------------------------ fused search (mcts_ctree.py) */

/* Binds a tree and a model; owns the latent pool [(num_simulations+1), B, C, h, w] and the CUDA
 * graph holding [traverse -> recurrent_inference -> backpropagate] x num_simulations. */
int lz_search_create(lz_tree *t, lz_model *m, int num_simulations, lz_search **out);
int lz_search_destroy(lz_search *q);
/* MuZeroMCTSCtree.search (mcts_ctree.py:267-368) on roots already prepared with lz_tree_prepare.
 * d_latent_roots f32 [B,C,h,w].  One graph launch, zero host syncs. */
int lz_search_run(lz_search *q, const float *d_latent_roots, int deterministic, lz_stream s);
/* MuZeroMCTSCtree.search_with_reuse (mcts_ctree.py:370-468; ReZero).  d_true_action int32 [B], d_reuse_value f32 [B] as for
 * lz_tree_traverse_with_reuse; d_infer_count int32 [num_simulations] or NULL receives, per simulation, how many trees needed
 * the network (the reference returns the last count and the mean).  One CUDA graph; "no inference" rows are computed and
 * ignored instead of compacted on the host. */
int lz_search_run_with_reuse(lz_search *q, const float *d_latent_roots, const int32_t *d_true_action, const float *d_reuse_value,
                             int32_t *d_infer_count, lz_stream s);
/* EfficientZeroMCTSCtree.search (mcts_ctree.py:671-876) for a search created from an EfficientZero model and a tree in
 * EfficientZero mode.  d_hidden{0,1}_roots: f32 [B, lstm_hidden_size] = reward_hidden_state_roots[0] / [1] (NULL = zeros,
 * what initial_inference returns).  The LSTM state of a leaf is zeroed every lstm_horizon_len steps of depth (:856-861). */
int lz_search_run_ez(lz_search *q, const float *d_latent_roots, const float *d_hidden0_roots, const float *d_hidden1_roots, lz_stream s);
/* EfficientZeroMCTSCtree.search_with_reuse (mcts_ctree.py:878-1003; ReZero on the value-prefix trees): arguments of lz_search_run_ez
 * plus d_true_action / d_reuse_value / d_infer_count of lz_search_run_with_reuse.  One CUDA graph (1 + 5 x num_simulations
 * kernels); is_reset is taken per TREE from the descent (search_len % lstm_horizon_len; the reference indexes a compacted list by
 * tree at :1040-1046 / cnode.cpp:646, see DESIGN.md 4.6). */
int lz_search_run_ez_with_reuse(lz_search *q, const float *d_latent_roots, const float *d_hidden0_roots, const float *d_hidden1_roots,
                                const int32_t *d_true_action, const float *d_reuse_value, int32_t *d_infer_count, lz_stream s);
/* GumbelMuZeroMCTSCtree.search (mcts_ctree.py:1076-1174) on roots prepared with lz_tree_prepare_gumbel, for a search created
 * from a MuZero model (conv or MLP) and a tree set to Gumbel mode with num_simulations equal to the search's.  One CUDA graph
 * [traverse] + S x [recurrent_inference, backpropagate (+ next traverse)], re-captured when the weights, the tree's Gumbel
 * parameters or the discount change. */
int lz_search_run_gumbel(lz_search *q, const float *d_latent_roots, float discount, lz_stream s);
/* The search-feeding part of _forward_collect (policy/muzero.py:749-779): initial_inference ->
 * reset(mask) -> prepare(noise) -> search.  d_obs f32 [B,obs_c,H,W]; d_mask uint8 [B,A] or NULL;
 * d_noise f32 [B,A] legal-order rows or NULL; d_to_play int32 [B] or NULL (-1).
 * Optional outputs: d_pred_value f32 [B] (root value prediction), d_policy_logits f32 [B,A]. */
int lz_search_collect(lz_search *q, const float *d_obs, const uint8_t *d_mask, const float *d_noise,
                      float noise_weight, const int32_t *d_to_play, int deterministic,
                      float *d_pred_value, float *d_policy_logits, lz_stream s);
/* Same with HOST buffers (pinned memory recommended): h_obs f32 [B,obs_c,H,W], h_mask uint8 [B,A] or NULL,
 * h_noise f32 [B,A] or NULL, h_to_play int32 [B] or NULL.  The observation batch is copied in `nchunks`
 * (1..8) pieces on an internal copy stream so that the copy of chunk i+1 overlaps the representation
 * network of chunk i; everything else is ordered on `s`.  The host buffers must stay valid until `s`
 * reaches the end of the call's work. */
int lz_search_collect_host(lz_search *q, const float *h_obs, const uint8_t *h_mask, const float *h_noise,
                           float noise_weight, const int32_t *h_to_play, int deterministic, int nchunks,
                           float *d_pred_value, float *d_policy_logits, lz_stream s);
/* The same two entry points for uint8 frames [B,obs_c,H,W] (Atari frames as the emulator delivers them; a quarter of the
 * bytes on the wire).  The [0, 1] scaling of the reference's env wrapper (ScaledFloatFrameWrapper: obs / 255 -> float32,
 * zoo/atari/envs/atari_wrappers.py:219-220, atari_lightzero_env.py:87-88) is applied inside the first conv kernel, bit-identical
 * to that host arithmetic.  tcgen05 conv model with 84x84 / 96x96 frames only. */
int lz_search_collect_u8(lz_search *q, const uint8_t *d_obs_u8, const uint8_t *d_mask, const float *d_noise,
                         float noise_weight, const int32_t *d_to_play, int deterministic,
                         float *d_pred_value, float *d_policy_logits, lz_stream s);
int lz_search_collect_host_u8(lz_search *q, const uint8_t *h_obs_u8, const uint8_t *h_mask, const float *h_noise,
                              float noise_weight, const int32_t *h_to_play, int deterministic, int nchunks,
                              float *d_pred_value, float *d_policy_logits, lz_stream s);
/* Number of kernel nodes one lz_search_run enqueues (for launch accounting). */
int lz_search_num_kernels(const lz_search *q);
/* Device pointer of the latent pool (NCHW per slot) for inspection in tests. */
const float *lz_search_latent_pool(const lz_search *q);
/* EfficientZero: device LSTM-state pool [(S+1)][B][H], which = 0 / 1 for tuple element 0 / 1 (NULL for MuZero). */
const float *lz_search_hidden_pool(const lz_search *q, int which);


/* ---- collector state on the device (SURVEY 8(f) row f-3) ----
 * Observation frame stacks: what the reference collector rebuilds on the host every step with
 * GameSegment.get_obs() = obs_segment[t : t + frame_stack_num] (lzero/mcts/buffer/game_segment.py:140-156), seeded with
 * frame_stack_num copies of the first frame (lzero/worker/muzero_collector.py:451-457) and fed one new frame per step
 * (GameSegment.append, game_segment.py:158-181; muzero_collector.py:520-545).  Here only the NEW uint8 frame of every environment
 * crosses PCIe (B*H*W bytes instead of B*stack*H*W*4); lz_frames_stacked() is the [B, stack, H, W] uint8 batch (oldest frame
 * first) that lz_search_collect_u8 consumes.  H*W must be a multiple of 16. */
int lz_frames_create(int B, int stack, int H, int W, lz_frames **out);
int lz_frames_destroy(lz_frames *f);
/* d_new_frames uint8 [B,H,W]; d_reset uint8 [B] or NULL: 1 = the environment was reset, its whole stack becomes the new frame. */
int lz_frames_push(lz_frames *f, const uint8_t *d_new_frames, const uint8_t *d_reset, lz_stream s);
/* The same from HOST buffers (pinned memory recommended); they must stay valid until `s` reaches the copies. */
int lz_frames_push_host(lz_frames *f, const uint8_t *h_new_frames, const uint8_t *h_reset, lz_stream s);
/* Device pointer of the current stacks; valid until the next push. */
const uint8_t *lz_frames_stacked(lz_frames *f);
/* GameSegment.store_search_stats (game_segment.py:241-263, idx=None) for B segments of capacity T: appends
 * child_visits[b][len[b]][k] = visit_counts[k] / sum(visit_counts) (computed in float64 as Python does, 1e-6 denominator when every
 * count is 0; k = position in the root's legal-action list, 0 beyond it) and root_values[b][len[b]].  d_visits int32 [B,A] / d_values
 * f32 [B] as lz_tree_results returns them (-1 beyond the legal list); d_active uint8 [B] or NULL selects the environments that
 * stepped.  A full segment (len == T) is left unchanged. */
int lz_segments_create(int B, int T, int A, lz_segments **out);
int lz_segments_destroy(lz_segments *g);
int lz_segments_store_search_stats(lz_segments *g, const int32_t *d_visits, const float *d_values, const uint8_t *d_active, lz_stream s);
/* GameSegment.reset (game_segment.py:340-362) of the statistics: len = 0 where d_done[b] != 0 (NULL: everywhere). */
int lz_segments_reset(lz_segments *g, const uint8_t *d_done, lz_stream s);
/* Device pointers: child_visits f32 [B,T,A], root_values f32 [B,T], len int32 [B] (any may be NULL). */
int lz_segments_data(lz_segments *g, float **d_child_visits, float **d_root_values, int32_t **d_len);

#ifdef __cplusplus
}
#endif
#endif /* LZB200_H */
