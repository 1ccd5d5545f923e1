// tree.cuh -- device-resident batched MuZero search trees: data layout + warp-per-tree device code.
//
// Replaces lzero/mcts/ctree/ctree_muzero/lib/cnode.{h,cpp} + common_lib/cminimax.{h,cpp}.
// Design (not a port of the std::map tree):
//   * one warp per tree, lane <-> child (legal position); all B trees advance in one launch;
//   * node slot k of a tree IS the latent-pool index k (root = 0, node expanded by simulation s = s+1),
//     so "current_latent_state_index" needs no storage and the pool gather index is (slot, tree);
//   * the statistics of a child (prior, value_sum, reward, visit_count, child slot) are stored on the
//     EDGE, in the parent's node block [5][A] of 32-bit words, contiguous per node, so one PUCT
//     scan touches one 20*A-byte block (A=6: a single 128 B line) with coalesced lane loads;
//   * order-sensitive fp32 reductions (softmax denominator cnode.cpp:127-132, compute_mean_q
//     cnode.cpp:179-191, the backup recurrence cnode.cpp:435-448) are evaluated in the reference's
//     sequential order via warp shuffles; max / argmax use exact (order-free) warp reductions;
//   * every fp32 operation uses an explicit round-to-nearest intrinsic (no FMA contraction: the
//     reference is built for baseline x86-64) and expf is the glibc-exact lz_expf_exact.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "lz_exact_math.h"

namespace lz {

constexpr float kFloatMax = 1000000.0f;   // cminimax.h:9
constexpr float kFloatMin = -kFloatMax;   // cminimax.h:10
constexpr int kEdgeFields = 5;            // prior, vsum, reward, visit, cslot
enum { F_PRIOR = 0, F_VSUM = 1, F_REWARD = 2, F_VISIT = 3, F_CSLOT = 4 };

struct TreeParams {
    int B, A, N;                 // trees, actions, node slots per tree (max_sims + 1)
    uint32_t *edges;             // [B][N][5][A]
    int *n_to_play, *n_best;     // [B][N]
    int *legal, *nlegal;         // [B][A], [B]
    int *root_visit;             // [B]
    float *root_vsum, *root_reward;
    float *mm_max, *mm_min;      // [B]
    int *to_play;                // [B] root to_play given at prepare
    int *players_max;            // [1] max over to_play (players = max == -1 ? 1 : 2, cnode.cpp:776-781)
    int *path_slot, *path_action, *path_len;   // [B][N], [B][N], [B]
    int *vtp;                    // [B] virtual to_play after the last traverse
    int *search_len;             // [B]
    const float *pbc;            // [N+1]: logf((n + base + 1) / base) + pb_c_init for n = visit_count - 1
    float discount, delta;
    unsigned long long rng_seed;
    unsigned long long *rng_epoch;   // [1] bumped by every reset so graph replays draw fresh ties
    // EfficientZero mode (ctree_efficientzero): the edge "reward" word holds the child's VALUE PREFIX, every expanded node
    // carries is_reset, and a step's reward is the prefix difference unless the parent was reset
    int ez, lstm_horizon;
    int tie_first;             // EfficientZero / *_with_reuse descents (the reference draws rand() % len(ties) there): 1 = first maximum (default), 0 = uniform draw
    int *n_reset;                // [B][N]
    // ReZero search_with_reuse (cnode.cpp:502-549, 597-652, 701-752, 828-932)
    int *n_batch;                // [B][N] batch_index recorded at expansion (the compacted inference row under reuse)
    int *reuse_state;            // [B] result of the last traverse_with_reuse: 0 normal leaf, 1 stopped at the root's true_action
                                 //     on an unexpanded child (expand, back up the reuse value), 2 stopped on an expanded child
                                 //     (no inference, no expansion, back up the reuse value)
    int *infer_count;            // [N] per-simulation number of trees that needed the network (search_with_reuse statistics)
};

__device__ __forceinline__ float u2f(uint32_t u) { return __uint_as_float(u); }
__device__ __forceinline__ uint32_t f2u(float f) { return __float_as_uint(f); }

__device__ __forceinline__ float warp_max_exact(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

__device__ __forceinline__ unsigned long long mix64(unsigned long long z)
{
    z += 0x9e3779b97f4a7c15ull;
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
    return z ^ (z >> 31);
}

// MinMaxStats::normalize (cminimax.cpp:33-45)
__device__ __forceinline__ float mm_normalize(float value, float mmax, float mmin, float delta_max)
{
    float norm_value = value;
    float delta = __fsub_rn(mmax, mmin);
    if (delta > 0.0f) {
        if (delta < delta_max) norm_value = __fdiv_rn(__fsub_rn(norm_value, mmin), delta_max);
        else norm_value = __fdiv_rn(__fsub_rn(norm_value, mmin), delta);
    }
    return norm_value;
}

// cucb_score (cnode.cpp:654-698; EZ: ctree_efficientzero/lib/cnode.cpp:756-814) for the child held by this lane.
// arm = true: carm_score (cnode.cpp:701-752) -- the stored reuse value replaces the child's mean value and a visited child
// scores without the prior term.
template <bool EZ = false>
__device__ __forceinline__ float ucb_score(const uint32_t *nb, int A, int a, bool active, float pbc, float sq,
                                           float mean_q, float discount, int players, float mmax,
                                           float mmin, float delta_max, float parent_vp = 0.0f, int parent_reset = 0,
                                           bool arm = false, float reuse_value = 0.0f)
{
    if (!active) return -INFINITY;
    int vis = (int)nb[F_VISIT * A + a];
    float prior = u2f(nb[F_PRIOR * A + a]);
    float pb_c = __fmul_rn(pbc, __fdiv_rn(sq, (float)(vis + 1)));
    float prior_score = __fmul_rn(pb_c, prior);
    float value_score;
    if (vis == 0) {
        value_score = mean_q;
    } else {
        float rw = u2f(nb[F_REWARD * A + a]);
        if (EZ && parent_reset != 1) rw = __fsub_rn(rw, parent_vp);   // true_reward = child prefix - parent prefix
        float v = arm ? reuse_value : __fdiv_rn(u2f(nb[F_VSUM * A + a]), (float)vis);
        value_score = __fadd_rn(rw, __fmul_rn(discount, players == 1 ? v : -v));
    }
    value_score = mm_normalize(value_score, mmax, mmin, delta_max);
    if (value_score < 0.0f) value_score = 0.0f;
    if (value_score > 1.0f) value_score = 1.0f;
    if (arm && vis != 0) return value_score;
    return __fadd_rn(prior_score, value_score);
}

// One PUCT descent of tree b by the calling warp: cbatch_traverse body (cnode.cpp:783-824) with
// compute_mean_q (169-203) and cselect_child (551-595).  Records the path for the backup.
// EZ = true: ctree_efficientzero/lib/cnode.cpp:876-958, 173-210, 651-697 (its rand() tie-break == deterministic for rand() == 0).
// REUSE = true: cbatch_traverse_with_reuse (cnode.cpp:828-932); out_ix gets -1 for "no inference", out_ix_net the same
// slot clamped to >= 0 (what a batched network launch may safely gather).
template <bool EZ = false, bool REUSE = false>
__device__ __forceinline__ void tree_traverse(const TreeParams &p, int b, int lane, int deterministic,
                                              unsigned step, int *out_ix, int *out_iy, int *out_action,
                                              int *out_len, int *out_vtp, const int *true_action = nullptr,
                                              const float *reuse_value = nullptr, int *out_ix_net = nullptr)
{
    const int A = p.A, N = p.N;
    uint32_t *tree_edges = p.edges + (size_t)b * N * kEdgeFields * A;
    const int *lg = p.legal + (size_t)b * A;
    const int nl = p.nlegal[b];
    const int players = (*p.players_max == -1) ? 1 : 2;
    const float discount = p.discount, delta_max = p.delta;
    const float mmax = p.mm_max[b], mmin = p.mm_min[b];
    int *pslot = p.path_slot + (size_t)b * N, *pact = p.path_action + (size_t)b * N;

    int slot = 0, node_visit = p.root_visit[b], plen = 0, last_action = -1;
    int vtp = p.to_play[b];
    bool is_root = true;
    float parent_q = 0.0f;
    float cur_vp = EZ ? p.root_reward[b] : 0.0f;      // value prefix / is_reset of the node being scanned
    int cur_reset = EZ ? p.n_reset[(size_t)b * N] : 0;
    const int ta = REUSE ? true_action[b] : -1;
    const float rv = REUSE ? reuse_value[b] : 0.0f;
    int rstate = 0;

    while (true) {
        const uint32_t *nb = tree_edges + (size_t)slot * kEdgeFields * A;
        const int n = is_root ? nl : A;
        // ---- compute_mean_q: sequential fp32 sum over visited children in legal order
        float total = 0.0f;
        int tv = 0;
        for (int c0 = 0; c0 < n; c0 += 32) {
            int k = c0 + lane;
            bool act = k < n;
            int a = act ? (is_root ? lg[k] : k) : 0;
            int vis = act ? (int)nb[F_VISIT * A + a] : 0;
            float q = 0.0f;
            if (vis > 0) {
                float v = __fdiv_rn(u2f(nb[F_VSUM * A + a]), (float)vis);
                float rw = u2f(nb[F_REWARD * A + a]);
                if (EZ && cur_reset != 1) rw = __fsub_rn(rw, cur_vp);
                q = __fadd_rn(rw, __fmul_rn(discount, v));
            }
            unsigned m = __ballot_sync(0xffffffffu, vis > 0);
            while (m) {
                int l = __ffs(m) - 1;
                m &= m - 1;
                total = __fadd_rn(total, __shfl_sync(0xffffffffu, q, l));
                ++tv;
            }
        }
        float mean_q;
        if (is_root && tv > 0) mean_q = __fdiv_rn(total, (float)tv);
        else mean_q = __fdiv_rn(__fadd_rn(parent_q, total), (float)(tv + 1));

        // ---- cselect_child: first legal position attaining the exact maximum
        const float total_children = (float)(node_visit - 1);   // cnode.cpp:574
        const float pbc = p.pbc[node_visit - 1];
        const float sq = __fsqrt_rn(total_children);
        float best = kFloatMin;
        int best_k = -1;
        for (int c0 = 0; c0 < n; c0 += 32) {
            int k = c0 + lane;
            bool act = k < n;
            int a = act ? (is_root ? lg[k] : k) : 0;
            float sc = ucb_score<EZ>(nb, A, a, act, pbc, sq, mean_q, discount, players, mmax, mmin, delta_max, cur_vp, cur_reset,
                                     REUSE && is_root && a == ta, rv);
            float cmax = warp_max_exact(sc);
            if (best < cmax) {
                best = cmax;
                best_k = c0 + __ffs(__ballot_sync(0xffffffffu, act && sc == cmax)) - 1;
            }
        }
        if (!deterministic && best_k >= 0) {
            // tie list of cnode.cpp:576-586: the arg-max position, then every LATER position whose
            // score >= max - 1e-6; draw uniformly (counter-based hash instead of rand()).
            const float thr = __fsub_rn(best, 0.000001f);
            int count = 1;
            for (int c0 = 0; c0 < n; c0 += 32) {
                int k = c0 + lane;
                bool act = k < n;
                int a = act ? (is_root ? lg[k] : k) : 0;
                float sc = ucb_score<EZ>(nb, A, a, act, pbc, sq, mean_q, discount, players, mmax, mmin, delta_max, cur_vp, cur_reset,
                                     REUSE && is_root && a == ta, rv);
                count += __popc(__ballot_sync(0xffffffffu, act && k > best_k && sc >= thr));
            }
            if (count > 1) {
                unsigned long long h = mix64(p.rng_seed ^ mix64(*p.rng_epoch) ^ mix64(((unsigned long long)b << 32) | step) ^ (unsigned)plen);
                int r = (int)(h % (unsigned)count);
                if (r > 0) {
                    int seen = 0, pick = best_k;
                    for (int c0 = 0; c0 < n; c0 += 32) {
                        int k = c0 + lane;
                        bool act = k < n;
                        int a = act ? (is_root ? lg[k] : k) : 0;
                        float sc = ucb_score<EZ>(nb, A, a, act, pbc, sq, mean_q, discount, players, mmax, mmin, delta_max, cur_vp, cur_reset,
                                     REUSE && is_root && a == ta, rv);
                        unsigned m = __ballot_sync(0xffffffffu, act && k > best_k && sc >= thr);
                        int c = __popc(m);
                        if (seen < r && r <= seen + c) {
                            int want = r - seen;   // want-th set bit (1-based)
                            unsigned mm2 = m;
                            for (int j = 1; j < want; ++j) mm2 &= mm2 - 1;
                            pick = c0 + __ffs(mm2) - 1;
                        }
                        seen += c;
                    }
                    best_k = pick;
                }
            }
        }
        int action = 0;
        if (best_k >= 0) action = is_root ? lg[best_k] : best_k;
        if (players > 1) vtp = (vtp == 1) ? 2 : 1;   // cnode.cpp:798-805

        if (lane == 0) {
            p.n_best[(size_t)b * N + slot] = action;   // cnode.cpp:807
            pslot[plen] = slot;
            pact[plen] = action;
        }
        ++plen;
        last_action = action;
        node_visit = (int)nb[F_VISIT * A + action];
        int cs = (int)nb[F_CSLOT * A + action];
        if (REUSE && is_root && action == ta) {      // cnode.cpp:899-902: stop right after the root
            rstate = cs >= 0 ? 2 : 1;
            break;
        }
        is_root = false;
        parent_q = mean_q;
        if (cs < 0 || plen >= N) break;
        if (EZ) { cur_vp = u2f(nb[F_REWARD * A + action]); cur_reset = p.n_reset[(size_t)b * N + cs]; }
        slot = cs;
    }
    if (lane == 0) {
        p.path_len[b] = plen;
        p.vtp[b] = vtp;
        p.search_len[b] = plen;
        if (out_ix) out_ix[b] = (REUSE && rstate == 2) ? -1 : slot;     // parent of the leaf: its slot == current_latent_state_index
        if (out_ix_net) out_ix_net[b] = slot;
        if (out_iy) out_iy[b] = (REUSE && rstate != 2) ? p.n_batch[(size_t)b * N + slot] : b;      // batch_index (cnode.cpp:907-923)
        if (REUSE) {
            p.reuse_state[b] = rstate;
            if (rstate != 2 && p.infer_count) atomicAdd(p.infer_count + step % (unsigned)N, 1);
        }
        if (out_action) out_action[b] = last_action;
        if (out_len) out_len[b] = plen;
        if (out_vtp) out_vtp[b] = vtp;
    }
    __syncwarp();
}

// CNode::expand (cnode.cpp:83-147) of node block `nb` by the calling warp.  lg == nullptr: all A
// actions in order (inner node); else the root's legal list of length n.
__device__ __forceinline__ void expand_block(uint32_t *nb, int A, const float *logits, const int *lg, int n, int lane)
{
    for (int a = lane; a < A; a += 32) {   // children that are never created have no statistics
        nb[F_PRIOR * A + a] = f2u(0.0f);
        nb[F_VSUM * A + a] = f2u(0.0f);
        nb[F_REWARD * A + a] = f2u(0.0f);
        nb[F_VISIT * A + a] = 0u;
        nb[F_CSLOT * A + a] = (uint32_t)-1;
    }
    __syncwarp();
    float pmax = kFloatMin;                // cnode.cpp:118-125 (running max from FLOAT_MIN)
    for (int c0 = 0; c0 < n; c0 += 32) {
        int k = c0 + lane;
        float l = -INFINITY;
        if (k < n) l = logits[lg ? lg[k] : k];
        pmax = fmaxf(pmax, warp_max_exact(l));
    }
    float sum = 0.0f;                      // cnode.cpp:127-132 sequential in legal order
    for (int c0 = 0; c0 < n; c0 += 32) {
        int k = c0 + lane;
        float e = 0.0f;
        if (k < n) e = lz_expf_exact(__fsub_rn(logits[lg ? lg[k] : k], pmax));
        int cnt = min(32, n - c0);
        for (int l = 0; l < cnt; ++l) sum = __fadd_rn(sum, __shfl_sync(0xffffffffu, e, l));
    }
    for (int c0 = 0; c0 < n; c0 += 32) {   // cnode.cpp:135-140
        int k = c0 + lane;
        if (k < n) {
            int a = lg ? lg[k] : k;
            float e = lz_expf_exact(__fsub_rn(logits[a], pmax));
            nb[F_PRIOR * A + a] = f2u(__fdiv_rn(e, sum));
        }
    }
}

// cbatch_backpropagate body for tree b (cnode.cpp:495-499): expand the leaf reached by the last
// traverse into slot `latent_index`, then cbackpropagate (cnode.cpp:419-478) along the recorded path.
// EZ = true: ctree_efficientzero/lib/cnode.cpp:577-601 + 482-575; `reward` is the value prefix, `leaf_reset` the leaf's is_reset.
// REUSE = true: cbatch_backpropagate_with_reuse (cnode.cpp:502-549) driven by the state the last traverse left: state 2 backs
// up `reuse_value` without expanding anything, state 1 expands but backs up `reuse_value`; batch_rank = the compact row of
// this tree in the inference batch (recorded as the new node's batch_index).
template <bool EZ = false, bool REUSE = false>
__device__ __forceinline__ void tree_backprop(const TreeParams &p, int b, int lane, int latent_index,
                                              float reward, float value, const float *logits,
                                              const int *to_play_override, int leaf_reset = 0, float reuse_value = 0.0f,
                                              int batch_rank = -1)
{
    const int A = p.A, N = p.N;
    const int plen = p.path_len[b];
    if (plen == 0 || latent_index >= N) return;
    uint32_t *tree_edges = p.edges + (size_t)b * N * kEdgeFields * A;
    const int *pslot = p.path_slot + (size_t)b * N, *pact = p.path_action + (size_t)b * N;
    const int tp = to_play_override ? to_play_override[b] : p.vtp[b];
    const float discount = p.discount;

    const int rstate = REUSE ? p.reuse_state[b] : 0;
    const bool no_expand = REUSE && rstate == 2;
    if (REUSE && rstate != 0) value = reuse_value;
    if (!no_expand) expand_block(tree_edges + (size_t)latent_index * kEdgeFields * A, A, logits, nullptr, A, lane);
    const int leaf_ps = pslot[plen - 1], leaf_pa = pact[plen - 1];
    uint32_t *leaf_nb = tree_edges + (size_t)leaf_ps * kEdgeFields * A;
    if (EZ && no_expand && lane == 0)      // ctree_efficientzero cnode.cpp:646: is_reset lands on the reached node even without expansion
        p.n_reset[(size_t)b * N + (int)leaf_nb[F_CSLOT * A + leaf_pa]] = leaf_reset;
    if (lane == 0 && !no_expand) {
        p.n_batch[(size_t)b * N + latent_index] = (REUSE && batch_rank >= 0) ? batch_rank : b;
        p.n_to_play[(size_t)b * N + latent_index] = tp;
        p.n_best[(size_t)b * N + latent_index] = -1;
        if (EZ) p.n_reset[(size_t)b * N + latent_index] = leaf_reset;
        leaf_nb[F_CSLOT * A + leaf_pa] = (uint32_t)latent_index;
        leaf_nb[F_REWARD * A + leaf_pa] = f2u(reward);
    }

    float mmax = p.mm_max[b], mmin = p.mm_min[b];
    float G = value;   // bootstrap_value
    // path nodes i = plen (leaf) ... 0 (root); node i>=1 hangs on edge (pslot[i-1], pact[i-1]).
    for (int hi = plen; hi >= 0; hi -= 32) {
        const int i = hi - lane;
        const bool act = i >= 0;
        float vs = 0.0f, rw = 0.0f, pvp = 0.0f;     // pvp / prs: value prefix and is_reset of the PARENT path node (EZ)
        int vc = 0, ntp = 0, prs = 0;
        uint32_t *enb = nullptr;
        int ea = 0;
        if (EZ && act && i >= 1) {
            pvp = (i == 1) ? p.root_reward[b] : u2f(tree_edges[(size_t)pslot[i - 2] * kEdgeFields * A + F_REWARD * A + pact[i - 2]]);
            prs = p.n_reset[(size_t)b * N + pslot[i - 1]];
        }
        if (act) {
            if (i == plen && !no_expand) { // the leaf: unvisited edge, reward just predicted
                rw = reward; ntp = tp;
                enb = leaf_nb; ea = leaf_pa;
            } else if (i == 0) {
                vs = p.root_vsum[b]; vc = p.root_visit[b]; rw = p.root_reward[b];
                ntp = p.n_to_play[(size_t)b * N];
            } else {
                enb = tree_edges + (size_t)pslot[i - 1] * kEdgeFields * A;
                ea = pact[i - 1];
                vs = u2f(enb[F_VSUM * A + ea]);
                vc = (int)enb[F_VISIT * A + ea];
                rw = u2f(enb[F_REWARD * A + ea]);
                // node i's own slot: recorded on the path, or (reuse stop on an expanded child) the child slot of the last edge
                ntp = p.n_to_play[(size_t)b * N + (i == plen ? (int)enb[F_CSLOT * A + ea] : pslot[i])];
            }
        }
        const int cnt = min(32, hi + 1);
        float my_vs = vs;
        int my_vc = vc;
        for (int l = 0; l < cnt; ++l) {
            float vs_l = __shfl_sync(0xffffffffu, vs, l);
            int vc_l = __shfl_sync(0xffffffffu, vc, l);
            float rw_l = __shfl_sync(0xffffffffu, rw, l);
            int ntp_l = __shfl_sync(0xffffffffu, ntp, l);
            float nvs, upd;
            if (EZ) {                      // ctree_efficientzero cnode.cpp:496-573
                const float pvp_l = __shfl_sync(0xffffffffu, pvp, l);
                const int prs_l = __shfl_sync(0xffffffffu, prs, l);
                const bool same = (tp == -1) || (ntp_l == tp);
                nvs = __fadd_rn(vs_l, same ? G : -G);
                const float nodeval = __fdiv_rn(nvs, (float)(vc_l + 1));
                float true_reward = __fsub_rn(rw_l, pvp_l);
                upd = __fadd_rn(true_reward, __fmul_rn(discount, nodeval));   // MinMax sees the un-reset difference and +value
                if (prs_l == 1) true_reward = rw_l;
                if (tp == -1) G = __fadd_rn(true_reward, __fmul_rn(discount, G));
                else G = same ? __fadd_rn(-true_reward, __fmul_rn(discount, G)) : __fadd_rn(true_reward, __fmul_rn(discount, G));
            } else if (tp == -1) {         // cnode.cpp:432-449
                nvs = __fadd_rn(vs_l, G);
                float nodeval = __fdiv_rn(nvs, (float)(vc_l + 1));
                upd = __fadd_rn(rw_l, __fmul_rn(discount, nodeval));
                G = __fadd_rn(rw_l, __fmul_rn(discount, G));
            } else {                       // cnode.cpp:450-477
                bool same = (ntp_l == tp);
                nvs = __fadd_rn(vs_l, same ? G : -G);
                float nodeval = __fdiv_rn(nvs, (float)(vc_l + 1));
                upd = __fadd_rn(rw_l, __fmul_rn(discount, -nodeval));
                G = same ? __fadd_rn(-rw_l, __fmul_rn(discount, G)) : __fadd_rn(rw_l, __fmul_rn(discount, G));
            }
            if (upd > mmax) mmax = upd;    // cminimax.cpp:19-26
            if (upd < mmin) mmin = upd;
            if (lane == l) { my_vs = nvs; my_vc = vc_l + 1; }
        }
        if (act) {
            if (i == 0) {
                p.root_vsum[b] = my_vs;
                p.root_visit[b] = my_vc;
            } else {
                enb[F_VSUM * A + ea] = f2u(my_vs);
                enb[F_VISIT * A + ea] = (uint32_t)my_vc;
            }
        }
    }
    if (lane == 0) {
        p.mm_max[b] = mmax;
        p.mm_min[b] = mmin;
    }
    __syncwarp();
}

// Gumbel MuZero mode (ctree_gumbel_muzero, gumbel.cu).  Allocated by lz_tree_set_gumbel only, so the MuZero / EfficientZero
// layouts and kernels are untouched; the descent and back-up reuse the node blocks, path storage and expand_block above.
struct GumbelParams {
    int S, m;                    // num_simulations, max_num_considered_actions
    float *raw_value;            // [B][N] value the node was expanded with (the root's from prepare)
    const float *gumbel;         // [A] 10 * extreme_value(0, 1) draws of std::mt19937(0); a root uses its first nlegal entries
    const int *visit_row;        // [S] get_sequence_of_considered_visits(min(m, S), S)
    const int *minus_one;        // [B] all -1: the back-up's to_play (no two-player sign flip, cnode.cpp:605-631)
};

}  // namespace lz

// ---- internal C++ launch API shared by tree.cu and search.cu ----
struct lz_tree {
    lz::TreeParams p;
    float *d_pbc;
    int max_sims;
    unsigned step_counter;
    bool params_set, prepared;
    unsigned long long generation;   // bumped whenever TreeParams values that captured graphs bake in change (set_params / set_ez)
    bool pdl;                    // launch tree kernels with programmatic stream serialization (set by the search graph)
    void *alloc_base;
    // Gumbel mode (lz_tree_set_gumbel): device tables + the number of traverses since the last prepare (checked on the host)
    bool gumbel;
    lz::GumbelParams gp;
    void *gumbel_alloc;
    int gumbel_traversals;
};

namespace lz {
int tree_launch_traverse(lz_tree *t, int deterministic, int32_t *d_ix, int32_t *d_iy, int32_t *d_action,
                         int32_t *d_len, int32_t *d_vtp, cudaStream_t s, int32_t *d_is_reset = nullptr);
int tree_launch_backprop(lz_tree *t, int latent_index, const float *d_reward, const float *d_value,
                         const float *d_logits, const int32_t *d_to_play, cudaStream_t s, const int32_t *d_is_reset = nullptr);
// fused: backup of simulation (latent_index - 1) followed by the descent of the next simulation
int tree_launch_backprop_traverse(lz_tree *t, int latent_index, const float *d_reward, const float *d_value,
                                  const float *d_logits, int deterministic, int32_t *d_ix, int32_t *d_action,
                                  cudaStream_t s, int32_t *d_is_reset = nullptr);
// ReZero reuse variants (MuZero trees): d_ix reports -1 for "no inference", d_ix_net is clamped for the network gather
int tree_launch_traverse_reuse(lz_tree *t, const int32_t *d_true_action, const float *d_reuse_value, int32_t *d_ix, int32_t *d_ix_net,
                               int32_t *d_iy, int32_t *d_action, int32_t *d_len, int32_t *d_vtp, cudaStream_t s, int32_t *d_is_reset = nullptr);
int tree_launch_backprop_reuse(lz_tree *t, int latent_index, const float *d_reward, const float *d_value, const float *d_logits,
                               const float *d_reuse_value, const int32_t *d_batch_rank, const int32_t *d_to_play, cudaStream_t s,
                               const int32_t *d_is_reset = nullptr);
int tree_launch_backprop_traverse_reuse(lz_tree *t, int latent_index, const float *d_reward, const float *d_value, const float *d_logits,
                                        const int32_t *d_true_action, const float *d_reuse_value, int32_t *d_ix_net, int32_t *d_action,
                                        cudaStream_t s);
// Gumbel MuZero (gumbel.cu)
int gumbel_launch_traverse(lz_tree *t, float discount, int32_t *d_ix, int32_t *d_iy, int32_t *d_action, int32_t *d_len,
                           int32_t *d_vtp, cudaStream_t s);
int gumbel_launch_backprop(lz_tree *t, int latent_index, float discount, const float *d_reward, const float *d_value,
                           const float *d_logits, cudaStream_t s);
// fused: backup of simulation (latent_index - 1) followed by the descent of the next simulation
int gumbel_launch_backprop_traverse(lz_tree *t, int latent_index, float discount, const float *d_reward, const float *d_value,
                                    const float *d_logits, int32_t *d_ix, int32_t *d_action, cudaStream_t s);
void gumbel_free(lz_tree *t);
}  // namespace lz
