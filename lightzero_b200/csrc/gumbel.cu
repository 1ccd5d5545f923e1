// gumbel.cu -- Gumbel MuZero search trees (lzero/mcts/ctree/ctree_gumbel_muzero/lib/cnode.cpp, gmz_tree.pyx) on the device
// trees of tree.cuh.  Compiled with -fmad=false, like tree.cu.
//
// The tree is the MuZero tree in Gumbel mode: same node blocks, path storage, expansion (expand_block) and back-up
// (tree_backprop with to_play -1, which is cback_propagate, cnode.cpp:605-631).  What differs is the choice of child:
//   * root (cselect_root_child, cnode.cpp:701-745): sequential halving -- the arg-max of
//     max(-1e9, gumbel + (prior - max prior) + completed_q) + (visits == considered_visit ? 0 : -inf);
//   * interior (cselect_interior_child, :747-790): the arg-max of softmax(prior + completed_q) - N / (1 + sum N);
// with completed_q = qtransform_completed_by_mix_value (:988-1039).  Nothing on this path draws random numbers, so every
// descent reproduces the reference bit for bit.  Conventions (DESIGN.md 4.1): one warp per tree, lane <-> child in chunks
// of 32, every fp32 operation an explicit round-to-nearest intrinsic, order-sensitive sums in the reference's order,
// max / min as exact warp reductions, arg-max as the reference's strict `>` scan (first maximum).
#include <limits.h>
#include <math.h>

#include <algorithm>
#include <random>
#include <vector>

#include "lz_common.cuh"
#include "tree.cuh"

namespace lz {

constexpr int kGmzBlock = 64;          // 2 warps = 2 trees per CTA, as tree.cu
constexpr float kMaxVisitInit = 50.0f; // qtransform_completed_by_mix_value defaults (cnode.h:100-102)
constexpr float kValueScale = 0.1f;
constexpr float kRescaleEps = 1e-8f;

__device__ __forceinline__ float warp_min_exact(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

__device__ __forceinline__ int warp_sum_int(int v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ int warp_max_int(int v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// One child of a node block: the statistics qtransform_completed_by_mix_value reads (get_q, cnode.cpp:181-197).
struct GmzChild {
    float prior, q;
    int visit;
};

__device__ __forceinline__ GmzChild gmz_child(const uint32_t *nb, int A, int a, float discount)
{
    GmzChild c;
    c.prior = u2f(nb[F_PRIOR * A + a]);
    c.visit = (int)nb[F_VISIT * A + a];
    const float v = c.visit == 0 ? 0.0f : __fdiv_rn(u2f(nb[F_VSUM * A + a]), (float)c.visit);   // CNode::value
    c.q = __fadd_rn(u2f(nb[F_REWARD * A + a]), __fmul_rn(discount, v));
    return c;
}

// Node-level terms of qtransform_completed_by_mix_value for the n children of block nb (legal list lg, or action ids 0..n-1
// when lg == nullptr).  The same in every lane.
struct GmzNode {
    float prior_max;      // max prior (score_considered's max logit)
    float lsm_max, lsm_log;   // softmax of the priors: max and logf(sum expf(p - max))
    float mixed;          // compute_mixed_value
    float cq_min, gap, visit_scale;
    int nsum;             // sum of child visits
};

__device__ __forceinline__ GmzNode gmz_node(const uint32_t *nb, int A, const int *lg, int n, float raw_value, float discount,
                                            int lane)
{
    GmzNode s;
    float pmax = -INFINITY;
    int nsum = 0, vmax = INT_MIN;
    for (int c0 = 0; c0 < n; c0 += 32) {
        const int k = c0 + lane;
        float p = -INFINITY;
        int v = 0, vm = INT_MIN;
        if (k < n) {
            const GmzChild c = gmz_child(nb, A, lg ? lg[k] : k, discount);
            p = c.prior; v = c.visit; vm = c.visit;
        }
        pmax = fmaxf(pmax, warp_max_exact(p));
        nsum += warp_sum_int(v);
        vmax = max(vmax, warp_max_int(vm));
    }
    s.prior_max = pmax;
    s.nsum = nsum;
    // csoftmax of the priors (cnode.cpp:903-932): running max from element 0 (== the exact max), sum of expf(p - m) in order
    float sum = 0.0f;
    for (int c0 = 0; c0 < n; c0 += 32) {
        const int k = c0 + lane;
        float e = 0.0f;
        if (k < n) e = lz_expf_exact(__fsub_rn(u2f(nb[F_PRIOR * A + (lg ? lg[k] : k)]), pmax));
        const int cnt = min(32, n - c0);
        for (int l = 0; l < cnt; ++l) sum = __fadd_rn(sum, __shfl_sync(0xffffffffu, e, l));
    }
    s.lsm_max = pmax;
    s.lsm_log = lz_logf_exact(sum);
    // compute_mixed_value (cnode.cpp:934-969) over the visited children in order: probs_sum, then sum of (p * q) / probs_sum
    float probs_sum = 0.0f;
    for (int c0 = 0; c0 < n; c0 += 32) {
        const int k = c0 + lane;
        float sp = 0.0f;
        bool vis = false;
        if (k < n) {
            const GmzChild c = gmz_child(nb, A, lg ? lg[k] : k, discount);
            vis = c.visit > 0;
            sp = lz_expf_exact(__fsub_rn(__fsub_rn(c.prior, pmax), s.lsm_log));
            if (sp < -10e7f) sp = -10e7f;                 // std::max(prior, -10e7)
        }
        unsigned m = __ballot_sync(0xffffffffu, vis);
        while (m) {
            const int l = __ffs(m) - 1;
            m &= m - 1;
            probs_sum = __fadd_rn(probs_sum, __shfl_sync(0xffffffffu, sp, l));
        }
    }
    float wq = 0.0f;
    for (int c0 = 0; c0 < n; c0 += 32) {
        const int k = c0 + lane;
        float term = 0.0f;
        bool vis = false;
        if (k < n) {
            const GmzChild c = gmz_child(nb, A, lg ? lg[k] : k, discount);
            vis = c.visit > 0;
            float sp = lz_expf_exact(__fsub_rn(__fsub_rn(c.prior, pmax), s.lsm_log));
            if (sp < -10e7f) sp = -10e7f;
            term = __fdiv_rn(__fmul_rn(sp, c.q), probs_sum);
        }
        unsigned m = __ballot_sync(0xffffffffu, vis);
        while (m) {
            const int l = __ffs(m) - 1;
            m &= m - 1;
            wq = __fadd_rn(wq, __shfl_sync(0xffffffffu, term, l));
        }
    }
    const float nsf = (float)nsum;                        // float visit_count_sum: exact integer sum below 2^24
    s.mixed = __fdiv_rn(__fadd_rn(raw_value, __fmul_rn(nsf, wq)), __fadd_rn(nsf, 1.0f));
    // completed values: q of visited children, the mixed value elsewhere; rescale_qvalues (cnode.cpp:971-986)
    float cmax = -INFINITY, cmin = INFINITY;
    for (int c0 = 0; c0 < n; c0 += 32) {
        const int k = c0 + lane;
        float hi = -INFINITY, lo = INFINITY;
        if (k < n) {
            const GmzChild c = gmz_child(nb, A, lg ? lg[k] : k, discount);
            hi = lo = c.visit > 0 ? c.q : s.mixed;
        }
        cmax = fmaxf(cmax, warp_max_exact(hi));
        cmin = fminf(cmin, warp_min_exact(lo));
    }
    float gap = __fsub_rn(cmax, cmin);
    if (gap < kRescaleEps) gap = kRescaleEps;             // std::max(gap, epsilon)
    s.cq_min = cmin;
    s.gap = gap;
    s.visit_scale = __fadd_rn(kMaxVisitInit, (float)vmax);
    return s;
}

// completed_qvalue of one child after rescaling and the visit scale: (rescaled * (50 + max_visit)) * 0.1
__device__ __forceinline__ float gmz_completed(const GmzNode &s, const GmzChild &c)
{
    const float cq = c.visit > 0 ? c.q : s.mixed;
    return __fmul_rn(__fmul_rn(__fdiv_rn(__fsub_rn(cq, s.cq_min), s.gap), s.visit_scale), kValueScale);
}

// arg-max by the reference's scan: strict `>` from -inf, first maximum, position 0 when every score is -inf (or NaN)
struct GmzArgmax {
    float best = -INFINITY;
    int pos = 0;
    __device__ __forceinline__ void chunk(float sc, bool act, int c0)
    {
        const float m = warp_max_exact(act ? sc : -INFINITY);
        if (m > best) {
            best = m;
            pos = c0 + __ffs(__ballot_sync(0xffffffffu, act && sc == m)) - 1;
        }
    }
};

// cselect_root_child (cnode.cpp:701-745) -> position in the legal list
__device__ __forceinline__ int gmz_select_root(const uint32_t *nb, int A, const int *lg, int n, const GmzNode &s,
                                               const GumbelParams &g, float discount, int lane)
{
    const int row = min(s.nsum, g.S - 1);              // simulation_index; the host refuses more than S traverses per prepare
    const int considered = g.visit_row[row];
    GmzArgmax am;
    for (int c0 = 0; c0 < n; c0 += 32) {
        const int k = c0 + lane;
        const bool act = k < n;
        float sc = -INFINITY;
        if (act) {
            const GmzChild c = gmz_child(nb, A, lg[k], discount);
            // score_considered (cnode.cpp:1096-1131): the priors stand in for the logits, less their max
            float x = __fadd_rn(__fadd_rn(g.gumbel[k], __fsub_rn(c.prior, s.prior_max)), gmz_completed(s, c));
            if (!(-1e9f < x)) x = -1e9f;                  // std::max(low_logit, x)
            sc = __fadd_rn(x, c.visit == considered ? 0.0f : -INFINITY);
        }
        am.chunk(sc, act, c0);
    }
    return am.pos;
}

// cselect_interior_child (cnode.cpp:747-790) over all A actions -> action id
__device__ __forceinline__ int gmz_select_interior(const uint32_t *nb, int A, const GmzNode &s, float discount, int lane)
{
    float m2 = -INFINITY;
    for (int c0 = 0; c0 < A; c0 += 32) {
        const int a = c0 + lane;
        float pr = -INFINITY;
        if (a < A) {
            const GmzChild c = gmz_child(nb, A, a, discount);
            pr = __fadd_rn(c.prior, gmz_completed(s, c));
        }
        m2 = fmaxf(m2, warp_max_exact(pr));
    }
    float sum = 0.0f;
    for (int c0 = 0; c0 < A; c0 += 32) {
        const int a = c0 + lane;
        float e = 0.0f;
        if (a < A) {
            const GmzChild c = gmz_child(nb, A, a, discount);
            e = lz_expf_exact(__fsub_rn(__fadd_rn(c.prior, gmz_completed(s, c)), m2));
        }
        const int cnt = min(32, A - c0);
        for (int l = 0; l < cnt; ++l) sum = __fadd_rn(sum, __shfl_sync(0xffffffffu, e, l));
    }
    const float lsum = lz_logf_exact(sum);
    const float denom = (float)(1 + s.nsum);
    GmzArgmax am;
    for (int c0 = 0; c0 < A; c0 += 32) {
        const int a = c0 + lane;
        const bool act = a < A;
        float sc = -INFINITY;
        if (act) {
            const GmzChild c = gmz_child(nb, A, a, discount);
            const float pr = lz_expf_exact(__fsub_rn(__fsub_rn(__fadd_rn(c.prior, gmz_completed(s, c)), m2), lsum));
            sc = __fsub_rn(pr, __fdiv_rn((float)c.visit, denom));
        }
        am.chunk(sc, act, c0);
    }
    return am.pos;
}

// cbatch_traverse (cnode.cpp:834-897) for tree b by the calling warp; records the path for tree_backprop
__device__ __forceinline__ void gmz_traverse(const TreeParams &p, const GumbelParams &g, int b, int lane, float discount,
                                             int32_t *out_ix, int32_t *out_iy, int32_t *out_action, int32_t *out_len,
                                             int32_t *out_vtp)
{
    const int A = p.A, N = p.N;
    const uint32_t *tree_edges = p.edges + (size_t)b * N * kEdgeFields * A;
    const int *lg = p.legal + (size_t)b * A;
    const int nl = p.nlegal[b];
    int *pslot = p.path_slot + (size_t)b * N, *pact = p.path_action + (size_t)b * N;
    int slot = 0, plen = 0, action = -1;
    bool is_root = true;
    while (true) {
        const uint32_t *nb = tree_edges + (size_t)slot * kEdgeFields * A;
        const float raw = g.raw_value[(size_t)b * N + slot];
        if (is_root) {
            const GmzNode s = gmz_node(nb, A, lg, nl, raw, discount, lane);
            action = lg[gmz_select_root(nb, A, lg, nl, s, g, discount, lane)];
        } else {
            const GmzNode s = gmz_node(nb, A, nullptr, A, raw, discount, lane);
            action = gmz_select_interior(nb, A, s, discount, lane);
        }
        if (lane == 0) {
            p.n_best[(size_t)b * N + slot] = action;   // node->best_action
            pslot[plen] = slot;
            pact[plen] = action;
        }
        ++plen;
        const int cs = (int)nb[F_CSLOT * A + action];
        is_root = false;
        if (cs < 0 || plen >= N) break;
        slot = cs;
    }
    if (lane == 0) {
        const int vtp = p.to_play[b];                  // virtual_to_play passes through unchanged (:894)
        p.path_len[b] = plen;
        p.search_len[b] = plen;
        p.vtp[b] = vtp;
        if (out_ix) out_ix[b] = slot;                  // the parent's current_latent_state_index (:886-888)
        if (out_iy) out_iy[b] = b;                     // its batch_index
        if (out_action) out_action[b] = action;
        if (out_len) out_len[b] = plen;
        if (out_vtp) out_vtp[b] = vtp;
    }
    __syncwarp();
}

// cbatch_back_propagate (cnode.cpp:633-652): expand the leaf (CNode::expand over all A actions, :94-156) and back up along
// the path.  cback_propagate is tree_backprop's single-player recurrence; the MinMax statistics it also updates are read by
// no Gumbel routine (the reference updates them too, cnode.cpp:627), so they are unobservable.
__device__ __forceinline__ void gmz_backprop(const TreeParams &p, const GumbelParams &g, int b, int lane, int latent_index,
                                             float reward, float value, const float *logits)
{
    if (p.path_len[b] == 0 || latent_index >= p.N) return;
    tree_backprop<false, false>(p, b, lane, latent_index, reward, value, logits, g.minus_one);
    if (lane == 0) g.raw_value[(size_t)b * p.N + latent_index] = value;   // CNode::raw_value
    __syncwarp();
}

__global__ void __launch_bounds__(kGmzBlock)
k_gmz_root_value(TreeParams p, GumbelParams g, const float *values)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < p.B) g.raw_value[(size_t)b * p.N] = values ? values[b] : 0.0f;
}

__global__ void __launch_bounds__(kGmzBlock)
k_gmz_traverse(TreeParams p, GumbelParams g, float discount, int32_t *ix, int32_t *iy, int32_t *act, int32_t *len, int32_t *vtp)
{
    const int b = blockIdx.x * (kGmzBlock / 32) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= p.B) return;
    gmz_traverse(p, g, b, lane, discount, ix, iy, act, len, vtp);
}

__global__ void __launch_bounds__(kGmzBlock)
k_gmz_backprop(TreeParams p, GumbelParams g, int latent_index, const float *reward, const float *value, const float *logits)
{
    const int b = blockIdx.x * (kGmzBlock / 32) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= p.B) return;
    gmz_backprop(p, g, b, lane, latent_index, reward[b], value[b], logits + (size_t)b * p.A);
}

__global__ void __launch_bounds__(kGmzBlock)
k_gmz_backprop_traverse(TreeParams p, GumbelParams g, int latent_index, const float *reward, const float *value,
                        const float *logits, int32_t *ix, int32_t *act)
{
    const int b = blockIdx.x * (kGmzBlock / 32) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= p.B) return;
    gmz_backprop(p, g, b, lane, latent_index, reward[b], value[b], logits + (size_t)b * p.A);
    gmz_traverse(p, g, b, lane, p.discount, ix, nullptr, act, nullptr, nullptr);
}

// get_children_values (cnode.cpp:309-338), get_policies (:355-385) and the collect policy's action
// (gumbel_muzero.py:591-592: np.argmax of the improved policy with illegal entries 0) of every root
__global__ void __launch_bounds__(kGmzBlock)
k_gmz_results(TreeParams p, GumbelParams g, float discount, float *children_values, float *policy, int32_t *action)
{
    const int b = blockIdx.x * (kGmzBlock / 32) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= p.B) return;
    const int A = p.A, N = p.N;
    const uint32_t *nb = p.edges + (size_t)b * N * kEdgeFields * A;      // root block
    const int *lg = p.legal + (size_t)b * A;
    const int n = p.nlegal[b];
    const GmzNode s = gmz_node(nb, A, lg, n, g.raw_value[(size_t)b * N], discount, lane);
    auto legal = [&](int a) { for (int j = 0; j < n; ++j) if (lg[j] == a) return true; return false; };
    // probs[a] = prior + completed_q for legal a, -inf elsewhere; csoftmax over all A entries in action-id order
    float m = -INFINITY;
    for (int c0 = 0; c0 < A; c0 += 32) {
        const int a = c0 + lane;
        float pr = -INFINITY;
        if (a < A && legal(a)) {
            const GmzChild c = gmz_child(nb, A, a, discount);
            const float cq = gmz_completed(s, c);
            pr = __fadd_rn(c.prior, cq);
            if (children_values) children_values[(size_t)b * A + a] = cq;
        } else if (a < A && children_values) {
            children_values[(size_t)b * A + a] = -INFINITY;
        }
        m = fmaxf(m, warp_max_exact(pr));
    }
    if (!policy && !action) return;
    float sum = 0.0f;
    for (int c0 = 0; c0 < A; c0 += 32) {
        const int a = c0 + lane;
        float e = 0.0f;
        if (a < A) {
            float pr = -INFINITY;
            if (legal(a)) { const GmzChild c = gmz_child(nb, A, a, discount); pr = __fadd_rn(c.prior, gmz_completed(s, c)); }
            e = lz_expf_exact(__fsub_rn(pr, m));
        }
        const int cnt = min(32, A - c0);
        for (int l = 0; l < cnt; ++l) sum = __fadd_rn(sum, __shfl_sync(0xffffffffu, e, l));
    }
    const float lsum = lz_logf_exact(sum);
    GmzArgmax am;
    for (int c0 = 0; c0 < A; c0 += 32) {
        const int a = c0 + lane;
        const bool act = a < A;
        float pv = 0.0f;
        if (act) {
            const bool lgl = legal(a);
            float pr = -INFINITY;
            if (lgl) { const GmzChild c = gmz_child(nb, A, a, discount); pr = __fadd_rn(c.prior, gmz_completed(s, c)); }
            pv = lz_expf_exact(__fsub_rn(__fsub_rn(pr, m), lsum));
            if (policy) policy[(size_t)b * A + a] = pv;
            if (!lgl) pv = 0.0f;
        }
        am.chunk(pv, act, c0);
    }
    if (action && lane == 0) action[b] = am.pos;
}

static inline dim3 gmz_grid(int B) { return dim3(ceil_div(B, kGmzBlock / 32)); }

int gumbel_launch_traverse(lz_tree *t, float discount, int32_t *d_ix, int32_t *d_iy, int32_t *d_action, int32_t *d_len,
                           int32_t *d_vtp, cudaStream_t s)
{
    k_gmz_traverse<<<gmz_grid(t->p.B), kGmzBlock, 0, s>>>(t->p, t->gp, discount, d_ix, d_iy, d_action, d_len, d_vtp);
    LZ_KERNEL_CHECK();
    return LZ_OK;
}

int gumbel_launch_backprop(lz_tree *t, int latent_index, float discount, const float *d_reward, const float *d_value,
                           const float *d_logits, cudaStream_t s)
{
    TreeParams p = t->p;
    p.discount = discount;
    k_gmz_backprop<<<gmz_grid(p.B), kGmzBlock, 0, s>>>(p, t->gp, latent_index, d_reward, d_value, d_logits);
    LZ_KERNEL_CHECK();
    return LZ_OK;
}

int gumbel_launch_backprop_traverse(lz_tree *t, int latent_index, float discount, const float *d_reward, const float *d_value,
                                    const float *d_logits, int32_t *d_ix, int32_t *d_action, cudaStream_t s)
{
    TreeParams p = t->p;
    p.discount = discount;       // the back-up's and the next descent's discount are the search's one discount factor
    k_gmz_backprop_traverse<<<gmz_grid(p.B), kGmzBlock, 0, s>>>(p, t->gp, latent_index, d_reward, d_value, d_logits, d_ix, d_action);
    LZ_KERNEL_CHECK();
    return LZ_OK;
}

void gumbel_free(lz_tree *t)
{
    if (t && t->gumbel_alloc) cudaFree(t->gumbel_alloc);
    if (t) { t->gumbel_alloc = nullptr; t->gumbel = false; }
}

// get_sequence_of_considered_visits (cnode.cpp:1041-1076), host-side parameter precomputation
static std::vector<int> considered_visits(int max_num_considered_actions, int num_simulations)
{
    std::vector<int> seq;
    if (max_num_considered_actions <= 1) {
        for (int i = 0; i < num_simulations; ++i) seq.push_back(i);
        return seq;
    }
    const int log2max = (int)std::ceil(std::log2(max_num_considered_actions));
    std::vector<int> visits(max_num_considered_actions, 0);
    int num_considered = max_num_considered_actions;
    while ((int)seq.size() < num_simulations) {
        const int extra = std::max(1, (int)(num_simulations / (log2max * num_considered)));
        for (int i = 0; i < extra; ++i) {
            seq.insert(seq.end(), visits.begin(), visits.begin() + num_considered);
            for (int j = 0; j < num_considered; ++j) visits[j] += 1;
        }
        num_considered = std::max(2, num_considered / 2);
    }
    seq.resize(num_simulations);
    return seq;
}

}  // namespace lz

using namespace lz;

extern "C" {

int lz_tree_set_gumbel(lz_tree *t, int num_simulations, int max_num_considered_actions)
{
    LZ_REQUIRE(t, LZ_EINVAL, "lz_tree_set_gumbel: null tree");
    LZ_REQUIRE(num_simulations > 0 && max_num_considered_actions > 0, LZ_EINVAL,
               "lz_tree_set_gumbel: num_simulations (%d) and max_num_considered_actions (%d) must be > 0", num_simulations,
               max_num_considered_actions);
    LZ_REQUIRE(num_simulations <= t->max_sims, LZ_EINVAL, "lz_tree_set_gumbel: num_simulations %d > tree capacity %d",
               num_simulations, t->max_sims);
    LZ_REQUIRE(!t->p.ez, LZ_ESTATE, "lz_tree_set_gumbel: tree is in EfficientZero mode");
    const int B = t->p.B, A = t->p.A, N = t->p.N;
    if (!t->gumbel_alloc) {      // raw_value [B][N], gumbel [A], visit row [max_sims], minus_one [B]
        uint32_t *base = nullptr;
        const size_t words = (size_t)B * N + A + t->max_sims + B;
        int rc = dev_alloc(&base, words);
        if (rc != LZ_OK) return rc;
        t->gumbel_alloc = base;
        t->gp.raw_value = (float *)base;
        t->gp.gumbel = (const float *)(base + (size_t)B * N);
        t->gp.visit_row = (const int *)(base + (size_t)B * N + A);
        t->gp.minus_one = (const int *)(base + (size_t)B * N + A + t->max_sims);
        LZ_CUDA_CHECK(cudaMemset(base, 0, (size_t)B * N * sizeof(float)));
        LZ_CUDA_CHECK(cudaMemset((void *)t->gp.minus_one, 0xff, (size_t)B * sizeof(int)));
        // generate_gumbel (cnode.cpp:1133-1151) with gumbel_rng = 0, gumbel_scale = 10: every root reseeds, so every root
        // draws the same prefix of this one sequence (the same libstdc++ distribution the reference is compiled with)
        std::mt19937 gen(0u);
        std::extreme_value_distribution<float> d(0, 1);
        const float scale = 10.0f;
        std::vector<float> gum(A);
        for (int i = 0; i < A; ++i) gum[i] = scale * d(gen);
        LZ_CUDA_CHECK(cudaMemcpy((void *)t->gp.gumbel, gum.data(), A * sizeof(float), cudaMemcpyHostToDevice));
    }
    if (t->gp.S != num_simulations || t->gp.m != max_num_considered_actions) {
        // cselect_root_child reads row min(m, S) of get_table_of_considered_visits(m, S) (cnode.cpp:724-729)
        const std::vector<int> row = considered_visits(std::min(max_num_considered_actions, num_simulations), num_simulations);
        LZ_CUDA_CHECK(cudaMemcpy((void *)t->gp.visit_row, row.data(), row.size() * sizeof(int), cudaMemcpyHostToDevice));
        t->gp.S = num_simulations;
        t->gp.m = max_num_considered_actions;
        ++t->generation;         // captured graphs bake GumbelParams in
    }
    t->gumbel = true;
    return LZ_OK;
}

int lz_tree_prepare_gumbel(lz_tree *t, const float *d_logits, const float *d_noise, float noise_weight, const float *d_rewards,
                           const float *d_values, const int32_t *d_to_play, lz_stream s)
{
    LZ_REQUIRE(t && d_logits, LZ_EINVAL, "lz_tree_prepare_gumbel: null argument");
    LZ_REQUIRE(t->gumbel, LZ_ESTATE, "lz_tree_prepare_gumbel: tree is not in Gumbel mode (lz_tree_set_gumbel)");
    // CRoots::prepare / prepare_no_noise (cnode.cpp:418-455) == the MuZero root expansion + noise + visit_count 1, plus raw_value
    int rc = lz_tree_prepare(t, d_logits, d_noise, noise_weight, d_rewards, d_to_play, s);
    if (rc) return rc;
    k_gmz_root_value<<<ceil_div(t->p.B, kGmzBlock), kGmzBlock, 0, (cudaStream_t)s>>>(t->p, t->gp, d_values);
    LZ_KERNEL_CHECK();
    t->gumbel_traversals = 0;
    return LZ_OK;
}

int lz_tree_traverse_gumbel(lz_tree *t, float discount, int32_t *d_ix, int32_t *d_iy, int32_t *d_last_action,
                            int32_t *d_search_len, int32_t *d_virtual_to_play, lz_stream s)
{
    LZ_REQUIRE(t, LZ_EINVAL, "lz_tree_traverse_gumbel: null tree");
    LZ_REQUIRE(t->gumbel, LZ_ESTATE, "lz_tree_traverse_gumbel: tree is not in Gumbel mode (lz_tree_set_gumbel)");
    LZ_REQUIRE(t->prepared, LZ_ESTATE, "lz_tree_traverse_gumbel: roots not prepared (call lz_tree_prepare_gumbel first)");
    LZ_REQUIRE(t->gumbel_traversals < t->gp.S, LZ_ESTATE,
               "lz_tree_traverse_gumbel: %d traverses since prepare already use all num_simulations=%d rows of the considered-visit table",
               t->gumbel_traversals, t->gp.S);
    ++t->gumbel_traversals;
    return gumbel_launch_traverse(t, discount, d_ix, d_iy, d_last_action, d_search_len, d_virtual_to_play, (cudaStream_t)s);
}

int lz_tree_backpropagate_gumbel(lz_tree *t, int latent_index, float discount, const float *d_reward, const float *d_value,
                                 const float *d_logits, lz_stream s)
{
    LZ_REQUIRE(t && d_reward && d_value && d_logits, LZ_EINVAL, "lz_tree_backpropagate_gumbel: null argument");
    LZ_REQUIRE(t->gumbel, LZ_ESTATE, "lz_tree_backpropagate_gumbel: tree is not in Gumbel mode (lz_tree_set_gumbel)");
    LZ_REQUIRE(t->prepared, LZ_ESTATE, "lz_tree_backpropagate_gumbel: roots not prepared");
    LZ_REQUIRE(latent_index >= 1 && latent_index <= t->max_sims, LZ_EINVAL,
               "lz_tree_backpropagate_gumbel: latent_index %d outside [1, %d]", latent_index, t->max_sims);
    return gumbel_launch_backprop(t, latent_index, discount, d_reward, d_value, d_logits, (cudaStream_t)s);
}

int lz_tree_results_gumbel(lz_tree *t, float discount, float *d_children_values, float *d_improved_policy, int32_t *d_action,
                           lz_stream s)
{
    LZ_REQUIRE(t, LZ_EINVAL, "lz_tree_results_gumbel: null tree");
    LZ_REQUIRE(t->gumbel, LZ_ESTATE, "lz_tree_results_gumbel: tree is not in Gumbel mode (lz_tree_set_gumbel)");
    k_gmz_results<<<gmz_grid(t->p.B), kGmzBlock, 0, (cudaStream_t)s>>>(t->p, t->gp, discount, d_children_values,
                                                                       d_improved_policy, d_action);
    LZ_KERNEL_CHECK();
    return LZ_OK;
}

}  // extern "C"
