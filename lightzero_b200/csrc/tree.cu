// tree.cu -- kernels + C ABI for the device-resident batched MuZero trees (see tree.cuh for the design).
// Compiled with -fmad=false: no fp32 contraction anywhere in this translation unit.
#include <math.h>
#include <stdarg.h>

#include <atomic>
#include <limits.h>
#include <vector>

#include "lz_common.cuh"
#include "tree.cuh"
#include "tc_ptx.cuh"

namespace lz {

static thread_local char g_err[512] = "";
static std::atomic<unsigned long long> g_launches{0};
void count_launch(int n) { g_launches.fetch_add((unsigned long long)n, std::memory_order_relaxed); }

void set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

constexpr int kTreeBlock = 64;   // 2 warps = 2 trees per CTA: latency-bound work, spread over all SMs

__global__ void __launch_bounds__(kTreeBlock)
k_tree_reset(TreeParams p, const int32_t *legal, const int32_t *nlegal, const uint8_t *mask)
{
    const int b = blockIdx.x * (kTreeBlock / 32) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        *p.players_max = INT_MIN;
        *p.rng_epoch += 1ull;
    }
    if (b >= p.B) return;
    const int A = p.A;
    int *lg = p.legal + (size_t)b * A;
    int n = 0;
    if (mask) {                              // ascending ids == np.nonzero order (policy/muzero.py:760)
        for (int c0 = 0; c0 < A; c0 += 32) {
            int a = c0 + lane;
            bool on = a < A && mask[(size_t)b * A + a] != 0;
            unsigned m = __ballot_sync(0xffffffffu, on);
            if (on) lg[n + __popc(m & ((1u << lane) - 1u))] = a;
            n += __popc(m);
        }
    } else if (legal && nlegal) {
        n = nlegal[b];
        for (int k = lane; k < n; k += 32) lg[k] = legal[(size_t)b * A + k];
    }
    if (n == 0) {                            // cnode.cpp:101-107: empty list == every action
        n = A;
        for (int k = lane; k < A; k += 32) lg[k] = k;
    }
    for (int k = n + lane; k < A; k += 32) lg[k] = -1;
    if (lane == 0) {
        p.nlegal[b] = n;
        p.root_visit[b] = 0;
        p.root_vsum[b] = 0.0f;
        p.root_reward[b] = 0.0f;
        p.mm_max[b] = kFloatMin;             // cminimax.cpp:7-11
        p.mm_min[b] = kFloatMax;
        p.path_len[b] = 0;
        p.search_len[b] = 0;
        p.n_reset[(size_t)b * p.N] = 0;      // the root is never reset (ctree_efficientzero cnode.cpp:54,75)
        p.n_batch[(size_t)b * p.N] = b;      // root.expand(to_play, 0, i, ...)
        p.reuse_state[b] = 0;
    }
}

// CRoots::prepare / prepare_no_noise (cnode.cpp:321-358)
__global__ void __launch_bounds__(kTreeBlock)
k_tree_prepare(TreeParams p, const float *logits, const float *noise, float noise_w, const float *rewards,
               const int32_t *to_play)
{
    const int b = blockIdx.x * (kTreeBlock / 32) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= p.B) return;
    const int A = p.A, N = p.N;
    uint32_t *nb = p.edges + (size_t)b * N * kEdgeFields * A;   // slot 0
    const int *lg = p.legal + (size_t)b * A;
    const int n = p.nlegal[b];
    expand_block(nb, A, logits + (size_t)b * A, lg, n, lane);
    __syncwarp();
    if (noise) {                             // add_exploration_noise (cnode.cpp:149-167)
        const float keep = __fsub_rn(1.0f, noise_w);
        for (int k = lane; k < n; k += 32) {
            int a = lg[k];
            float prior = u2f(nb[F_PRIOR * A + a]);
            float nz = noise[(size_t)b * A + k];
            nb[F_PRIOR * A + a] = f2u(__fadd_rn(__fmul_rn(prior, keep), __fmul_rn(nz, noise_w)));
        }
    }
    if (lane == 0) {
        const int tp = to_play ? to_play[b] : -1;
        p.to_play[b] = tp;
        p.n_to_play[(size_t)b * N] = tp;
        p.n_best[(size_t)b * N] = -1;
        p.root_reward[b] = rewards ? rewards[b] : 0.0f;
        p.root_visit[b] += 1;                // cnode.cpp:338,356
        p.vtp[b] = tp;
        atomicMax(p.players_max, tp);
    }
}

template <bool EZ>
__global__ void __launch_bounds__(kTreeBlock)
k_tree_traverse(TreeParams p, int deterministic, unsigned step, int32_t *ix, int32_t *iy, int32_t *act,
                int32_t *len, int32_t *vtp, int32_t *is_reset)
{
    const int b = blockIdx.x * (kTreeBlock / 32) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    pdl_launch_dependents();
    pdl_wait();
    if (b >= p.B) return;
    tree_traverse<EZ>(p, b, lane, deterministic, step, ix, iy, act, len, vtp);
    // mcts_ctree.py:856-861: the LSTM state of a leaf is reset every lstm_horizon_len steps of depth
    if (EZ && is_reset && lane == 0) is_reset[b] = (p.search_len[b] % p.lstm_horizon == 0) ? 1 : 0;
}

template <bool EZ>
__global__ void __launch_bounds__(kTreeBlock)
k_tree_backprop(TreeParams p, int latent_index, const float *reward, const float *value, const float *logits,
                const int32_t *to_play, const int32_t *is_reset)
{
    const int b = blockIdx.x * (kTreeBlock / 32) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    pdl_launch_dependents();
    pdl_wait();
    if (b >= p.B) return;
    tree_backprop<EZ>(p, b, lane, latent_index, reward[b], value[b], logits + (size_t)b * p.A, to_play,
                      (EZ && is_reset) ? is_reset[b] : 0);
}

template <bool EZ>
__global__ void __launch_bounds__(kTreeBlock)
k_tree_backprop_traverse(TreeParams p, int latent_index, const float *reward, const float *value,
                         const float *logits, int deterministic, unsigned step, int32_t *ix, int32_t *act, int32_t *is_reset)
{
    const int b = blockIdx.x * (kTreeBlock / 32) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    pdl_launch_dependents();      // lets the next network kernel set up (TMEM, barriers, first weight taps) meanwhile
    pdl_wait();                   // reward / value / logits come from the preceding network kernel
    if (b >= p.B) return;
    tree_backprop<EZ>(p, b, lane, latent_index, reward[b], value[b], logits + (size_t)b * p.A, nullptr,
                      (EZ && is_reset) ? is_reset[b] : 0);
    tree_traverse<EZ>(p, b, lane, deterministic, step, ix, nullptr, act, nullptr, nullptr);
    if (EZ && is_reset && lane == 0) is_reset[b] = (p.search_len[b] % p.lstm_horizon == 0) ? 1 : 0;
}

// ---- ReZero search_with_reuse (MuZero trees) ----
template <bool EZ>
__global__ void __launch_bounds__(kTreeBlock)
k_tree_traverse_reuse(TreeParams p, unsigned step, const int32_t *true_action, const float *reuse_value, int32_t *ix, int32_t *ix_net,
                      int32_t *iy, int32_t *act, int32_t *len, int32_t *vtp, int32_t *is_reset)
{
    const int b = blockIdx.x * (kTreeBlock / 32) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= p.B) return;
    tree_traverse<EZ, true>(p, b, lane, p.tie_first, step, ix, iy, act, len, vtp, true_action, reuse_value, ix_net);
    // EfficientZero, fused search: is_reset of the reached node per TREE (mcts_ctree.py:856-861 / 1040-1046: search_len % lstm_horizon_len)
    if (EZ && is_reset && lane == 0) is_reset[b] = (p.search_len[b] % p.lstm_horizon == 0) ? 1 : 0;
}

template <bool EZ>
__global__ void __launch_bounds__(kTreeBlock)
k_tree_backprop_reuse(TreeParams p, int latent_index, const float *reward, const float *value, const float *logits,
                      const float *reuse_value, const int32_t *batch_rank, const int32_t *to_play, const int32_t *is_reset)
{
    const int b = blockIdx.x * (kTreeBlock / 32) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= p.B) return;
    tree_backprop<EZ, true>(p, b, lane, latent_index, reward[b], value[b], logits + (size_t)b * p.A, to_play,
                            (EZ && is_reset) ? is_reset[b] : 0, reuse_value[b], batch_rank ? batch_rank[b] : -1);
}

__global__ void __launch_bounds__(kTreeBlock)
k_tree_backprop_traverse_reuse(TreeParams p, int latent_index, const float *reward, const float *value, const float *logits,
                               unsigned step, const int32_t *true_action, const float *reuse_value, int32_t *ix_net, int32_t *act)
{
    const int b = blockIdx.x * (kTreeBlock / 32) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= p.B) return;
    tree_backprop<false, true>(p, b, lane, latent_index, reward[b], value[b], logits + (size_t)b * p.A, nullptr, 0, reuse_value[b], -1);
    tree_traverse<false, true>(p, b, lane, p.tie_first, step, nullptr, nullptr, act, nullptr, nullptr, true_action, reuse_value, ix_net);
}

// get_distributions / get_values / get_trajectories (cnode.cpp:237-277,369-417)
__global__ void __launch_bounds__(kTreeBlock)
k_tree_results(TreeParams p, int32_t *visits, float *values, int32_t *nlegal, int32_t *traj)
{
    const int b = blockIdx.x * (kTreeBlock / 32) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= p.B) return;
    const int A = p.A, N = p.N;
    const uint32_t *tree_edges = p.edges + (size_t)b * N * kEdgeFields * A;
    const int n = p.nlegal[b];
    if (visits) {
        for (int k = lane; k < A; k += 32)
            visits[(size_t)b * A + k] = k < n ? (int)tree_edges[F_VISIT * A + p.legal[(size_t)b * A + k]] : -1;
    }
    if (lane == 0) {
        if (values) {
            int vc = p.root_visit[b];
            values[b] = vc == 0 ? 0.0f : __fdiv_rn(p.root_vsum[b], (float)vc);
        }
        if (nlegal) nlegal[b] = n;
    }
    if (traj) {
        for (int k = lane; k < N; k += 32) traj[(size_t)b * N + k] = -1;
        __syncwarp();
        if (lane == 0) {
            int slot = 0, len = 0;
            while (slot >= 0 && len < N) {
                int a = p.n_best[(size_t)b * N + slot];
                if (a < 0) break;
                traj[(size_t)b * N + len++] = a;
                slot = (int)tree_edges[(size_t)slot * kEdgeFields * A + F_CSLOT * A + a];
            }
        }
    }
}

// select_action (lzero/policy/utils.py:637-661) on the root visit counts of every tree: probabilities
// visit ** (1 / temperature) / sum in fp64 like the reference's Python floats, entropy in bits = -sum p ln p / ln 2 (scipy.stats.entropy(p, base=2), policy/utils.py:660),
// action = arg-max (deterministic, first maximum like np.argmax) or an inverse-CDF draw from a counter-based uniform.
__global__ void __launch_bounds__(kTreeBlock)
k_tree_select_action(TreeParams p, double inv_temperature, int deterministic, unsigned long long seed,
                     int32_t *action, int32_t *action_pos, float *entropy)
{
    const int b = blockIdx.x * (kTreeBlock / 32) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= p.B) return;
    const int A = p.A, n = p.nlegal[b];
    const uint32_t *nb = p.edges + (size_t)b * p.N * kEdgeFields * A;      // root block
    const int *lg = p.legal + (size_t)b * A;
    double total = 0.0;
    for (int k = lane; k < n; k += 32) total += pow((double)(int)nb[F_VISIT * A + lg[k]], inv_temperature);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) total += __shfl_xor_sync(0xffffffffu, total, o);
    double ent = 0.0;
    for (int k = lane; k < n; k += 32) {
        const double pr = pow((double)(int)nb[F_VISIT * A + lg[k]], inv_temperature) / total;
        if (pr > 0.0) ent -= pr * log(pr);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ent += __shfl_xor_sync(0xffffffffu, ent, o);
    if (lane == 0) {
        int pos = 0;
        if (deterministic) {
            int best = -1;
            for (int k = 0; k < n; ++k) { int v = (int)nb[F_VISIT * A + lg[k]]; if (v > best) { best = v; pos = k; } }
        } else {
            const unsigned long long h = mix64(seed ^ mix64((unsigned long long)b + 0x1234567ull));
            const double u = (double)(h >> 11) * (1.0 / 9007199254740992.0);       // uniform [0, 1)
            double cum = 0.0;
            pos = n - 1;
            for (int k = 0; k < n; ++k) {
                cum += pow((double)(int)nb[F_VISIT * A + lg[k]], inv_temperature) / total;
                if (u < cum) { pos = k; break; }
            }
        }
        if (action_pos) action_pos[b] = pos;
        if (action) action[b] = lg[pos];            // np.where(action_mask == 1)[0][pos], policy/muzero.py:800
        if (entropy) entropy[b] = (float)(ent / 0.69314718055994530942);    // base 2, as scipy divides the natural-log entropy by ln 2
    }
}

static inline dim3 tree_grid(int B) { return dim3(ceil_div(B, kTreeBlock / 32)); }

template <typename... KArgs, typename... Args>
static cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, cudaStream_t s, bool pdl, Args... args)
{
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = grid; cfg.blockDim = dim3(kTreeBlock); cfg.dynamicSmemBytes = 0; cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = pdl ? 1 : 0;
    cfg.attrs = attr; cfg.numAttrs = 1;
    count_launch();
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

int tree_launch_traverse(lz_tree *t, int deterministic, int32_t *d_ix, int32_t *d_iy, int32_t *d_action,
                         int32_t *d_len, int32_t *d_vtp, cudaStream_t s, int32_t *d_is_reset)
{
    if (t->p.ez)
        LZ_CUDA_CHECK(launch_pdl(k_tree_traverse<true>, tree_grid(t->p.B), s, t->pdl, t->p, deterministic, t->step_counter++, d_ix, d_iy,
                                 d_action, d_len, d_vtp, d_is_reset));
    else
        LZ_CUDA_CHECK(launch_pdl(k_tree_traverse<false>, tree_grid(t->p.B), s, t->pdl, t->p, deterministic, t->step_counter++, d_ix, d_iy,
                                 d_action, d_len, d_vtp, d_is_reset));
    return LZ_OK;
}

int tree_launch_backprop(lz_tree *t, int latent_index, const float *d_reward, const float *d_value,
                         const float *d_logits, const int32_t *d_to_play, cudaStream_t s, const int32_t *d_is_reset)
{
    if (t->p.ez)
        LZ_CUDA_CHECK(launch_pdl(k_tree_backprop<true>, tree_grid(t->p.B), s, t->pdl, t->p, latent_index, d_reward, d_value, d_logits,
                                 d_to_play, d_is_reset));
    else
        LZ_CUDA_CHECK(launch_pdl(k_tree_backprop<false>, tree_grid(t->p.B), s, t->pdl, t->p, latent_index, d_reward, d_value, d_logits,
                                 d_to_play, d_is_reset));
    return LZ_OK;
}

int tree_launch_backprop_traverse(lz_tree *t, int latent_index, const float *d_reward, const float *d_value,
                                  const float *d_logits, int deterministic, int32_t *d_ix, int32_t *d_action,
                                  cudaStream_t s, int32_t *d_is_reset)
{
    if (t->p.ez)
        LZ_CUDA_CHECK(launch_pdl(k_tree_backprop_traverse<true>, tree_grid(t->p.B), s, t->pdl, t->p, latent_index, d_reward, d_value,
                                 d_logits, deterministic, t->step_counter++, d_ix, d_action, d_is_reset));
    else
        LZ_CUDA_CHECK(launch_pdl(k_tree_backprop_traverse<false>, tree_grid(t->p.B), s, t->pdl, t->p, latent_index, d_reward, d_value,
                                 d_logits, deterministic, t->step_counter++, d_ix, d_action, d_is_reset));
    return LZ_OK;
}

int tree_launch_traverse_reuse(lz_tree *t, const int32_t *d_true_action, const float *d_reuse_value, int32_t *d_ix, int32_t *d_ix_net,
                               int32_t *d_iy, int32_t *d_action, int32_t *d_len, int32_t *d_vtp, cudaStream_t s, int32_t *d_is_reset)
{
    if (t->p.ez)
        k_tree_traverse_reuse<true><<<tree_grid(t->p.B), kTreeBlock, 0, s>>>(t->p, t->step_counter++, d_true_action, d_reuse_value, d_ix, d_ix_net,
                                                                            d_iy, d_action, d_len, d_vtp, d_is_reset);
    else
        k_tree_traverse_reuse<false><<<tree_grid(t->p.B), kTreeBlock, 0, s>>>(t->p, t->step_counter++, d_true_action, d_reuse_value, d_ix, d_ix_net,
                                                                             d_iy, d_action, d_len, d_vtp, nullptr);
    LZ_KERNEL_CHECK();
    return LZ_OK;
}

int tree_launch_backprop_reuse(lz_tree *t, int latent_index, const float *d_reward, const float *d_value, const float *d_logits,
                               const float *d_reuse_value, const int32_t *d_batch_rank, const int32_t *d_to_play, cudaStream_t s,
                               const int32_t *d_is_reset)
{
    if (t->p.ez)
        k_tree_backprop_reuse<true><<<tree_grid(t->p.B), kTreeBlock, 0, s>>>(t->p, latent_index, d_reward, d_value, d_logits, d_reuse_value,
                                                                            d_batch_rank, d_to_play, d_is_reset);
    else
        k_tree_backprop_reuse<false><<<tree_grid(t->p.B), kTreeBlock, 0, s>>>(t->p, latent_index, d_reward, d_value, d_logits, d_reuse_value,
                                                                             d_batch_rank, d_to_play, d_is_reset);
    LZ_KERNEL_CHECK();
    return LZ_OK;
}

int tree_launch_backprop_traverse_reuse(lz_tree *t, int latent_index, const float *d_reward, const float *d_value, const float *d_logits,
                                        const int32_t *d_true_action, const float *d_reuse_value, int32_t *d_ix_net, int32_t *d_action,
                                        cudaStream_t s)
{
    k_tree_backprop_traverse_reuse<<<tree_grid(t->p.B), kTreeBlock, 0, s>>>(t->p, latent_index, d_reward, d_value, d_logits,
                                                                           t->step_counter++, d_true_action, d_reuse_value, d_ix_net, d_action);
    LZ_KERNEL_CHECK();
    return LZ_OK;
}

}  // namespace lz

using namespace lz;

extern "C" {

int lz_version(void) { return 200; }
unsigned long long lz_debug_launch_count(void) { return lz::g_launches.load(std::memory_order_relaxed); }
const char *lz_last_error(void) { return lz::g_err; }

int lz_tree_create(int B, int A, int max_sims, lz_tree **out)
{
    LZ_REQUIRE(out && B > 0 && A > 0 && max_sims > 0, LZ_EINVAL, "lz_tree_create: bad arguments B=%d A=%d max_sims=%d", B, A, max_sims);
    int ndev = 0;
    LZ_CUDA_CHECK(cudaGetDeviceCount(&ndev));
    LZ_REQUIRE(ndev > 0, LZ_ECUDA, "lz_tree_create: no CUDA device (this library has no CPU fallback)");
    lz_tree *t = new lz_tree();
    memset(t, 0, sizeof(*t));
    const int N = max_sims + 1;
    TreeParams &p = t->p;
    p.B = B; p.A = A; p.N = N;
    t->max_sims = max_sims;
    // one allocation, carved
    size_t words = 0;
    auto take = [&](size_t n) { size_t o = words; words += (n + 31) & ~(size_t)31; return o; };
    size_t o_edges = take((size_t)B * N * kEdgeFields * A);
    size_t o_ntp = take((size_t)B * N), o_nbest = take((size_t)B * N), o_nreset = take((size_t)B * N), o_nbatch = take((size_t)B * N);
    size_t o_rstate = take(B), o_infer = take(N);
    size_t o_legal = take((size_t)B * A), o_nlegal = take(B);
    size_t o_rvis = take(B), o_rvsum = take(B), o_rrew = take(B), o_mmax = take(B), o_mmin = take(B);
    size_t o_tp = take(B), o_players = take(1), o_pslot = take((size_t)B * N), o_pact = take((size_t)B * N);
    size_t o_plen = take(B), o_vtp = take(B), o_slen = take(B), o_pbc = take(N + 1), o_epoch = take(2);
    uint32_t *base = nullptr;
    int rc = dev_alloc(&base, words);
    if (rc != LZ_OK) { delete t; return rc; }
    cudaError_t e = cudaMemset(base, 0, words * 4);
    if (e != cudaSuccess) { set_error("cudaMemset failed: %s", cudaGetErrorString(e)); cudaFree(base); delete t; return LZ_ECUDA; }
    t->alloc_base = base;
    p.edges = base + o_edges;
    p.n_to_play = (int *)(base + o_ntp); p.n_best = (int *)(base + o_nbest); p.n_reset = (int *)(base + o_nreset);
    p.n_batch = (int *)(base + o_nbatch); p.reuse_state = (int *)(base + o_rstate); p.infer_count = (int *)(base + o_infer);
    p.ez = 0; p.lstm_horizon = 5; p.tie_first = 1;
    p.legal = (int *)(base + o_legal); p.nlegal = (int *)(base + o_nlegal);
    p.root_visit = (int *)(base + o_rvis); p.root_vsum = (float *)(base + o_rvsum); p.root_reward = (float *)(base + o_rrew);
    p.mm_max = (float *)(base + o_mmax); p.mm_min = (float *)(base + o_mmin);
    p.to_play = (int *)(base + o_tp); p.players_max = (int *)(base + o_players);
    p.path_slot = (int *)(base + o_pslot); p.path_action = (int *)(base + o_pact); p.path_len = (int *)(base + o_plen);
    p.vtp = (int *)(base + o_vtp); p.search_len = (int *)(base + o_slen);
    t->d_pbc = (float *)(base + o_pbc); p.pbc = t->d_pbc;
    p.rng_epoch = (unsigned long long *)(base + o_epoch);
    p.rng_seed = 0x5eed5eedull;
    *out = t;
    return lz_tree_set_params(t, 19652, 1.25f, 0.997f, 0.01f);
}

int lz_tree_destroy(lz_tree *t)
{
    if (!t) return LZ_OK;
    gumbel_free(t);
    cudaFree(t->alloc_base);
    delete t;
    return LZ_OK;
}

int lz_tree_set_params(lz_tree *t, int pb_c_base, float pb_c_init, float discount, float value_delta_max)
{
    LZ_REQUIRE(t, LZ_EINVAL, "lz_tree_set_params: null tree");
    LZ_REQUIRE(pb_c_base > 0, LZ_EINVAL, "lz_tree_set_params: pb_c_base must be > 0");
    // cucb_score (cnode.cpp:672): pb_c = log((N + base + 1) / base) + init, all fp32, N = visit_count - 1.
    // The argument only depends on the integer visit count, so the S+2 possible values are tabulated
    // once on the host with the same libm logf the reference binary links against.
    const int n = t->p.N + 1;
    std::vector<float> tab(n);
    const float base = (float)pb_c_base;
    for (int i = 0; i < n; ++i) {
        volatile float num = (float)i + base;
        num = num + 1;
        volatile float arg = num / base;
        volatile float lg = logf(arg);
        tab[i] = lg + pb_c_init;
    }
    LZ_CUDA_CHECK(cudaMemcpy(t->d_pbc, tab.data(), n * sizeof(float), cudaMemcpyHostToDevice));
    if (t->p.discount != discount || t->p.delta != value_delta_max) ++t->generation;   // passed BY VALUE into captured search graphs
    t->p.discount = discount;
    t->p.delta = value_delta_max;
    t->params_set = true;
    return LZ_OK;
}

int lz_tree_reset(lz_tree *t, const int32_t *d_legal, const int32_t *d_nlegal, lz_stream s)
{
    LZ_REQUIRE(t, LZ_EINVAL, "lz_tree_reset: null tree");
    LZ_REQUIRE((d_legal == nullptr) == (d_nlegal == nullptr), LZ_EINVAL, "lz_tree_reset: pass both d_legal and d_nlegal or neither");
    k_tree_reset<<<tree_grid(t->p.B), kTreeBlock, 0, (cudaStream_t)s>>>(t->p, d_legal, d_nlegal, nullptr);
    LZ_KERNEL_CHECK();
    t->prepared = false;
    return LZ_OK;
}

int lz_tree_reset_mask(lz_tree *t, const uint8_t *d_mask, lz_stream s)
{
    LZ_REQUIRE(t, LZ_EINVAL, "lz_tree_reset_mask: null tree");
    k_tree_reset<<<tree_grid(t->p.B), kTreeBlock, 0, (cudaStream_t)s>>>(t->p, nullptr, nullptr, d_mask);
    LZ_KERNEL_CHECK();
    t->prepared = false;
    return LZ_OK;
}

int lz_tree_prepare(lz_tree *t, const float *d_logits, const float *d_noise, float noise_weight,
                    const float *d_rewards, const int32_t *d_to_play, lz_stream s)
{
    LZ_REQUIRE(t && d_logits, LZ_EINVAL, "lz_tree_prepare: null argument");
    k_tree_prepare<<<tree_grid(t->p.B), kTreeBlock, 0, (cudaStream_t)s>>>(t->p, d_logits, d_noise, noise_weight,
                                                                         d_rewards, d_to_play);
    LZ_KERNEL_CHECK();
    t->prepared = true;
    return LZ_OK;
}

int lz_tree_traverse(lz_tree *t, int deterministic, int32_t *d_ix, int32_t *d_iy, int32_t *d_last_action,
                     int32_t *d_search_len, int32_t *d_virtual_to_play, lz_stream s)
{
    LZ_REQUIRE(t, LZ_EINVAL, "lz_tree_traverse: null tree");
    LZ_REQUIRE(t->prepared, LZ_ESTATE, "lz_tree_traverse: roots not prepared (call lz_tree_prepare first)");
    LZ_REQUIRE(!t->p.ez, LZ_ESTATE, "lz_tree_traverse: tree is in EfficientZero mode, use lz_tree_traverse_ez");
    return tree_launch_traverse(t, deterministic, d_ix, d_iy, d_last_action, d_search_len, d_virtual_to_play,
                                (cudaStream_t)s);
}

int lz_tree_backpropagate(lz_tree *t, int latent_index, const float *d_reward, const float *d_value,
                          const float *d_logits, const int32_t *d_to_play, lz_stream s)
{
    LZ_REQUIRE(t && d_reward && d_value && d_logits, LZ_EINVAL, "lz_tree_backpropagate: null argument");
    LZ_REQUIRE(t->prepared, LZ_ESTATE, "lz_tree_backpropagate: roots not prepared");
    LZ_REQUIRE(!t->p.ez, LZ_ESTATE, "lz_tree_backpropagate: tree is in EfficientZero mode, use lz_tree_backpropagate_ez");
    LZ_REQUIRE(latent_index >= 1 && latent_index <= t->max_sims, LZ_EINVAL,
               "lz_tree_backpropagate: latent_index %d outside [1, %d]", latent_index, t->max_sims);
    return tree_launch_backprop(t, latent_index, d_reward, d_value, d_logits, d_to_play, (cudaStream_t)s);
}

int lz_tree_set_ez(lz_tree *t, int efficientzero, int lstm_horizon_len)
{
    LZ_REQUIRE(t, LZ_EINVAL, "lz_tree_set_ez: null tree");
    LZ_REQUIRE(!efficientzero || lstm_horizon_len > 0, LZ_EINVAL, "lz_tree_set_ez: lstm_horizon_len must be > 0 (mcts_ctree.py:857)");
    const int ez = efficientzero ? 1 : 0, hor = efficientzero ? lstm_horizon_len : t->p.lstm_horizon;
    if (t->p.ez != ez || t->p.lstm_horizon != hor) ++t->generation;
    t->p.ez = ez;
    t->p.lstm_horizon = hor;
    return LZ_OK;
}

int lz_tree_set_tiebreak(lz_tree *t, int first_maximum)
{
    LZ_REQUIRE(t, LZ_EINVAL, "lz_tree_set_tiebreak: null tree");
    const int v = first_maximum ? 1 : 0;
    if (t->p.tie_first != v) ++t->generation;       // captured graphs bake TreeParams in
    t->p.tie_first = v;
    return LZ_OK;
}

int lz_tree_traverse_ez(lz_tree *t, int32_t *d_ix, int32_t *d_iy, int32_t *d_last_action, int32_t *d_search_len,
                        int32_t *d_virtual_to_play, int32_t *d_is_reset, lz_stream s)
{
    LZ_REQUIRE(t && t->p.ez, LZ_ESTATE, "lz_tree_traverse_ez: tree is not in EfficientZero mode (lz_tree_set_ez)");
    LZ_REQUIRE(t->prepared, LZ_ESTATE, "lz_tree_traverse_ez: roots not prepared (call lz_tree_prepare first)");
    return tree_launch_traverse(t, t->p.tie_first, d_ix, d_iy, d_last_action, d_search_len, d_virtual_to_play, (cudaStream_t)s, d_is_reset);
}

int lz_tree_backpropagate_ez(lz_tree *t, int latent_index, const float *d_value_prefix, const float *d_value,
                             const float *d_logits, const int32_t *d_is_reset, const int32_t *d_to_play, lz_stream s)
{
    LZ_REQUIRE(t && d_value_prefix && d_value && d_logits && d_is_reset, LZ_EINVAL, "lz_tree_backpropagate_ez: null argument");
    LZ_REQUIRE(t->p.ez, LZ_ESTATE, "lz_tree_backpropagate_ez: tree is not in EfficientZero mode (lz_tree_set_ez)");
    LZ_REQUIRE(t->prepared, LZ_ESTATE, "lz_tree_backpropagate_ez: roots not prepared");
    LZ_REQUIRE(latent_index >= 1 && latent_index <= t->max_sims, LZ_EINVAL,
               "lz_tree_backpropagate_ez: latent_index %d outside [1, %d]", latent_index, t->max_sims);
    return tree_launch_backprop(t, latent_index, d_value_prefix, d_value, d_logits, d_to_play, (cudaStream_t)s, d_is_reset);
}

int lz_tree_traverse_with_reuse(lz_tree *t, const int32_t *d_true_action, const float *d_reuse_value, int32_t *d_ix, int32_t *d_iy,
                                int32_t *d_last_action, int32_t *d_search_len, int32_t *d_virtual_to_play, lz_stream s)
{
    LZ_REQUIRE(t && d_true_action && d_reuse_value, LZ_EINVAL, "lz_tree_traverse_with_reuse: null argument");
    LZ_REQUIRE(t->prepared, LZ_ESTATE, "lz_tree_traverse_with_reuse: roots not prepared");
    return tree_launch_traverse_reuse(t, d_true_action, d_reuse_value, d_ix, nullptr, d_iy, d_last_action, d_search_len, d_virtual_to_play,
                                      (cudaStream_t)s);
}

int lz_tree_backpropagate_with_reuse(lz_tree *t, int latent_index, const float *d_reward, const float *d_value, const float *d_logits,
                                     const float *d_reuse_value, const int32_t *d_batch_rank, const int32_t *d_is_reset,
                                     const int32_t *d_to_play, lz_stream s)
{
    LZ_REQUIRE(t && d_reward && d_value && d_logits && d_reuse_value, LZ_EINVAL, "lz_tree_backpropagate_with_reuse: null argument");
    LZ_REQUIRE(t->prepared, LZ_ESTATE, "lz_tree_backpropagate_with_reuse: roots not prepared");
    LZ_REQUIRE(!t->p.ez || d_is_reset, LZ_EINVAL, "lz_tree_backpropagate_with_reuse: EfficientZero trees need d_is_reset");
    LZ_REQUIRE(latent_index >= 1 && latent_index <= t->max_sims, LZ_EINVAL,
               "lz_tree_backpropagate_with_reuse: latent_index %d outside [1, %d]", latent_index, t->max_sims);
    return tree_launch_backprop_reuse(t, latent_index, d_reward, d_value, d_logits, d_reuse_value, d_batch_rank, d_to_play, (cudaStream_t)s,
                                      d_is_reset);
}

int lz_tree_select_action(lz_tree *t, float temperature, int deterministic, uint64_t seed, int32_t *d_action,
                          int32_t *d_action_pos, float *d_entropy, lz_stream s)
{
    LZ_REQUIRE(t && temperature > 0.0f, LZ_EINVAL, "lz_tree_select_action: bad argument (temperature must be > 0)");
    k_tree_select_action<<<tree_grid(t->p.B), kTreeBlock, 0, (cudaStream_t)s>>>(t->p, 1.0 / (double)temperature, deterministic,
                                                                               (unsigned long long)seed, d_action, d_action_pos, d_entropy);
    LZ_KERNEL_CHECK();
    return LZ_OK;
}

int lz_tree_results(lz_tree *t, int32_t *d_visits, float *d_values, int32_t *d_nlegal, int32_t *d_traj, lz_stream s)
{
    LZ_REQUIRE(t, LZ_EINVAL, "lz_tree_results: null tree");
    k_tree_results<<<tree_grid(t->p.B), kTreeBlock, 0, (cudaStream_t)s>>>(t->p, d_visits, d_values, d_nlegal, d_traj);
    LZ_KERNEL_CHECK();
    return LZ_OK;
}

}  // extern "C"
