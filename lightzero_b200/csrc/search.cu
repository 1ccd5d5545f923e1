// search.cu -- the whole MuZeroMCTSCtree.search loop (lzero/mcts/tree_search/mcts_ctree.py:267-368) as ONE
// CUDA graph: [traverse] + num_simulations x [recurrent_inference -> backpropagate(+next traverse)].
// The reference's per-simulation host work (Python list gather of latents :323-324, two H2D copies
// :326-329, a duplicated recurrent_inference :338/:345, four blocking D2H copies :347-350 and three
// .tolist() conversions :355-357) has no counterpart here: the tree hands (slot, action) to the
// network through device memory and the network hands (reward, value, logits) back the same way.
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "model.cuh"
#include "tree.cuh"

struct lz_search {
    lz_tree *tree;
    lz_model *model;
    int S, B, A;
    float *pool;                 // [(S+1)][B][C*P] latent pool, slot-major, NCHW per root
    size_t slot_stride;          // B*C*P floats
    int32_t *d_ix, *d_action;    // [B]
    float *d_reward, *d_value;   // [B]
    float *d_policy;             // [B][A]
    float *d_root_logits;        // [B][A]
    float *d_root_value;         // [B]
    float *d_skip;               // [B][C*P] ResBlock skip scratch of the tcgen05 network kernel (per search: searches may overlap on streams)
    // EfficientZero: LSTM state pools [(S+1)][B][H] (tuple element 0 / 1 of reward_hidden_state, mcts_ctree.py:775-776)
    // and the per-leaf is_reset flags handed from the traverse to the LSTM kernel and the back-up (:856-861)
    float *hpool, *cpool;
    size_t hslot_stride;
    int32_t *d_is_reset;
    // ReZero search_with_reuse: library-owned copies of the caller's per-root true action / reuse value (graph-stable addresses)
    int32_t *d_true_action;
    float *d_reuse_value;
    cudaGraphExec_t exec_reuse;
    // Gumbel MuZero search graph: captured for one discount (baked into the kernel arguments); the tree generation covers S and m
    cudaGraphExec_t exec_gumbel;
    unsigned long long gen_model_gumbel, gen_tree_gumbel;
    float discount_gumbel;
    cudaGraphExec_t exec[2];     // [deterministic]
    unsigned long long gen_model[3], gen_tree[3];   // model / tree generation each graph (exec[0], exec[1], exec_reuse) was captured at
    cudaStream_t capture_stream; // library-owned: the caller's stream may be the legacy default stream,
                                 // which cannot be captured; the instantiated graph launches on the caller's
    int num_kernels;
    // host-buffer collect: staging + copy stream so the H2D of chunk i+1 overlaps the tower of chunk i
    cudaStream_t copy_stream, copy_stream2;   // chunks alternate between two copy streams (two DMA engines)
    cudaEvent_t ev_chunk[8], ev_start;
    float *d_obs_stage, *d_noise_stage, *d_pre_stage;
    uint8_t *d_mask_stage;
    int32_t *d_tp_stage;
    size_t obs_elems;            // floats per observation
};

using namespace lz;

static int enqueue_search(lz_search *q, int deterministic, cudaStream_t s)
{
    int rc;
    lz_tree *t = q->tree;
    t->step_counter = 0;
    // Persistent search: roots never interact, so the CTA that owns 7 roots can run their whole search -- tree
    // back-up / descent and the network -- for all num_simulations inside ONE launch of the tcgen05 kernel.
    const bool ez = q->model->kind == 0 && q->model->cfg.efficientzero;
    if (ez) {
        // EfficientZeroMCTSCtree.search (mcts_ctree.py:671-876): the LSTM step is a GEMM over all roots, so the network
        // is several launches per simulation and the loop stays a multi-kernel graph
        if ((rc = tree_launch_traverse(t, t->p.tie_first, q->d_ix, nullptr, q->d_action, nullptr, nullptr, s, q->d_is_reset))) return rc;
        for (int sim = 0; sim < q->S; ++sim) {
            RecIO io;
            memset(&io, 0, sizeof(io));
            io.B = q->B; io.latent_base = q->pool; io.ix = q->d_ix; io.slot_stride = q->slot_stride; io.action = q->d_action;
            io.next_latent = q->pool + (size_t)(sim + 1) * q->slot_stride;
            io.reward = q->d_reward; io.value = q->d_value; io.policy_logits = q->d_policy;
            io.h_base = q->hpool; io.c_base = q->cpool; io.hslot_stride = q->hslot_stride;
            io.h_out = q->hpool + (size_t)(sim + 1) * q->hslot_stride; io.c_out = q->cpool + (size_t)(sim + 1) * q->hslot_stride;
            io.is_reset = q->d_is_reset;
            io.skip_scratch = q->d_skip;
            if ((rc = model_recurrent(q->model, io, s))) return rc;
            if (sim + 1 < q->S)
                rc = tree_launch_backprop_traverse(t, sim + 1, q->d_reward, q->d_value, q->d_policy, t->p.tie_first, q->d_ix, q->d_action, s, q->d_is_reset);
            else
                rc = tree_launch_backprop(t, sim + 1, q->d_reward, q->d_value, q->d_policy, nullptr, s, q->d_is_reset);
            if (rc) return rc;
        }
        return LZ_OK;
    }
    if (q->model->kind == 0 && q->model->math != 0 && t->p.A <= 32 && !getenv("LZ_NO_PERSIST")) {   // tree_persist.cuh: one lane per child
        TcIO io;
        memset(&io, 0, sizeof(io));
        io.B = q->B; io.npass = (q->model->math == 1) ? 3 : 1;
        io.latent_base = q->pool; io.latent_pool_rw = q->pool; io.slot_stride = q->slot_stride;
        io.ix = q->d_ix; io.ix_rw = q->d_ix; io.action = q->d_action; io.action_rw = q->d_action;
        io.reward = q->d_reward; io.value = q->d_value; io.policy_logits = q->d_policy;
        io.persistent = 1; io.nsims = q->S; io.sim0 = 0; io.deterministic = deterministic;
        io.skip_scratch = q->d_skip;
        io.pool_cl = 1;      // slots >= 1 are written and read only by this kernel: channels-last (vector loads / stores); slot 0 stays NCHW
        return tc_launch(q->model->tc_rec, io, s, &t->p);
    }
    const bool pdl = q->model->kind == 0 && q->model->math != 0 && getenv("LZ_PDL");   // opt-in: measured slower (6.26 vs 5.90 ms per 50-sim search)
    t->pdl = pdl;
    if ((rc = tree_launch_traverse(t, deterministic, q->d_ix, nullptr, q->d_action, nullptr, nullptr, s))) return rc;
    for (int sim = 0; sim < q->S; ++sim) {
        RecIO io;
        memset(&io, 0, sizeof(io));
        io.B = q->B;
        io.latent_base = q->pool;
        io.ix = q->d_ix;
        io.slot_stride = q->slot_stride;
        io.action = q->d_action;
        io.next_latent = q->pool + (size_t)(sim + 1) * q->slot_stride;   // mcts_ctree.py:352,364
        io.reward = q->d_reward;
        io.value = q->d_value;
        io.policy_logits = q->d_policy;
        io.pdl = pdl ? 1 : 0;
        io.skip_scratch = q->d_skip;
        if ((rc = model_recurrent(q->model, io, s))) { t->pdl = false; return rc; }
        if (sim + 1 < q->S)
            rc = tree_launch_backprop_traverse(t, sim + 1, q->d_reward, q->d_value, q->d_policy, deterministic, q->d_ix, q->d_action, s);
        else
            rc = tree_launch_backprop(t, sim + 1, q->d_reward, q->d_value, q->d_policy, nullptr, s);
        if (rc) { t->pdl = false; return rc; }
    }
    t->pdl = false;
    return LZ_OK;
}

// MuZeroMCTSCtree.search_with_reuse (mcts_ctree.py:370-468): every tree goes through the network every simulation (the
// reference compacts the batch on the host; here the rows of "no inference" trees are computed and ignored, which keeps the
// loop one static CUDA graph): [traverse_with_reuse] + S x [recurrent_inference, backpropagate_with_reuse (+ next traverse)].
static int enqueue_search_reuse(lz_search *q, cudaStream_t s)
{
    int rc;
    lz_tree *t = q->tree;
    t->step_counter = 0;
    if (q->hpool) {
        // EfficientZeroMCTSCtree.search_with_reuse (mcts_ctree.py:878-1003): value-prefix trees, the LSTM step over all roots, is_reset
        // per tree from the descent; [traverse_with_reuse] + S x [conv trunk + heads, LSTM value-prefix head, backpropagate_with_reuse,
        // next traverse_with_reuse]
        if ((rc = tree_launch_traverse_reuse(t, q->d_true_action, q->d_reuse_value, nullptr, q->d_ix, nullptr, q->d_action, nullptr, nullptr, s,
                                             q->d_is_reset))) return rc;
        for (int sim = 0; sim < q->S; ++sim) {
            RecIO io;
            memset(&io, 0, sizeof(io));
            io.B = q->B; io.latent_base = q->pool; io.ix = q->d_ix; io.slot_stride = q->slot_stride; io.action = q->d_action;
            io.next_latent = q->pool + (size_t)(sim + 1) * q->slot_stride;
            io.reward = q->d_reward; io.value = q->d_value; io.policy_logits = q->d_policy;
            io.h_base = q->hpool; io.c_base = q->cpool; io.hslot_stride = q->hslot_stride;
            io.h_out = q->hpool + (size_t)(sim + 1) * q->hslot_stride; io.c_out = q->cpool + (size_t)(sim + 1) * q->hslot_stride;
            io.is_reset = q->d_is_reset;
            io.skip_scratch = q->d_skip;
            if ((rc = model_recurrent(q->model, io, s))) return rc;
            if ((rc = tree_launch_backprop_reuse(t, sim + 1, q->d_reward, q->d_value, q->d_policy, q->d_reuse_value, nullptr, nullptr, s,
                                                 q->d_is_reset))) return rc;
            if (sim + 1 < q->S &&
                (rc = tree_launch_traverse_reuse(t, q->d_true_action, q->d_reuse_value, nullptr, q->d_ix, nullptr, q->d_action, nullptr, nullptr, s,
                                                 q->d_is_reset))) return rc;
        }
        return LZ_OK;
    }
    if ((rc = tree_launch_traverse_reuse(t, q->d_true_action, q->d_reuse_value, nullptr, q->d_ix, nullptr, q->d_action, nullptr, nullptr, s))) return rc;
    for (int sim = 0; sim < q->S; ++sim) {
        RecIO io;
        memset(&io, 0, sizeof(io));
        io.B = q->B; io.latent_base = q->pool; io.ix = q->d_ix; io.slot_stride = q->slot_stride; io.action = q->d_action;
        io.next_latent = q->pool + (size_t)(sim + 1) * q->slot_stride;
        io.reward = q->d_reward; io.value = q->d_value; io.policy_logits = q->d_policy;
        io.skip_scratch = q->d_skip;
        if ((rc = model_recurrent(q->model, io, s))) return rc;
        if (sim + 1 < q->S)
            rc = tree_launch_backprop_traverse_reuse(t, sim + 1, q->d_reward, q->d_value, q->d_policy, q->d_true_action, q->d_reuse_value,
                                                     q->d_ix, q->d_action, s);
        else
            rc = tree_launch_backprop_reuse(t, sim + 1, q->d_reward, q->d_value, q->d_policy, q->d_reuse_value, nullptr, nullptr, s);
        if (rc) return rc;
    }
    return LZ_OK;
}

// GumbelMuZeroMCTSCtree.search (mcts_ctree.py:1076-1174): [traverse] + S x [recurrent_inference, backpropagate (+ next traverse)].
// The network is the multi-launch model_recurrent of the MuZero search (conv tcgen05 / SIMT or MLP); the persistent MuZero kernel
// (tree_persist.cuh) has no Gumbel descent.
static int enqueue_search_gumbel(lz_search *q, float discount, cudaStream_t s)
{
    int rc;
    lz_tree *t = q->tree;
    if ((rc = gumbel_launch_traverse(t, discount, q->d_ix, nullptr, q->d_action, nullptr, nullptr, s))) return rc;
    for (int sim = 0; sim < q->S; ++sim) {
        RecIO io;
        memset(&io, 0, sizeof(io));
        io.B = q->B; io.latent_base = q->pool; io.ix = q->d_ix; io.slot_stride = q->slot_stride; io.action = q->d_action;
        io.next_latent = q->pool + (size_t)(sim + 1) * q->slot_stride;
        io.reward = q->d_reward; io.value = q->d_value; io.policy_logits = q->d_policy;
        io.skip_scratch = q->d_skip;
        if ((rc = model_recurrent(q->model, io, s))) return rc;
        if (sim + 1 < q->S)
            rc = gumbel_launch_backprop_traverse(t, sim + 1, discount, q->d_reward, q->d_value, q->d_policy, q->d_ix, q->d_action, s);
        else
            rc = gumbel_launch_backprop(t, sim + 1, discount, q->d_reward, q->d_value, q->d_policy, s);
        if (rc) return rc;
    }
    return LZ_OK;
}

static int run_graph(lz_search *q, int deterministic, cudaStream_t s)
{
    const int d = deterministic ? 1 : 0;
    // a captured graph bakes in device pointers of the model's tables (passed by value in TcNet / NetDev / EzNet), the math mode
    // and the tree parameters (TreeParams by value): re-capture when any of them changed since (weight reload, set_math,
    // model_reserve growth, lz_tree_set_params / lz_tree_set_ez)
    if (q->exec[d] && (q->gen_model[d] != q->model->generation || q->gen_tree[d] != q->tree->generation)) {
        cudaGraphExecDestroy(q->exec[d]);
        q->exec[d] = nullptr;
    }
    if (!q->exec[d]) {
        q->gen_model[d] = q->model->generation;
        q->gen_tree[d] = q->tree->generation;
        cudaGraph_t graph = nullptr;
        if (!q->capture_stream) LZ_CUDA_CHECK(cudaStreamCreateWithFlags(&q->capture_stream, cudaStreamNonBlocking));
        LZ_CUDA_CHECK(cudaStreamBeginCapture(q->capture_stream, cudaStreamCaptureModeThreadLocal));
        int rc = enqueue_search(q, deterministic, q->capture_stream);
        cudaError_t e = cudaStreamEndCapture(q->capture_stream, &graph);
        if (rc != LZ_OK) { if (graph) cudaGraphDestroy(graph); return rc; }
        if (e != cudaSuccess) { set_error("cudaStreamEndCapture failed: %s", cudaGetErrorString(e)); return LZ_ECUDA; }
        size_t n = 0;
        LZ_CUDA_CHECK(cudaGraphGetNodes(graph, nullptr, &n));
        q->num_kernels = (int)n;
        e = cudaGraphInstantiate(&q->exec[d], graph, 0);
        cudaGraphDestroy(graph);
        if (e != cudaSuccess) { set_error("cudaGraphInstantiate failed: %s", cudaGetErrorString(e)); return LZ_ECUDA; }
    }
    LZ_CUDA_CHECK(cudaGraphLaunch(q->exec[d], s));
    count_launch(q->num_kernels);       // the graph's kernel nodes
    return LZ_OK;
}

extern "C" {

int lz_search_create(lz_tree *t, lz_model *m, int num_simulations, lz_search **out)
{
    LZ_REQUIRE(t && m && out && num_simulations > 0, LZ_EINVAL, "lz_search_create: bad argument");
    LZ_REQUIRE(m->finalized, LZ_ESTATE, "lz_search_create: model not finalized");
    LZ_REQUIRE(num_simulations <= t->max_sims, LZ_EINVAL, "lz_search_create: num_simulations %d > tree capacity %d", num_simulations, t->max_sims);
    LZ_REQUIRE(t->p.A == m->cfg.action_space_size, LZ_EINVAL, "lz_search_create: tree has %d actions, model %d", t->p.A, m->cfg.action_space_size);
    const bool ez = m->kind == 0 && m->cfg.efficientzero;
    LZ_REQUIRE(ez == (t->p.ez != 0), LZ_EINVAL, "lz_search_create: %s model needs a tree in %s mode (lz_tree_set_ez)",
               ez ? "an EfficientZero" : "a MuZero", ez ? "EfficientZero" : "MuZero");
    lz_search *q = new lz_search();
    memset(q, 0, sizeof(*q));
    q->tree = t; q->model = m; q->S = num_simulations; q->B = t->p.B; q->A = t->p.A;
    q->slot_stride = (size_t)q->B * m->latent_floats;
    int rc = dev_alloc(&q->pool, q->slot_stride * (size_t)(q->S + 1));
    if (rc == LZ_OK) rc = dev_alloc(&q->d_ix, (size_t)q->B);
    if (rc == LZ_OK) rc = dev_alloc(&q->d_action, (size_t)q->B);
    if (rc == LZ_OK) rc = dev_alloc(&q->d_reward, (size_t)q->B);
    if (rc == LZ_OK) rc = dev_alloc(&q->d_value, (size_t)q->B);
    if (rc == LZ_OK) rc = dev_alloc(&q->d_policy, (size_t)q->B * q->A);
    if (rc == LZ_OK) rc = dev_alloc(&q->d_root_logits, (size_t)q->B * q->A);
    if (rc == LZ_OK) rc = dev_alloc(&q->d_root_value, (size_t)q->B);
    if (rc == LZ_OK) rc = dev_alloc(&q->d_skip, q->slot_stride);
    if (rc == LZ_OK && ez) {
        q->hslot_stride = (size_t)q->B * m->cfg.lstm_hidden_size;
        rc = dev_alloc(&q->hpool, q->hslot_stride * (size_t)(q->S + 1));
        if (rc == LZ_OK) rc = dev_alloc(&q->cpool, q->hslot_stride * (size_t)(q->S + 1));
        if (rc == LZ_OK) rc = dev_alloc(&q->d_is_reset, (size_t)q->B);
    }
    if (rc == LZ_OK) rc = model_reserve(m, q->B);
    if (rc != LZ_OK) { lz_search_destroy(q); return rc; }
    *out = q;
    return LZ_OK;
}

int lz_search_destroy(lz_search *q)
{
    if (!q) return LZ_OK;
    for (int d = 0; d < 2; ++d) if (q->exec[d]) cudaGraphExecDestroy(q->exec[d]);
    if (q->capture_stream) cudaStreamDestroy(q->capture_stream);
    if (q->copy_stream) {
        cudaStreamDestroy(q->copy_stream);
        cudaStreamDestroy(q->copy_stream2);
        for (int i = 0; i < 8; ++i) cudaEventDestroy(q->ev_chunk[i]);
        cudaEventDestroy(q->ev_start);
    }
    cudaFree(q->d_obs_stage); cudaFree(q->d_noise_stage); cudaFree(q->d_pre_stage); cudaFree(q->d_mask_stage); cudaFree(q->d_tp_stage);
    cudaFree(q->pool); cudaFree(q->d_ix); cudaFree(q->d_action); cudaFree(q->d_reward); cudaFree(q->d_value);
    cudaFree(q->d_policy); cudaFree(q->d_root_logits); cudaFree(q->d_root_value); cudaFree(q->d_skip);
    cudaFree(q->hpool); cudaFree(q->cpool); cudaFree(q->d_is_reset);
    cudaFree(q->d_true_action); cudaFree(q->d_reuse_value);
    if (q->exec_reuse) cudaGraphExecDestroy(q->exec_reuse);
    if (q->exec_gumbel) cudaGraphExecDestroy(q->exec_gumbel);
    delete q;
    return LZ_OK;
}

static int ez_root_hidden(lz_search *q, const float *d_hidden0, const float *d_hidden1, cudaStream_t s)
{
    const size_t bytes = q->hslot_stride * sizeof(float);
    if (d_hidden0) LZ_CUDA_CHECK(cudaMemcpyAsync(q->hpool, d_hidden0, bytes, cudaMemcpyDeviceToDevice, s));
    else LZ_CUDA_CHECK(cudaMemsetAsync(q->hpool, 0, bytes, s));        // efficientzero_model.py:231-236: zeros after initial_inference
    if (d_hidden1) LZ_CUDA_CHECK(cudaMemcpyAsync(q->cpool, d_hidden1, bytes, cudaMemcpyDeviceToDevice, s));
    else LZ_CUDA_CHECK(cudaMemsetAsync(q->cpool, 0, bytes, s));
    return LZ_OK;
}

int lz_search_run_ez(lz_search *q, const float *d_latent_roots, const float *d_hidden0_roots, const float *d_hidden1_roots, lz_stream s)
{
    LZ_REQUIRE(q && q->hpool, LZ_EINVAL, "lz_search_run_ez: not an EfficientZero search");
    LZ_REQUIRE(q->tree->prepared, LZ_ESTATE, "lz_search_run_ez: roots not prepared (call lz_tree_prepare first)");
    if (d_latent_roots && d_latent_roots != q->pool)
        LZ_CUDA_CHECK(cudaMemcpyAsync(q->pool, d_latent_roots, q->slot_stride * sizeof(float), cudaMemcpyDeviceToDevice, (cudaStream_t)s));
    int rc = ez_root_hidden(q, d_hidden0_roots, d_hidden1_roots, (cudaStream_t)s);
    if (rc) return rc;
    return run_graph(q, 1, (cudaStream_t)s);
}

static int run_with_reuse(lz_search *q, const float *d_latent_roots, const int32_t *d_true_action, const float *d_reuse_value,
                          int32_t *d_infer_count, cudaStream_t s);

int lz_search_run_with_reuse(lz_search *q, const float *d_latent_roots, const int32_t *d_true_action, const float *d_reuse_value,
                             int32_t *d_infer_count, lz_stream s_)
{
    LZ_REQUIRE(q && d_true_action && d_reuse_value, LZ_EINVAL, "lz_search_run_with_reuse: null argument");
    LZ_REQUIRE(!q->hpool, LZ_ESTATE, "lz_search_run_with_reuse: EfficientZero search, use lz_search_run_ez_with_reuse");
    LZ_REQUIRE(q->tree->prepared, LZ_ESTATE, "lz_search_run_with_reuse: roots not prepared (call lz_tree_prepare first)");
    return run_with_reuse(q, d_latent_roots, d_true_action, d_reuse_value, d_infer_count, (cudaStream_t)s_);
}

int lz_search_run_ez_with_reuse(lz_search *q, const float *d_latent_roots, const float *d_hidden0_roots, const float *d_hidden1_roots,
                                const int32_t *d_true_action, const float *d_reuse_value, int32_t *d_infer_count, lz_stream s_)
{
    LZ_REQUIRE(q && d_true_action && d_reuse_value, LZ_EINVAL, "lz_search_run_ez_with_reuse: null argument");
    LZ_REQUIRE(q->hpool, LZ_ESTATE, "lz_search_run_ez_with_reuse: not an EfficientZero search");
    LZ_REQUIRE(q->tree->prepared, LZ_ESTATE, "lz_search_run_ez_with_reuse: roots not prepared (call lz_tree_prepare first)");
    int rc = ez_root_hidden(q, d_hidden0_roots, d_hidden1_roots, (cudaStream_t)s_);
    if (rc) return rc;
    return run_with_reuse(q, d_latent_roots, d_true_action, d_reuse_value, d_infer_count, (cudaStream_t)s_);
}

static int run_with_reuse(lz_search *q, const float *d_latent_roots, const int32_t *d_true_action, const float *d_reuse_value,
                          int32_t *d_infer_count, cudaStream_t s)
{
    if (!q->d_true_action) {
        int rc = dev_alloc(&q->d_true_action, (size_t)q->B);
        if (rc == LZ_OK) rc = dev_alloc(&q->d_reuse_value, (size_t)q->B);
        if (rc != LZ_OK) return rc;
    }
    if (d_latent_roots && d_latent_roots != q->pool)
        LZ_CUDA_CHECK(cudaMemcpyAsync(q->pool, d_latent_roots, q->slot_stride * sizeof(float), cudaMemcpyDeviceToDevice, s));
    LZ_CUDA_CHECK(cudaMemcpyAsync(q->d_true_action, d_true_action, (size_t)q->B * sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
    LZ_CUDA_CHECK(cudaMemcpyAsync(q->d_reuse_value, d_reuse_value, (size_t)q->B * sizeof(float), cudaMemcpyDeviceToDevice, s));
    LZ_CUDA_CHECK(cudaMemsetAsync(q->tree->p.infer_count, 0, (size_t)q->tree->p.N * sizeof(int), s));
    if (q->exec_reuse && (q->gen_model[2] != q->model->generation || q->gen_tree[2] != q->tree->generation)) {
        cudaGraphExecDestroy(q->exec_reuse);
        q->exec_reuse = nullptr;
    }
    if (!q->exec_reuse) {
        q->gen_model[2] = q->model->generation;
        q->gen_tree[2] = q->tree->generation;
        cudaGraph_t graph = nullptr;
        if (!q->capture_stream) LZ_CUDA_CHECK(cudaStreamCreateWithFlags(&q->capture_stream, cudaStreamNonBlocking));
        LZ_CUDA_CHECK(cudaStreamBeginCapture(q->capture_stream, cudaStreamCaptureModeThreadLocal));
        int rc = enqueue_search_reuse(q, q->capture_stream);
        cudaError_t e = cudaStreamEndCapture(q->capture_stream, &graph);
        if (rc != LZ_OK) { if (graph) cudaGraphDestroy(graph); return rc; }
        if (e != cudaSuccess) { set_error("cudaStreamEndCapture failed: %s", cudaGetErrorString(e)); return LZ_ECUDA; }
        e = cudaGraphInstantiate(&q->exec_reuse, graph, 0);
        cudaGraphDestroy(graph);
        if (e != cudaSuccess) { set_error("cudaGraphInstantiate failed: %s", cudaGetErrorString(e)); return LZ_ECUDA; }
    }
    LZ_CUDA_CHECK(cudaGraphLaunch(q->exec_reuse, s));
    if (d_infer_count)      // per simulation: how many trees needed the network (mcts_ctree.py:433,466-467)
        LZ_CUDA_CHECK(cudaMemcpyAsync(d_infer_count, q->tree->p.infer_count, (size_t)q->S * sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
    return LZ_OK;
}

int lz_search_run(lz_search *q, const float *d_latent_roots, int deterministic, lz_stream s)
{
    LZ_REQUIRE(q, LZ_EINVAL, "lz_search_run: null search");
    LZ_REQUIRE(!q->hpool, LZ_ESTATE, "lz_search_run: EfficientZero search, use lz_search_run_ez");
    LZ_REQUIRE(q->tree->prepared, LZ_ESTATE, "lz_search_run: roots not prepared (call lz_tree_prepare first)");
    if (d_latent_roots && d_latent_roots != q->pool)
        LZ_CUDA_CHECK(cudaMemcpyAsync(q->pool, d_latent_roots, q->slot_stride * sizeof(float), cudaMemcpyDeviceToDevice, (cudaStream_t)s));
    return run_graph(q, deterministic, (cudaStream_t)s);
}

int lz_search_run_gumbel(lz_search *q, const float *d_latent_roots, float discount, lz_stream s_)
{
    LZ_REQUIRE(q, LZ_EINVAL, "lz_search_run_gumbel: null search");
    LZ_REQUIRE(!q->hpool, LZ_EINVAL, "lz_search_run_gumbel: Gumbel MuZero runs on MuZero models, not EfficientZero");
    lz_tree *t = q->tree;
    LZ_REQUIRE(t->gumbel, LZ_ESTATE, "lz_search_run_gumbel: tree is not in Gumbel mode (lz_tree_set_gumbel)");
    LZ_REQUIRE(t->gp.S == q->S, LZ_EINVAL, "lz_search_run_gumbel: tree set for num_simulations=%d, search created for %d", t->gp.S, q->S);
    LZ_REQUIRE(t->prepared, LZ_ESTATE, "lz_search_run_gumbel: roots not prepared (call lz_tree_prepare_gumbel first)");
    LZ_REQUIRE(t->gumbel_traversals == 0, LZ_ESTATE, "lz_search_run_gumbel: %d traverses since prepare (prepare again)", t->gumbel_traversals);
    cudaStream_t s = (cudaStream_t)s_;
    if (d_latent_roots && d_latent_roots != q->pool)
        LZ_CUDA_CHECK(cudaMemcpyAsync(q->pool, d_latent_roots, q->slot_stride * sizeof(float), cudaMemcpyDeviceToDevice, s));
    if (q->exec_gumbel && (q->gen_model_gumbel != q->model->generation || q->gen_tree_gumbel != t->generation ||
                           q->discount_gumbel != discount)) {
        cudaGraphExecDestroy(q->exec_gumbel);
        q->exec_gumbel = nullptr;
    }
    if (!q->exec_gumbel) {
        q->gen_model_gumbel = q->model->generation;
        q->gen_tree_gumbel = t->generation;
        q->discount_gumbel = discount;
        cudaGraph_t graph = nullptr;
        if (!q->capture_stream) LZ_CUDA_CHECK(cudaStreamCreateWithFlags(&q->capture_stream, cudaStreamNonBlocking));
        LZ_CUDA_CHECK(cudaStreamBeginCapture(q->capture_stream, cudaStreamCaptureModeThreadLocal));
        int rc = enqueue_search_gumbel(q, discount, q->capture_stream);
        cudaError_t e = cudaStreamEndCapture(q->capture_stream, &graph);
        if (rc != LZ_OK) { if (graph) cudaGraphDestroy(graph); q->exec_gumbel = nullptr; return rc; }
        if (e != cudaSuccess) { set_error("cudaStreamEndCapture failed: %s", cudaGetErrorString(e)); return LZ_ECUDA; }
        size_t n = 0;
        LZ_CUDA_CHECK(cudaGraphGetNodes(graph, nullptr, &n));
        q->num_kernels = (int)n;
        e = cudaGraphInstantiate(&q->exec_gumbel, graph, 0);
        cudaGraphDestroy(graph);
        if (e != cudaSuccess) { q->exec_gumbel = nullptr; set_error("cudaGraphInstantiate failed: %s", cudaGetErrorString(e)); return LZ_ECUDA; }
    }
    LZ_CUDA_CHECK(cudaGraphLaunch(q->exec_gumbel, s));
    count_launch(q->num_kernels);
    t->gumbel_traversals = q->S;
    return LZ_OK;
}

static int collect_device(lz_search *q, const float *d_obs, const uint8_t *d_obs_u8, const uint8_t *d_mask, const float *d_noise,
                          float noise_weight, const int32_t *d_to_play, int deterministic, float *d_pred_value,
                          float *d_policy_logits, lz_stream s)
{
    LZ_REQUIRE(q && (d_obs || d_obs_u8), LZ_EINVAL, "lz_search_collect: bad argument");
    TailIO io;
    memset(&io, 0, sizeof(io));
    io.latent2 = q->pool;                                   // latent roots go straight into pool slot 0
    io.policy_logits = d_policy_logits ? d_policy_logits : q->d_root_logits;
    io.value = d_pred_value ? d_pred_value : q->d_root_value;
    int rc;
    if (d_obs_u8) {
        LZ_REQUIRE(q->model->kind == 0 && q->model->math != 0 && q->model->cfg.obs_h != 64, LZ_EINVAL,
                   "lz_search_collect_u8: uint8 frames need the tcgen05 conv model (84x84 / 96x96)");
        if (!q->d_pre_stage && (rc = dev_alloc(&q->d_pre_stage, (size_t)q->B * q->model->latent_floats))) return rc;
        rc = model_initial_tower(q->model, q->B, nullptr, q->d_pre_stage, (cudaStream_t)s, d_obs_u8);
        if (rc == LZ_OK) rc = model_initial_tail(q->model, q->B, q->d_pre_stage, io, (cudaStream_t)s);
    } else {
        rc = model_initial(q->model, q->B, d_obs, io, (cudaStream_t)s);          // policy/muzero.py:749
    }
    if (rc) return rc;
    if ((rc = lz_tree_reset_mask(q->tree, d_mask, s))) return rc;                // :760,769
    if ((rc = lz_tree_prepare(q->tree, io.policy_logits, d_noise, noise_weight, nullptr, d_to_play, s))) return rc;   // :774
    if (q->hpool) {      // EfficientZero: zero LSTM state at the roots; the tree has no deterministic argument, the collect call's flag selects its tie-breaking
        if ((rc = ez_root_hidden(q, nullptr, nullptr, (cudaStream_t)s))) return rc;
        if ((rc = lz_tree_set_tiebreak(q->tree, deterministic))) return rc;
    }
    return run_graph(q, deterministic, (cudaStream_t)s);                         // :775
}

int lz_search_collect(lz_search *q, const float *d_obs, const uint8_t *d_mask, const float *d_noise, float noise_weight,
                      const int32_t *d_to_play, int deterministic, float *d_pred_value, float *d_policy_logits, lz_stream s)
{
    return collect_device(q, d_obs, nullptr, d_mask, d_noise, noise_weight, d_to_play, deterministic, d_pred_value, d_policy_logits, s);
}

int lz_search_collect_u8(lz_search *q, const uint8_t *d_obs_u8, const uint8_t *d_mask, const float *d_noise, float noise_weight,
                         const int32_t *d_to_play, int deterministic, float *d_pred_value, float *d_policy_logits, lz_stream s)
{
    return collect_device(q, nullptr, d_obs_u8, d_mask, d_noise, noise_weight, d_to_play, deterministic, d_pred_value, d_policy_logits, s);
}

static int collect_host(lz_search *q, const void *h_obs, int obs_u8, const uint8_t *h_mask, const float *h_noise, float noise_weight,
                        const int32_t *h_to_play, int deterministic, int nchunks, float *d_pred_value,
                        float *d_policy_logits, lz_stream s_)
{
    LZ_REQUIRE(q && h_obs, LZ_EINVAL, "lz_search_collect_host: bad argument");
    LZ_REQUIRE(!obs_u8 || (q->model->kind == 0 && q->model->math != 0 && q->model->cfg.obs_h != 64), LZ_EINVAL,
               "lz_search_collect_host_u8: uint8 frames need the tcgen05 conv model (84x84 / 96x96)");
    const size_t esz = obs_u8 ? 1 : sizeof(float);         // bytes per observation element on the wire and in the staging buffer
    cudaStream_t s = (cudaStream_t)s_;
    const lz_model_config &c = q->model->cfg;
    const int B = q->B, A = q->A;
    const size_t obs_elems = q->model->kind == 1 ? (size_t)q->model->mcfg.obs_dim : (size_t)c.obs_c * c.obs_h * c.obs_w;
    nchunks = nchunks < 1 ? 1 : (nchunks > 8 ? 8 : nchunks);
    if (!q->copy_stream) {
        q->obs_elems = obs_elems;
        LZ_CUDA_CHECK(cudaStreamCreateWithFlags(&q->copy_stream, cudaStreamNonBlocking));
        LZ_CUDA_CHECK(cudaStreamCreateWithFlags(&q->copy_stream2, cudaStreamNonBlocking));
        for (int i = 0; i < 8; ++i) LZ_CUDA_CHECK(cudaEventCreateWithFlags(&q->ev_chunk[i], cudaEventDisableTiming));
        LZ_CUDA_CHECK(cudaEventCreateWithFlags(&q->ev_start, cudaEventDisableTiming));
        int rc = dev_alloc(&q->d_obs_stage, q->obs_elems * B);
        if (rc == LZ_OK) rc = dev_alloc(&q->d_noise_stage, (size_t)B * A);
        if (rc == LZ_OK && !q->d_pre_stage) rc = dev_alloc(&q->d_pre_stage, (size_t)B * q->model->latent_floats);
        if (rc == LZ_OK) rc = dev_alloc(&q->d_mask_stage, (size_t)B * A);
        if (rc == LZ_OK) rc = dev_alloc(&q->d_tp_stage, (size_t)B);
        if (rc != LZ_OK) return rc;
    }
    // the copy stream may not overwrite the staging buffer before earlier work on `s` has consumed it
    LZ_CUDA_CHECK(cudaEventRecord(q->ev_start, s));
    LZ_CUDA_CHECK(cudaStreamWaitEvent(q->copy_stream, q->ev_start, 0));
    LZ_CUDA_CHECK(cudaStreamWaitEvent(q->copy_stream2, q->ev_start, 0));
    const bool two = !getenv("LZ_ONE_COPY_STREAM");
    const int per = (B + nchunks - 1) / nchunks;
    for (int i = 0; i < nchunks; ++i) {
        const int b0 = i * per, bc = std::min(per, B - b0);
        if (bc <= 0) { nchunks = i; break; }
        cudaStream_t cs = (two && (i & 1)) ? q->copy_stream2 : q->copy_stream;
        LZ_CUDA_CHECK(cudaMemcpyAsync(reinterpret_cast<unsigned char *>(q->d_obs_stage) + (size_t)b0 * q->obs_elems * esz,
                                      static_cast<const unsigned char *>(h_obs) + (size_t)b0 * q->obs_elems * esz,
                                      (size_t)bc * q->obs_elems * esz, cudaMemcpyHostToDevice, cs));
        LZ_CUDA_CHECK(cudaEventRecord(q->ev_chunk[i], cs));
    }
    if (h_mask) LZ_CUDA_CHECK(cudaMemcpyAsync(q->d_mask_stage, h_mask, (size_t)B * A, cudaMemcpyHostToDevice, s));
    if (h_noise) LZ_CUDA_CHECK(cudaMemcpyAsync(q->d_noise_stage, h_noise, (size_t)B * A * sizeof(float), cudaMemcpyHostToDevice, s));
    if (h_to_play) LZ_CUDA_CHECK(cudaMemcpyAsync(q->d_tp_stage, h_to_play, (size_t)B * sizeof(int32_t), cudaMemcpyHostToDevice, s));
    float *logits = d_policy_logits ? d_policy_logits : q->d_root_logits;
    float *pred = d_pred_value ? d_pred_value : q->d_root_value;
    const bool split = q->model->kind == 0 && q->model->math != 0 && c.obs_h != 64;   // tower per chunk, tail once
    for (int i = 0; i < nchunks; ++i) {
        const int b0 = i * per, bc = std::min(per, B - b0);
        LZ_CUDA_CHECK(cudaStreamWaitEvent(s, q->ev_chunk[i], 0));
        int rc;
        if (split) {
            const unsigned char *stage = reinterpret_cast<const unsigned char *>(q->d_obs_stage) + (size_t)b0 * q->obs_elems * esz;
            rc = model_initial_tower(q->model, bc, obs_u8 ? nullptr : reinterpret_cast<const float *>(stage),
                                     q->d_pre_stage + (size_t)b0 * q->model->latent_floats, s, obs_u8 ? stage : nullptr);
        } else {
            TailIO io;
            memset(&io, 0, sizeof(io));
            io.latent2 = q->pool + (size_t)b0 * q->model->latent_floats;
            io.policy_logits = logits + (size_t)b0 * A;
            io.value = pred + b0;
            rc = model_initial(q->model, bc, q->d_obs_stage + (size_t)b0 * q->obs_elems, io, s);
        }
        if (rc) return rc;
    }
    if (split) {
        TailIO io;
        memset(&io, 0, sizeof(io));
        io.latent2 = q->pool;
        io.policy_logits = logits;
        io.value = pred;
        int rc = model_initial_tail(q->model, B, q->d_pre_stage, io, s);
        if (rc) return rc;
    }
    int rc;
    if ((rc = lz_tree_reset_mask(q->tree, h_mask ? q->d_mask_stage : nullptr, s))) return rc;
    if ((rc = lz_tree_prepare(q->tree, logits, h_noise ? q->d_noise_stage : nullptr, noise_weight, nullptr,
                              h_to_play ? q->d_tp_stage : nullptr, s))) return rc;
    if (q->hpool) {
        if ((rc = ez_root_hidden(q, nullptr, nullptr, s))) return rc;
        if ((rc = lz_tree_set_tiebreak(q->tree, deterministic))) return rc;
    }
    return run_graph(q, deterministic, s);
}

int lz_search_collect_host(lz_search *q, const float *h_obs, const uint8_t *h_mask, const float *h_noise, float noise_weight,
                           const int32_t *h_to_play, int deterministic, int nchunks, float *d_pred_value,
                           float *d_policy_logits, lz_stream s)
{
    return collect_host(q, h_obs, 0, h_mask, h_noise, noise_weight, h_to_play, deterministic, nchunks, d_pred_value, d_policy_logits, s);
}

int lz_search_collect_host_u8(lz_search *q, const uint8_t *h_obs_u8, const uint8_t *h_mask, const float *h_noise, float noise_weight,
                              const int32_t *h_to_play, int deterministic, int nchunks, float *d_pred_value,
                              float *d_policy_logits, lz_stream s)
{
    return collect_host(q, h_obs_u8, 1, h_mask, h_noise, noise_weight, h_to_play, deterministic, nchunks, d_pred_value, d_policy_logits, s);
}

int lz_search_num_kernels(const lz_search *q) { return q ? q->num_kernels : 0; }
const float *lz_search_latent_pool(const lz_search *q) { return q ? q->pool : nullptr; }
const float *lz_search_hidden_pool(const lz_search *q, int which) { return q ? (which ? q->cpool : q->hpool) : nullptr; }

}  // extern "C"
