// rr_engine.cu — one model replica on one GPU: chunked prefill + continuous-batching greedy decode.
//
// Replaces one `litellm_params.model: bedrock/...` deployment of the reference
// (config/config.yaml:39,47,54,62,69,77,84,91) and the remote bedrock:InvokeModel call behind it
// (iam/policy.json:8, src/demo_cris.py:233-238).  The request-facing call shape
// (submit -> wait -> tokens + timestamps) is what chat.completions.create needs
// (src/demo_load_balancing.py:106-116).
//
// Layout in HBM (one replica): bf16 weights (caller-owned), KV cache
// [layer][slot][kv_head][ctx_max][128] bf16 for K and for V, a decode working set of max_batch
// rows (row b == KV slot b) and a prefill working set of max_prefill_tokens rows.
// The decode step is a fixed sequence of 6 launches per layer + 4, captured once in a CUDA graph
// and replayed; per-row metadata (token, position, active flag) lives on the device so replays
// need no parameter changes.
#include "rr_kernels.h"
#include "rr_launch.cuh"

#include <atomic>
#include <chrono>
#include <condition_variable>
#include <deque>
#include <map>
#include <mutex>
#include <new>
#include <string.h>
#include <thread>
#include <unordered_map>
#include <vector>

#define RR_API extern "C" __attribute__((visibility("default")))

namespace rr {
void note_cuda_error(cudaError_t e);

__global__ void gather_rows_kernel(const __nv_bfloat16* __restrict__ src, const int32_t* __restrict__ idx,
                                   __nv_bfloat16* __restrict__ dst, int hidden) {
    griddep_launch();
    griddep_wait();
    const int r = blockIdx.x;
    const uint4* s = reinterpret_cast<const uint4*>(src + (size_t)idx[r] * hidden);
    uint4* d = reinterpret_cast<uint4*>(dst + (size_t)r * hidden);
    for (int c = threadIdx.x; c < hidden / 8; c += blockDim.x) d[c] = s[c];
}

// Last layer of a prefill chunk: only the last token of every prompt still matters after attention.  Gather those
// rows (attention output bf16, residual fp32) into the decode working set; the rest of the layer and lm_head then run
// on n_seqs rows with the weight-streaming (decode-orientation) kernels instead of on all T tokens.
__global__ void gather_last_kernel(const __nv_bfloat16* __restrict__ attn, const float* __restrict__ x,
                                   const int32_t* __restrict__ last, __nv_bfloat16* __restrict__ attn_out,
                                   float* __restrict__ x_out, int nq, int hidden) {
    griddep_launch();
    griddep_wait();
    const int r = blockIdx.x;
    const size_t src = (size_t)last[r];
    const uint4* a = reinterpret_cast<const uint4*>(attn + src * nq);
    uint4* ao = reinterpret_cast<uint4*>(attn_out + (size_t)r * nq);
    for (int c = threadIdx.x; c < nq / 8; c += blockDim.x) ao[c] = a[c];
    const float4* xs = reinterpret_cast<const float4*>(x + src * hidden);
    float4* xo = reinterpret_cast<float4*>(x_out + (size_t)r * hidden);
    for (int c = threadIdx.x; c < hidden / 4; c += blockDim.x) xo[c] = xs[c];
}

// After a prefill chunk: row/slot s becomes an active decode row fed with its first token.
__global__ void activate_rows_kernel(const int32_t* __restrict__ seq_slot, const int32_t* __restrict__ first_tok,
                                     const int32_t* __restrict__ seq_start, int n, int32_t* __restrict__ d_tok,
                                     int32_t* __restrict__ d_pos, int32_t* __restrict__ d_slot) {
    griddep_launch();
    griddep_wait();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int s = seq_slot[i];
    d_tok[s] = first_tok[i];
    d_pos[s] = seq_start[i + 1] - seq_start[i];
    d_slot[s] = s;
}

struct Request {
    uint64_t ticket;
    std::vector<int32_t> prompt;
    int max_new;
    std::vector<int32_t> out;
    int status = RR_OK;
    bool done = false;
    double t_submit = 0, t_first = 0, t_done = 0;
    int slot = -1;
    uint64_t tag = 0;          // opaque caller value handed to the done hook (the gateway's request id)
    bool cancel = false;       // rr_engine_cancel: the worker drops the row at the next step
    bool detached = false;     // nobody will call rr_engine_wait: the worker frees the request when it finishes
};

}  // namespace rr

using namespace rr;

#define CK(x)                                   \
    do {                                        \
        cudaError_t e__ = (x);                  \
        if (e__ != cudaSuccess) {               \
            rr::note_cuda_error(e__);           \
            return RR_CUDA_ERROR;               \
        }                                       \
    } while (0)

struct rr_engine {
    rr_model_desc d;
    rr_engine_opts o;
    int Bm, bn_dec, nq, nkv_dim, nqkv;
    std::vector<const void*> wqkv, wo, wgu, wdown, norm_attn, norm_mlp;
    const void *embed, *lm_head, *final_norm;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    std::vector<void*> allocs;

    // decode working set
    int32_t *d_tok, *d_pos, *d_slot;
    float* x;
    __nv_bfloat16 *xn, *qbuf, *attn_out, *act;
    float *part_qkv, *part_o, *part_gu, *part_down, *logits, *attn_ws;   // split-K partial planes
    float2* rope_table;
    __nv_bfloat16 *kcache, *vcache;
    size_t kv_layer_stride;
    int kv_splits;
    std::vector<GemmPlan> pl_qkv, pl_o, pl_gu, pl_down;
    std::vector<DecodeAttnArgs> attn_args;   // per layer (TMA maps of that layer's K / V cache)
    std::vector<PrefillAttnArgs> pf_attn;    // per layer (TMA maps of q and of that layer's K / V cache)
    GemmPlan pl_head, pl_head_pf;
    int s_qkv, s_o, s_gu, s_down;
    bool fuse_rope_pf = false;        // prefill: RoPE + KV append live in the QKV GEMM epilogue (head_dim 128)
    bool defer_norm_pf = false;       // prefill: no norm kernels -- RESID epilogues emit bf16(x * gamma) + sum(x^2), the next
                                      // GEMM's epilogue applies 1 / rms (RopeEpi)
    float* p_rowss = nullptr;         // [Tmax][pf_parts]
    int pf_parts = 0;
    bool fuse_silu = false;           // wgu interleaved + one gate/up plane: SiLU*mul lives in the GEMM epilogue
    bool fuse_mlp = false;            // decode: gate/up and down GEMMs in one persistent launch (gemm_mlp_tcgen05)
    std::vector<MlpPlan> mlp;         // per layer
    MlpItem* mlp_items = nullptr;     // device copy of the schedule (shared by all layers)
    unsigned* mlp_ready = nullptr;    // [n_slices] dependency counters, reset by the norm kernel before each launch
    int mlp_slices = 0, mlp_slice_kb = 0;
    cudaGraphExec_t graph = nullptr;
    bool warmed = false;

    // prefill working set
    int Tmax;
    int32_t *p_ids, *p_pos, *p_slot, *p_seq_start, *p_seq_slot, *p_last, *p_first;
    float* px;
    __nv_bfloat16 *pxn, *pqkv, *pq, *pattn, *po, *pgu, *pact, *xn_last;
    struct PfPlans { std::vector<GemmPlan> qkv, o, gu, down; };
    std::map<int, PfPlans> pf_plans;

    // pinned staging
    int32_t* h_stage;     // ids | pos | slot | seq_start | seq_slot | last   (prefill) / rows meta (decode)
    size_t h_stage_ints;
    int32_t* h_tok;       // [Bm] tokens read back each step
    float* h_logits = nullptr;

    // serving state
    std::mutex mu;                       // queues + request table
    std::condition_variable cv_work, cv_done;
    std::mutex gpu_mu;                   // serialises GPU work between worker and low-level API
    std::deque<Request*> waiting;
    std::unordered_map<uint64_t, Request*> table;
    std::vector<Request*> row_req;       // [Bm]
    std::vector<int32_t> h_slot_mirror;  // host mirror of d_slot
    bool slots_dirty = false;
    std::thread worker;
    std::atomic<bool> stop{false};
    uint64_t next_ticket = 1;
    std::chrono::steady_clock::time_point t0;

    rr_engine_stats st;                  // written under gpu_mu (launch / timing counters) or mu (queued, active_rows)
    uint64_t step_launches = 0;
    // completion hook (the native gateway, rr_gateway.cu): called on the worker / submitting thread, outside `mu`
    rr::EngineDoneHook hook = nullptr;
    void* hook_ctx = nullptr;
};

static double now_s(rr_engine* e) {
    return std::chrono::duration<double>(std::chrono::steady_clock::now() - e->t0).count();
}

template <typename T>
static int dalloc(rr_engine* e, T** p, size_t n, bool zero = true) {
    void* q = nullptr;
    cudaError_t err = cudaMalloc(&q, n * sizeof(T) ? n * sizeof(T) : 16);
    if (err != cudaSuccess) { rr::note_cuda_error(err); return RR_CUDA_ERROR; }
    if (zero) cudaMemset(q, 0, n * sizeof(T));
    e->allocs.push_back(q);
    *p = (T*)q;
    return RR_OK;
}

static int pick_bn(int rows) {
    const int opts[5] = {16, 32, 64, 128, 256};
    for (int b : opts) if (rows <= b) return b;
    return -1;
}
static int pick_splits(int N, int K) {
    const int tilesA = (N + 127) / 128;
    int s = num_sms() / tilesA;
    const int kblocks = (K + 63) / 64;
    if (s < 1) s = 1;
    if (s > 8) s = 8;
    while (s > 1 && kblocks / s < 8) --s;
    return s;
}

// One engine at a time per device.  The fused MLP kernel is a persistent grid whose CTAs spin on work of sibling CTAs;
// two such grids interleaved on one GPU (two engines, two streams) could each hold SMs the other's not-yet-resident CTAs
// need.  Every path below synchronises its stream before it releases this lock, so
// engines that share a device alternate at prefill-chunk / decode-step granularity.  (The gateway creates one engine per
// GPU, so this lock is uncontended there.)
static std::mutex& device_mutex(int dev) {
    static std::mutex mu[64];
    return mu[dev & 63];
}

static PartIn part_f32(const float* p, int splits, int rows, int ld) {
    PartIn r; r.ptr = p; r.is_bf16 = 0; r.n_splits = splits; r.split_stride = (long long)rows * ld; r.ld = ld;
    return r;
}
static PartIn part_bf16(const __nv_bfloat16* p, int ld) {
    PartIn r; r.ptr = p; r.is_bf16 = 1; r.n_splits = 1; r.split_stride = 0; r.ld = ld;
    return r;
}
static PartIn part_none() { PartIn r; r.ptr = nullptr; r.is_bf16 = 0; r.n_splits = 1; r.split_stride = 0; r.ld = 0; return r; }

// ---------------------------------------------------------------- decode step (enqueue only)
static int enqueue_decode_step(rr_engine* e, cudaStream_t s, uint64_t* n_launch) {
    const rr_model_desc& d = e->d;
    const int B = e->Bm, L = d.n_layers;
    uint64_t nl = 0;
    launch_embed(e->d_tok, (const __nv_bfloat16*)e->embed, e->x, B, d.hidden, e->d_slot, s); ++nl;
    launch_add_rmsnorm(e->x, part_none(), (const __nv_bfloat16*)e->norm_attn[0], e->xn, B, d.hidden, d.rms_eps, s); ++nl;
    for (int l = 0; l < L; ++l) {
        __nv_bfloat16* kc = e->kcache + (size_t)l * e->kv_layer_stride;
        __nv_bfloat16* vc = e->vcache + (size_t)l * e->kv_layer_stride;
        if (gemm_launch(e->pl_qkv[l], s) != RR_OK) return RR_CUDA_ERROR; ++nl;
        // RoPE + KV append are fused into the attention kernel (reads the QKV split-K planes directly)
        launch_decode_attn(e->attn_args[l], s); nl += e->kv_splits > 1 ? 2 : 1;
        if (gemm_launch(e->pl_o[l], s) != RR_OK) return RR_CUDA_ERROR; ++nl;
        const void* nw = (l + 1 < L) ? e->norm_attn[l + 1] : e->final_norm;
        if (e->fuse_mlp) {
            launch_add_rmsnorm(e->x, part_f32(e->part_o, e->s_o, B, d.hidden), (const __nv_bfloat16*)e->norm_mlp[l],
                               e->xn, B, d.hidden, d.rms_eps, s, e->mlp_ready, e->mlp_slices + 1); ++nl;
            if (mlp_launch(e->mlp[l], s) != RR_OK) return RR_CUDA_ERROR; ++nl;
            launch_add_rmsnorm(e->x, part_f32(e->part_down, e->mlp_slices, B, d.hidden), (const __nv_bfloat16*)nw, e->xn, B,
                               d.hidden, d.rms_eps, s); ++nl;
            continue;
        }
        launch_add_rmsnorm(e->x, part_f32(e->part_o, e->s_o, B, d.hidden), (const __nv_bfloat16*)e->norm_mlp[l],
                           e->xn, B, d.hidden, d.rms_eps, s); ++nl;
        if (gemm_launch(e->pl_gu[l], s) != RR_OK) return RR_CUDA_ERROR; ++nl;
        if (!e->fuse_silu) { launch_silu_mul(part_f32(e->part_gu, e->s_gu, B, 2 * d.inter), e->act, B, d.inter, s); ++nl; }
        if (gemm_launch(e->pl_down[l], s) != RR_OK) return RR_CUDA_ERROR; ++nl;
        launch_add_rmsnorm(e->x, part_f32(e->part_down, e->s_down, B, d.hidden), (const __nv_bfloat16*)nw, e->xn, B,
                           d.hidden, d.rms_eps, s); ++nl;
    }
    if (gemm_launch(e->pl_head, s) != RR_OK) return RR_CUDA_ERROR; ++nl;
    launch_argmax(part_f32(e->logits, 1, B, d.vocab), B, d.vocab, e->d_tok, nullptr, e->d_slot, e->d_pos, s); ++nl;
    if (n_launch) *n_launch = nl;
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) { rr::note_cuda_error(err); return RR_CUDA_ERROR; }
    return RR_OK;
}

static int run_decode_step(rr_engine* e) {
    cudaStream_t s = e->stream;
    if (!e->warmed || !e->o.use_cuda_graph) {
        uint64_t nl = 0;
        int rc = enqueue_decode_step(e, s, &nl);
        if (rc != RR_OK) return rc;
        e->step_launches = nl;
        // NOTE: the warm-up step is a real step (it advances positions); graph capture follows.
        if (!e->warmed) {
            e->warmed = true;
            if (e->o.use_cuda_graph) {
                CK(cudaStreamSynchronize(s));
                // capture for subsequent steps
                cudaGraph_t g = nullptr;
                CK(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
                rc = enqueue_decode_step(e, s, nullptr);
                cudaError_t ce = cudaStreamEndCapture(s, &g);
                if (rc != RR_OK || ce != cudaSuccess) { rr::note_cuda_error(ce); return RR_CUDA_ERROR; }
                CK(cudaGraphInstantiate(&e->graph, g, 0));
                cudaGraphDestroy(g);
            }
        }
    } else {
        CK(cudaGraphLaunch(e->graph, s));
    }
    e->st.kernel_launches += e->step_launches;
    return RR_OK;
}

// ---------------------------------------------------------------- prefill chunk
static int get_pf_plans(rr_engine* e, int T, rr_engine::PfPlans** out) {
    auto it = e->pf_plans.find(T);
    if (it != e->pf_plans.end()) { *out = &it->second; return RR_OK; }
    const rr_model_desc& d = e->d;
    rr_engine::PfPlans P;
    const int L = d.n_layers;
    P.qkv.resize(L); P.o.resize(L); P.gu.resize(L); P.down.resize(L);
    for (int l = 0; l < L; ++l) {
        int rc = gemm_plan_init(&P.qkv[l], e->pxn, T, d.hidden, e->wqkv[l], e->nqkv, d.hidden, d.hidden, e->pqkv,
                                e->nqkv, 0, 1, e->fuse_rope_pf ? OUT_ROWMAJOR_ROPE : OUT_ROWMAJOR_BF16, 256);
        if (rc) return rc;
        if (e->fuse_rope_pf) {
            RopeEpi& r = P.qkv[l].rope;
            r.q_out = e->pq; r.k_cache = e->kcache + (size_t)l * e->kv_layer_stride;
            r.v_cache = e->vcache + (size_t)l * e->kv_layer_stride;
            r.slot = nullptr; r.pos = nullptr;                     // set per chunk (offsets inside the staging buffer)
            r.table = e->rope_table; r.n_heads = d.n_heads; r.n_kv_heads = d.n_kv_heads; r.ctx_max = e->o.ctx_max;
        }
        rc = gemm_plan_init(&P.o[l], e->pattn, T, e->nq, e->wo[l], d.hidden, e->nq, e->nq, e->px, d.hidden, 0, 1,
                            OUT_ROWMAJOR_RESID, 256);                  // residual add in the epilogue
        if (rc) return rc;
        if (e->defer_norm_pf) {
            auto consumer = [&](RopeEpi& r) {
                r.rowss = e->p_rowss; r.n_part = e->pf_parts; r.inv_hidden = 1.0f / (float)d.hidden; r.eps = d.rms_eps;
            };
            auto producer = [&](RopeEpi& r, const void* gamma) {
                r.gamma = (const __nv_bfloat16*)gamma; r.xhat = e->pxn; r.rowss_out = e->p_rowss; r.n_part_out = e->pf_parts;
            };
            consumer(P.qkv[l].rope);
            producer(P.o[l].rope, e->norm_mlp[l]);
        }
        if (e->fuse_silu)
            rc = gemm_plan_init(&P.gu[l], e->pxn, T, d.hidden, e->wgu[l], 2 * d.inter, d.hidden, d.hidden, e->pact,
                                d.inter, 0, 1, OUT_ROWMAJOR_SILU, 256);
        else
            rc = gemm_plan_init(&P.gu[l], e->pxn, T, d.hidden, e->wgu[l], 2 * d.inter, d.hidden, d.hidden, e->pgu,
                                2 * d.inter, 0, 1, OUT_ROWMAJOR_BF16, 256);
        if (rc) return rc;
        rc = gemm_plan_init(&P.down[l], e->pact, T, d.inter, e->wdown[l], d.hidden, d.inter, d.inter, e->px,
                            d.hidden, 0, 1, OUT_ROWMAJOR_RESID, 256);
        if (rc) return rc;
        if (e->defer_norm_pf) {
            RopeEpi& c = P.gu[l].rope;
            c.rowss = e->p_rowss; c.n_part = e->pf_parts; c.inv_hidden = 1.0f / (float)d.hidden; c.eps = d.rms_eps;
            RopeEpi& r = P.down[l].rope;
            r.gamma = (const __nv_bfloat16*)(l + 1 < L ? e->norm_attn[l + 1] : e->final_norm);
            r.xhat = e->pxn; r.rowss_out = e->p_rowss; r.n_part_out = e->pf_parts;
        }
    }
    auto ins = e->pf_plans.emplace(T, std::move(P));
    *out = &ins.first->second;
    return RR_OK;
}

// ids: T tokens of n_seqs prompts; slots[n_seqs]. Leaves first tokens in e->p_first (device) and
// activates the rows. Caller holds gpu_mu.
static int run_prefill(rr_engine* e, const int32_t* ids, const int32_t* seq_start, const int32_t* slots,
                       int n_seqs, int32_t* first_tok_host, float* logits_host) {
    const rr_model_desc& d = e->d;
    const int T = seq_start[n_seqs];
    if (T <= 0 || T > e->Tmax || n_seqs > e->Bm) return RR_INVALID_ARGUMENT;
    cudaStream_t s = e->stream;
    // pinned staging: ids[T] | pos[T] | slot_tok[T] | seq_start[n+1] | seq_slot[n] | last[n]
    int32_t* h = e->h_stage;
    int32_t *h_ids = h, *h_pos = h + T, *h_slt = h + 2 * T, *h_ss = h + 3 * T, *h_sl = h_ss + n_seqs + 1,
            *h_last = h_sl + n_seqs;
    int max_len = 0;
    memcpy(h_ids, ids, sizeof(int32_t) * T);
    for (int i = 0; i < n_seqs; ++i) {
        const int a = seq_start[i], b = seq_start[i + 1];
        if (b <= a || b - a + 1 > e->o.ctx_max || slots[i] < 0 || slots[i] >= e->Bm) return RR_INVALID_ARGUMENT;
        for (int t = a; t < b; ++t) { h_pos[t] = t - a; h_slt[t] = slots[i]; }
        h_ss[i] = a; h_sl[i] = slots[i]; h_last[i] = b - 1;
        if (b - a > max_len) max_len = b - a;
    }
    h_ss[n_seqs] = T;
    const size_t n_ints = (size_t)3 * T + 3 * n_seqs + 1;
    CK(cudaEventRecord(e->ev0, s));
    CK(cudaMemcpyAsync(e->p_ids, h, n_ints * sizeof(int32_t), cudaMemcpyHostToDevice, s));
    e->st.h2d_bytes += n_ints * sizeof(int32_t);
    int32_t *p_ids = e->p_ids, *p_pos = p_ids + T, *p_slt = p_ids + 2 * T, *p_ss = p_ids + 3 * T,
            *p_sl = p_ss + n_seqs + 1, *p_last = p_sl + n_seqs;

    // One set of plans (4 L TMA descriptors) built for Tmax rows; the live row count is a launch argument: TMA reads of
    // rows >= T stay inside the Tmax-row buffers and every store is guarded by rowsA.
    rr_engine::PfPlans* P = nullptr;
    int rc = get_pf_plans(e, e->Tmax, &P);
    if (rc != RR_OK) return rc;
    auto launch_rows = [&](const GemmPlan& pl) { GemmPlan q = pl; q.rowsA = T; return gemm_launch(q, s); };
    uint64_t nl = 0;
    launch_embed(p_ids, (const __nv_bfloat16*)e->embed, e->px, T, d.hidden, nullptr, s); ++nl;
    if (e->defer_norm_pf)       // layer 0's operand in the deferred form: bf16(x * gamma), sum(x^2) in partial 0
        launch_add_rmsnorm(e->px, part_none(), (const __nv_bfloat16*)e->norm_attn[0], e->pxn, T, d.hidden, d.rms_eps, s,
                           nullptr, 0, e->p_rowss, e->pf_parts);
    else
        launch_add_rmsnorm(e->px, part_none(), (const __nv_bfloat16*)e->norm_attn[0], e->pxn, T, d.hidden, d.rms_eps, s);
    ++nl;
    for (int l = 0; l < d.n_layers; ++l) {
        __nv_bfloat16* kc = e->kcache + (size_t)l * e->kv_layer_stride;
        __nv_bfloat16* vc = e->vcache + (size_t)l * e->kv_layer_stride;
        if (e->fuse_rope_pf) {
            P->qkv[l].rope.slot = p_slt; P->qkv[l].rope.pos = p_pos;
        }
        if (launch_rows(P->qkv[l]) != RR_OK) return RR_CUDA_ERROR; ++nl;
        RopeArgs ra;
        ra.qkv = part_bf16(e->pqkv, e->nqkv);
        ra.q_out = e->pq; ra.k_cache = kc; ra.v_cache = vc; ra.slot = p_slt; ra.pos = p_pos; ra.rows = T;
        ra.n_heads = d.n_heads; ra.n_kv_heads = d.n_kv_heads; ra.ctx_max = e->o.ctx_max; ra.theta = d.rope_theta;
        ra.table = e->rope_table; ra.head_dim = d.head_dim;
        if (!e->fuse_rope_pf) { launch_rope_kv(ra, s); ++nl; }
        PrefillAttnArgs pa = e->pf_attn[l];          // per-layer TMA maps made at create
        pa.q = e->pq; pa.k_cache = kc; pa.v_cache = vc; pa.out = e->pattn; pa.seq_start = p_ss; pa.seq_slot = p_sl;
        pa.n_seqs = n_seqs; pa.max_len = max_len; pa.n_heads = d.n_heads; pa.n_kv_heads = d.n_kv_heads;
        pa.ctx_max = e->o.ctx_max; pa.scale = 1.0f / sqrtf((float)d.head_dim); pa.head_dim = d.head_dim;
        if (launch_prefill_attn(pa, s) != RR_OK) return RR_CUDA_ERROR; ++nl;
        if (l + 1 == d.n_layers) {
            // ---- trimmed tail: n_seqs rows through O, MLP, final norm (decode-orientation kernels, decode buffers)
            const int B = e->Bm;
            launch_pdl(gather_last_kernel, dim3(n_seqs), dim3(256), 0, s, (const __nv_bfloat16*)e->pattn, (const float*)e->px,
                       (const int32_t*)p_last, e->attn_out, e->x, e->nq, d.hidden); ++nl;
            if (gemm_launch(e->pl_o[l], s) != RR_OK) return RR_CUDA_ERROR; ++nl;
            launch_add_rmsnorm(e->x, part_f32(e->part_o, e->s_o, B, d.hidden), (const __nv_bfloat16*)e->norm_mlp[l], e->xn,
                               n_seqs, d.hidden, d.rms_eps, s); ++nl;
            if (gemm_launch(e->pl_gu[l], s) != RR_OK) return RR_CUDA_ERROR; ++nl;
            if (!e->fuse_silu) { launch_silu_mul(part_f32(e->part_gu, e->s_gu, B, 2 * d.inter), e->act, n_seqs, d.inter, s); ++nl; }
            if (gemm_launch(e->pl_down[l], s) != RR_OK) return RR_CUDA_ERROR; ++nl;
            launch_add_rmsnorm(e->x, part_f32(e->part_down, e->s_down, B, d.hidden), (const __nv_bfloat16*)e->final_norm, e->xn,
                               n_seqs, d.hidden, d.rms_eps, s); ++nl;
            break;
        }
        if (launch_rows(P->o[l]) != RR_OK) return RR_CUDA_ERROR; ++nl;
        if (!e->defer_norm_pf) {
            launch_add_rmsnorm(e->px, part_none(), (const __nv_bfloat16*)e->norm_mlp[l], e->pxn, T,
                               d.hidden, d.rms_eps, s); ++nl;
        }
        if (launch_rows(P->gu[l]) != RR_OK) return RR_CUDA_ERROR; ++nl;
        if (!e->fuse_silu) { launch_silu_mul(part_bf16(e->pgu, 2 * d.inter), e->pact, T, d.inter, s); ++nl; }
        if (launch_rows(P->down[l]) != RR_OK) return RR_CUDA_ERROR; ++nl;
        if (!e->defer_norm_pf) {
            launch_add_rmsnorm(e->px, part_none(), (const __nv_bfloat16*)e->norm_attn[l + 1], e->pxn, T, d.hidden,
                               d.rms_eps, s); ++nl;
        }
    }
    if (gemm_launch(e->pl_head, s) != RR_OK) return RR_CUDA_ERROR; ++nl;      // B = e->xn (rows 0..n_seqs-1)
    launch_argmax(part_f32(e->logits, 1, e->Bm, d.vocab), n_seqs, d.vocab, e->p_first, nullptr, nullptr, nullptr, s); ++nl;
    launch_pdl(activate_rows_kernel, dim3((n_seqs + 127) / 128), dim3(128), 0, s, (const int32_t*)p_sl,
               (const int32_t*)e->p_first, (const int32_t*)p_ss, n_seqs, e->d_tok, e->d_pos, e->d_slot); ++nl;
    CK(cudaMemcpyAsync(e->h_tok, e->p_first, sizeof(int32_t) * n_seqs, cudaMemcpyDeviceToHost, s));
    e->st.d2h_bytes += sizeof(int32_t) * n_seqs;
    if (logits_host) {
        CK(cudaMemcpyAsync(logits_host, e->logits, sizeof(float) * (size_t)n_seqs * d.vocab, cudaMemcpyDeviceToHost, s));
    }
    CK(cudaEventRecord(e->ev1, s));
    CK(cudaStreamSynchronize(s));
    float ms = 0;
    cudaEventElapsedTime(&ms, e->ev0, e->ev1);
    e->st.prefill_ms_total += ms;
    e->st.prefill_chunks += 1;
    e->st.prefill_tokens += T;
    e->st.kernel_launches += nl;
    for (int i = 0; i < n_seqs; ++i) {
        if (first_tok_host) first_tok_host[i] = e->h_tok[i];
        e->h_slot_mirror[slots[i]] = slots[i];
    }
    return RR_OK;
}

// ---------------------------------------------------------------- worker (continuous batching)
struct DoneNote { uint64_t tag, ticket; int status, n_gen; };

// Caller holds e->mu.  Returns the hook call to make once the lock is released (tag == 0 and no hook: nothing).
static void finish_request(rr_engine* e, Request* r, int status, std::vector<DoneNote>* notes = nullptr) {
    r->status = status;
    r->t_done = now_s(e);
    r->done = true;
    if (notes && e->hook) notes->push_back(DoneNote{r->tag, r->ticket, status, (int)r->out.size()});
    if (r->detached) {                   // cancelled by its owner: nobody waits for it
        e->table.erase(r->ticket);
        delete r;
    }
}
static void run_hooks(rr_engine* e, std::vector<DoneNote>& notes) {
    for (const DoneNote& n : notes) e->hook(e->hook_ctx, n.tag, n.ticket, n.status, n.n_gen);
    notes.clear();
}

static void worker_main(rr_engine* e) {
    cudaSetDevice(e->o.device);
    std::vector<int32_t> ids, seq_start, slots;
    std::vector<Request*> chunk;
    std::vector<DoneNote> notes;
    while (!e->stop.load()) {
        run_hooks(e, notes);
        // ---- admit waiting requests into free rows (prefill has priority: best TTFT)
        chunk.clear(); ids.clear(); seq_start.assign(1, 0); slots.clear();
        int active = 0;
        {
            std::unique_lock<std::mutex> lk(e->mu);
            for (int b = 0; b < e->Bm; ++b) {
                Request* r = e->row_req[b];
                if (r && r->cancel) {                      // rr_engine_cancel: free the row, keep what was generated
                    e->row_req[b] = nullptr; e->h_slot_mirror[b] = -1; e->slots_dirty = true;
                    finish_request(e, r, RR_CANCELLED, &notes);
                    continue;
                }
                active += r != nullptr;
            }
            if (e->waiting.empty() && active == 0) {
                e->cv_work.wait_for(lk, std::chrono::milliseconds(50));
                continue;
            }
            int b = 0;
            while (!e->waiting.empty()) {
                Request* r = e->waiting.front();
                if ((int)ids.size() + (int)r->prompt.size() > e->Tmax) break;
                while (b < e->Bm && e->row_req[b] != nullptr) ++b;
                if (b >= e->Bm) break;
                e->waiting.pop_front();
                e->row_req[b] = r;
                r->slot = b;
                chunk.push_back(r);
                slots.push_back(b);
                ids.insert(ids.end(), r->prompt.begin(), r->prompt.end());
                seq_start.push_back((int)ids.size());
                ++active;
            }
            e->st.queued = (int)e->waiting.size();
            e->st.active_rows = active;
        }
        std::lock_guard<std::mutex> gl(e->gpu_mu);
        std::lock_guard<std::mutex> dl(device_mutex(e->o.device));
        if (!chunk.empty()) {
            int rc = run_prefill(e, ids.data(), seq_start.data(), slots.data(), (int)chunk.size(), nullptr, nullptr);
            const double t = now_s(e);
            std::lock_guard<std::mutex> lk(e->mu);
            for (size_t i = 0; i < chunk.size(); ++i) {
                Request* r = chunk[i];
                if (rc != RR_OK) {
                    e->row_req[r->slot] = nullptr;
                    e->h_slot_mirror[r->slot] = -1; e->slots_dirty = true;
                    finish_request(e, r, RR_INTERNAL, &notes);
                    continue;
                }
                r->t_first = t;
                r->out.push_back(e->h_tok[i]);
                e->st.generated_tokens += 1;
                if ((int)r->out.size() >= r->max_new) {
                    e->row_req[r->slot] = nullptr;
                    e->h_slot_mirror[r->slot] = -1; e->slots_dirty = true;
                    finish_request(e, r, RR_OK, &notes);
                }
            }
            e->cv_done.notify_all();
            continue;   // look for more waiting prompts before decoding
        }
        if (active == 0) continue;
        // ---- one decode step for all active rows
        cudaStream_t s = e->stream;
        if (e->slots_dirty) {
            memcpy(e->h_stage, e->h_slot_mirror.data(), sizeof(int32_t) * e->Bm);
            cudaMemcpyAsync(e->d_slot, e->h_stage, sizeof(int32_t) * e->Bm, cudaMemcpyHostToDevice, s);
            e->st.h2d_bytes += sizeof(int32_t) * e->Bm;
            e->slots_dirty = false;
        }
        cudaEventRecord(e->ev0, s);
        int rc = run_decode_step(e);
        cudaEventRecord(e->ev1, s);
        cudaMemcpyAsync(e->h_tok, e->d_tok, sizeof(int32_t) * e->Bm, cudaMemcpyDeviceToHost, s);
        cudaError_t se = cudaStreamSynchronize(s);
        e->st.d2h_bytes += sizeof(int32_t) * e->Bm;
        if (se != cudaSuccess) { rr::note_cuda_error(se); rc = RR_CUDA_ERROR; }
        float ms = 0;
        cudaEventElapsedTime(&ms, e->ev0, e->ev1);
        e->st.decode_ms_total += ms;
        e->st.decode_steps += 1;
        {
            std::lock_guard<std::mutex> lk(e->mu);
            for (int b = 0; b < e->Bm; ++b) {
                Request* r = e->row_req[b];
                if (!r) continue;
                if (rc != RR_OK) {
                    e->row_req[b] = nullptr; e->h_slot_mirror[b] = -1; e->slots_dirty = true;
                    finish_request(e, r, RR_INTERNAL, &notes);
                    continue;
                }
                r->out.push_back(e->h_tok[b]);
                e->st.generated_tokens += 1;
                if ((int)r->out.size() >= r->max_new) {
                    e->row_req[b] = nullptr; e->h_slot_mirror[b] = -1; e->slots_dirty = true;
                    finish_request(e, r, RR_OK, &notes);
                }
            }
        }
        e->cv_done.notify_all();
    }
    run_hooks(e, notes);
}

// ---------------------------------------------------------------- C-ABI
RR_API int rr_engine_create(const rr_model_desc* desc, const rr_model_weights* w, const rr_engine_opts* opts,
                            rr_engine** out) {
    if (!desc || !w || !opts || !out) return RR_INVALID_ARGUMENT;
    const rr_model_desc& d = *desc;
    // head_dim: 64..128, multiple of 16; attention operands (q, KV cache rows) are zero-padded to 128
    if (d.head_dim < 64 || d.head_dim > 128 || d.head_dim % 16 || d.n_heads % d.n_kv_heads || d.hidden % 64 ||
        d.inter % 64 || d.n_layers < 1)
        return RR_INVALID_ARGUMENT;
    const int G = d.n_heads / d.n_kv_heads;
    if (!(G == 1 || G == 2 || G == 4 || G == 8)) return RR_INVALID_ARGUMENT;
    if (d.hidden > 8192) return RR_INVALID_ARGUMENT;      // add_rmsnorm_kernel keeps one row in registers (rr_elementwise.cu)
    if (opts->max_batch < 1 || opts->max_batch > 256 || opts->ctx_max < 64 || opts->ctx_max % 64)
        return RR_INVALID_ARGUMENT;
    CK(cudaSetDevice(opts->device));
    rr_engine* e = new (std::nothrow) rr_engine();
    if (!e) return RR_INTERNAL;
    e->d = d; e->o = *opts;
    e->Bm = opts->max_batch;
    e->bn_dec = pick_bn(e->Bm);
    e->nq = d.n_heads * d.head_dim; e->nkv_dim = d.n_kv_heads * d.head_dim; e->nqkv = e->nq + 2 * e->nkv_dim;
    e->Tmax = opts->max_prefill_tokens > 0 ? opts->max_prefill_tokens : 8192;
    if (e->Tmax < 16) e->Tmax = 16;
    e->embed = w->embed; e->lm_head = w->lm_head; e->final_norm = w->final_norm;
    const int L = d.n_layers;
    for (int l = 0; l < L; ++l) {
        e->wqkv.push_back(w->wqkv[l]); e->wo.push_back(w->wo[l]); e->wgu.push_back(w->wgu[l]);
        e->wdown.push_back(w->wdown[l]); e->norm_attn.push_back(w->norm_attn[l]); e->norm_mlp.push_back(w->norm_mlp[l]);
    }
    memset(&e->st, 0, sizeof(e->st));
    e->t0 = std::chrono::steady_clock::now();
    int rc = RR_OK;
#define TRY(x) do { rc = (x); if (rc != RR_OK) { rr_engine_destroy(e); return rc; } } while (0)
#define TRYC(x) do { cudaError_t e__ = (x); if (e__ != cudaSuccess) { rr::note_cuda_error(e__); rr_engine_destroy(e); return RR_CUDA_ERROR; } } while (0)
    TRYC(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
    TRYC(cudaEventCreate(&e->ev0));
    TRYC(cudaEventCreate(&e->ev1));
    const int B = e->Bm;
    // Uniform split-K planes.
    e->s_qkv = pick_splits(e->nqkv, d.hidden); e->s_o = pick_splits(d.hidden, e->nq);
    e->s_gu = pick_splits(2 * d.inter, d.hidden); e->s_down = pick_splits(d.hidden, d.inter);
    e->fuse_silu = (w->flags & RR_WEIGHTS_WGU_INTERLEAVED64) && e->s_gu == 1 && e->bn_dec >= 32 &&
                   (2 * d.inter) % 128 == 0;
    if ((w->flags & RR_WEIGHTS_WGU_INTERLEAVED64) && !e->fuse_silu) { rr_engine_destroy(e); return RR_INVALID_ARGUMENT; }
    TRY(dalloc(e, &e->d_tok, B)); TRY(dalloc(e, &e->d_pos, B)); TRY(dalloc(e, &e->d_slot, B));
    TRYC(cudaMemset(e->d_slot, 0xff, sizeof(int32_t) * B));
    TRY(dalloc(e, &e->x, (size_t)B * d.hidden));
    TRY(dalloc(e, &e->xn, (size_t)B * d.hidden));
    TRY(dalloc(e, &e->qbuf, (size_t)B * d.n_heads * 128));
    TRY(dalloc(e, &e->attn_out, (size_t)B * e->nq));
    TRY(dalloc(e, &e->act, (size_t)B * d.inter));
    TRY(dalloc(e, &e->part_qkv, (size_t)e->s_qkv * B * e->nqkv));
    TRY(dalloc(e, &e->part_o, (size_t)e->s_o * B * d.hidden));
    TRY(dalloc(e, &e->part_gu, (size_t)e->s_gu * B * 2 * d.inter));
    // fused decode MLP: the down GEMM's K range in <= 8 slices (one output plane each); 8 x 28 k-blocks for
    // Llama-3-8B balances the per-CTA lists to within 5 % (see mlp_schedule)
    {
        const int kb1n = d.inter / 64;
        int n_sl = (kb1n + 15) / 16;
        n_sl = n_sl > 8 ? 8 : (n_sl < 1 ? 1 : n_sl);
        e->mlp_slice_kb = (kb1n + n_sl - 1) / n_sl;
        n_sl = (kb1n + e->mlp_slice_kb - 1) / e->mlp_slice_kb;
        e->fuse_mlp = e->fuse_silu && opts->reserved[2] == 0 && d.inter % 64 == 0 && kb1n >= 1 && !getenv("RR_NO_MLP_FUSE");
        e->mlp_slices = e->fuse_mlp ? n_sl : 0;
    }
    TRY(dalloc(e, &e->part_down, (size_t)(e->s_down > e->mlp_slices ? e->s_down : e->mlp_slices) * B * d.hidden));
    TRY(dalloc(e, &e->logits, (size_t)B * d.vocab));
    TRY(dalloc(e, &e->xn_last, (size_t)B * d.hidden));
    TRY(dalloc(e, &e->rope_table, (size_t)opts->ctx_max * 64));
    launch_rope_table(e->rope_table, opts->ctx_max, d.rope_theta, d.head_dim, e->stream);
    e->kv_layer_stride = (size_t)B * d.n_kv_heads * opts->ctx_max * 128;
    TRY(dalloc(e, &e->kcache, e->kv_layer_stride * L));
    TRY(dalloc(e, &e->vcache, e->kv_layer_stride * L));
    {   // split-KV only when the grid would not fill the GPU
        int ctas = B * d.n_kv_heads;
        int ks = 1;
        while (ctas * ks < 2 * num_sms() && ks < 8) ks *= 2;
        e->kv_splits = ks;
        e->attn_ws = nullptr;
        if (ks > 1) TRY(dalloc(e, &e->attn_ws, decode_attn_ws_bytes(B, d.n_heads, ks) / sizeof(float)));
    }
    const int T = e->Tmax;
    TRY(dalloc(e, &e->p_ids, (size_t)3 * T + 3 * B + 8));
    TRY(dalloc(e, &e->p_first, B));
    TRY(dalloc(e, &e->px, (size_t)T * d.hidden, false));
    TRY(dalloc(e, &e->pxn, (size_t)T * d.hidden, false));
    TRY(dalloc(e, &e->pqkv, (size_t)T * e->nqkv, false));
    TRY(dalloc(e, &e->pq, (size_t)T * d.n_heads * 128));                 // zeroed: columns beyond head_dim stay 0
    TRY(dalloc(e, &e->pattn, (size_t)T * e->nq, false));
    TRY(dalloc(e, &e->po, (size_t)T * d.hidden, false));
    TRY(dalloc(e, &e->pgu, (size_t)T * 2 * d.inter, false));
    TRY(dalloc(e, &e->pact, (size_t)T * d.inter, false));
    e->h_stage_ints = (size_t)3 * T + 3 * B + 8;
    TRYC(cudaMallocHost(&e->h_stage, e->h_stage_ints * sizeof(int32_t)));
    TRYC(cudaMallocHost(&e->h_tok, sizeof(int32_t) * (B > 16 ? B : 16)));

    e->pl_qkv.resize(L); e->pl_o.resize(L); e->pl_gu.resize(L); e->pl_down.resize(L);
    e->attn_args.resize(L);
    e->pf_attn.resize(L);
    for (int l = 0; l < L; ++l) {
        {
            PrefillAttnArgs& pa = e->pf_attn[l];
            pa.q = e->pq; pa.k_cache = e->kcache + (size_t)l * e->kv_layer_stride;
            pa.v_cache = e->vcache + (size_t)l * e->kv_layer_stride; pa.n_heads = d.n_heads;
            pa.n_kv_heads = d.n_kv_heads; pa.ctx_max = opts->ctx_max; pa.head_dim = d.head_dim;
            TRY(prefill_attn_make_maps(&pa, T, (long long)B * d.n_kv_heads * opts->ctx_max));   // ctx_max % 64 == 0 (checked above)
        }
        DecodeAttnArgs& da = e->attn_args[l];
        da.q = e->qbuf; da.k_cache = e->kcache + (size_t)l * e->kv_layer_stride;
        da.v_cache = e->vcache + (size_t)l * e->kv_layer_stride; da.out = e->attn_out; da.slot = e->d_slot;
        da.pos = e->d_pos; da.rows = B; da.n_heads = d.n_heads; da.n_kv_heads = d.n_kv_heads;
        da.ctx_max = opts->ctx_max; da.scale = 1.0f / sqrtf((float)d.head_dim); da.ws = e->attn_ws;
        da.kv_splits = e->kv_splits;
        da.fuse_rope = 1; da.qkv = part_f32(e->part_qkv, e->s_qkv, B, e->nqkv); da.rope_table = e->rope_table;
        da.head_dim = d.head_dim;
        TRY(decode_attn_make_maps(&da, B));
        TRY(gemm_plan_init(&e->pl_qkv[l], e->wqkv[l], e->nqkv, d.hidden, e->xn, B, d.hidden, d.hidden, e->part_qkv,
                           e->nqkv, B, e->s_qkv, OUT_TRANSPOSED_F32, e->bn_dec));
        TRY(gemm_plan_init(&e->pl_o[l], e->wo[l], d.hidden, e->nq, e->attn_out, B, e->nq, e->nq, e->part_o, d.hidden,
                           B, e->s_o, OUT_TRANSPOSED_F32, e->bn_dec));
        if (e->fuse_silu)
            TRY(gemm_plan_init(&e->pl_gu[l], e->wgu[l], 2 * d.inter, d.hidden, e->xn, B, d.hidden, d.hidden, e->act,
                               d.inter, B, 1, OUT_TRANSPOSED_SILU, e->bn_dec));
        else
            TRY(gemm_plan_init(&e->pl_gu[l], e->wgu[l], 2 * d.inter, d.hidden, e->xn, B, d.hidden, d.hidden, e->part_gu,
                               2 * d.inter, B, e->s_gu, OUT_TRANSPOSED_F32, e->bn_dec));
        TRY(gemm_plan_init(&e->pl_down[l], e->wdown[l], d.hidden, d.inter, e->act, B, d.inter, d.inter, e->part_down,
                           d.hidden, B, e->s_down, OUT_TRANSPOSED_F32, e->bn_dec));
    }
    TRY(gemm_plan_init(&e->pl_head, e->lm_head, d.vocab, d.hidden, e->xn, B, d.hidden, d.hidden, e->logits, d.vocab,
                       B, 1, OUT_TRANSPOSED_F32, e->bn_dec));
    TRY(gemm_plan_init(&e->pl_head_pf, e->lm_head, d.vocab, d.hidden, e->xn_last, B, d.hidden, d.hidden, e->logits,
                       d.vocab, B, 1, OUT_TRANSPOSED_F32, e->bn_dec));
    e->fuse_rope_pf = d.head_dim == 128 && opts->reserved[1] == 0;
    e->pf_parts = (d.hidden + 255) / 256;
    // On by default (reserved[3] = 1 or RR_NO_DEFER_NORM=1 restores the two norm kernels per layer).  In-process A/B
    // (tools/prefill_ab.py): 91.0 -> 85.2 ms per 8192-token chunk once the residual epilogue became line-coalesced;
    // with the earlier row-per-thread epilogue the same fusion LOST 1.4 % (o-proj +35 %).
    e->defer_norm_pf = opts->reserved[3] == 0 && !getenv("RR_NO_DEFER_NORM") && d.hidden % 8 == 0 && e->pf_parts <= 64;
    if (e->defer_norm_pf) TRY(dalloc(e, &e->p_rowss, (size_t)e->Tmax * e->pf_parts));
    if (e->fuse_mlp) {
        std::vector<MlpItem> sched;
        const int grid = num_sms();
        const int dyn = getenv("RR_MLP_STATIC") ? 0 : 1;      // down items dealt by the kernel (default) or by the host list schedule
        const int max_items = mlp_schedule(grid, d.inter, d.hidden, e->mlp_slice_kb, &sched, dyn);
        TRY(dalloc(e, &e->mlp_items, sched.size()));
        TRYC(cudaMemcpy(e->mlp_items, sched.data(), sched.size() * sizeof(MlpItem), cudaMemcpyHostToDevice));
        TRY(dalloc(e, &e->mlp_ready, 16));
        e->mlp.resize(L);
        for (int l = 0; l < L; ++l) {
            TRY(mlp_plan_init(&e->mlp[l], e->wgu[l], e->wdown[l], d.inter, d.hidden, e->xn, B, e->act, e->part_down, B,
                              e->bn_dec, e->mlp_items, max_items, grid, e->mlp_ready, e->mlp_slice_kb, dyn));
        }
    }
    TRYC(cudaDeviceSynchronize());
    e->row_req.assign(B, nullptr);
    e->h_slot_mirror.assign(B, -1);
    e->worker = std::thread(worker_main, e);
    *out = e;
    return RR_OK;
#undef TRY
#undef TRYC
}

RR_API void rr_engine_destroy(rr_engine* e) {
    if (!e) return;
    e->stop.store(true);
    e->cv_work.notify_all();
    if (e->worker.joinable()) e->worker.join();
    cudaSetDevice(e->o.device);
    if (e->stream) cudaStreamSynchronize(e->stream);
    if (e->graph) cudaGraphExecDestroy(e->graph);
    for (void* p : e->allocs) cudaFree(p);
    if (e->h_stage) cudaFreeHost(e->h_stage);
    if (e->h_tok) cudaFreeHost(e->h_tok);
    if (e->ev0) cudaEventDestroy(e->ev0);
    if (e->ev1) cudaEventDestroy(e->ev1);
    if (e->stream) cudaStreamDestroy(e->stream);
    for (auto& kv : e->table) delete kv.second;
    delete e;
}

RR_API int rr_engine_prefill(rr_engine* e, const int32_t* ids, const int32_t* seq_start, const int32_t* slots,
                             int n_seqs, int32_t* first_tok, float* logits_out) {
    if (!e || !ids || !seq_start || !slots || n_seqs < 1) return RR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> gl(e->gpu_mu);
    std::lock_guard<std::mutex> dl(device_mutex(e->o.device));
    CK(cudaSetDevice(e->o.device));
    return run_prefill(e, ids, seq_start, slots, n_seqs, first_tok, logits_out);
}

RR_API int rr_engine_decode_step(rr_engine* e, const int32_t* slots, const int32_t* tok, const int32_t* pos, int n,
                                 int32_t* next_tok, float* logits_out) {
    if (!e || !slots || !tok || !pos || n < 1 || n > e->Bm || !next_tok) return RR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> gl(e->gpu_mu);
    std::lock_guard<std::mutex> dl(device_mutex(e->o.device));
    CK(cudaSetDevice(e->o.device));
    const int B = e->Bm;
    int32_t* h = e->h_stage;                 // tok[B] | pos[B] | slot[B]
    for (int b = 0; b < B; ++b) { h[b] = 0; h[B + b] = 0; h[2 * B + b] = -1; }
    for (int i = 0; i < n; ++i) {
        const int s = slots[i];
        if (s < 0 || s >= B || pos[i] < 0 || pos[i] >= e->o.ctx_max) return RR_INVALID_ARGUMENT;
        h[s] = tok[i]; h[B + s] = pos[i]; h[2 * B + s] = s;
    }
    cudaStream_t st = e->stream;
    CK(cudaMemcpyAsync(e->d_tok, h, sizeof(int32_t) * B, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(e->d_pos, h + B, sizeof(int32_t) * B, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(e->d_slot, h + 2 * B, sizeof(int32_t) * B, cudaMemcpyHostToDevice, st));
    uint64_t nl = 0;
    int rc = enqueue_decode_step(e, st, &nl);
    if (rc != RR_OK) return rc;
    e->st.kernel_launches += nl;
    CK(cudaMemcpyAsync(e->h_tok, e->d_tok, sizeof(int32_t) * B, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    for (int i = 0; i < n; ++i) {
        next_tok[i] = e->h_tok[slots[i]];
        if (logits_out)
            CK(cudaMemcpy(logits_out + (size_t)i * e->d.vocab, e->logits + (size_t)slots[i] * e->d.vocab,
                          sizeof(float) * e->d.vocab, cudaMemcpyDeviceToHost));
    }
    // leave the rows inactive for the serving loop
    CK(cudaMemsetAsync(e->d_slot, 0xff, sizeof(int32_t) * B, st));
    CK(cudaStreamSynchronize(st));
    for (int b = 0; b < B; ++b) e->h_slot_mirror[b] = -1;
    return RR_OK;
}

static bool injected_failure(const rr_engine* e, uint64_t ticket) {
    if (e->o.fail_prob <= 0.f) return false;
    uint64_t z = ticket + 0x9E3779B97F4A7C15ull * (uint64_t)(uint32_t)(e->o.fail_seed + 1);   // splitmix64
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    z ^= z >> 31;
    return (double)(z >> 11) * (1.0 / 9007199254740992.0) < (double)e->o.fail_prob;
}

namespace rr {
int engine_submit_tagged(rr_engine* e, const int32_t* prompt_ids, int n_prompt, int max_new_tokens, uint64_t tag,
                         uint64_t* ticket) {
    if (!e || !prompt_ids || !ticket || n_prompt < 1 || max_new_tokens < 1) return RR_INVALID_ARGUMENT;
    if (n_prompt + max_new_tokens > e->o.ctx_max || n_prompt > e->Tmax) return RR_INVALID_ARGUMENT;
    for (int i = 0; i < n_prompt; ++i)
        if (prompt_ids[i] < 0 || prompt_ids[i] >= e->d.vocab) return RR_INVALID_ARGUMENT;
    Request* r = new (std::nothrow) Request();
    if (!r) return RR_INTERNAL;
    r->prompt.assign(prompt_ids, prompt_ids + n_prompt);
    r->max_new = max_new_tokens;
    r->out.reserve(max_new_tokens);
    r->tag = tag;
    std::vector<DoneNote> notes;
    {
        std::lock_guard<std::mutex> lk(e->mu);
        r->ticket = e->next_ticket++;
        r->t_submit = now_s(e);
        e->table[r->ticket] = r;
        *ticket = r->ticket;
        if (injected_failure(e, r->ticket)) {
            r->t_first = r->t_submit;
            finish_request(e, r, RR_BACKEND_FAILED, &notes);
        } else {
            e->waiting.push_back(r);
        }
    }
    e->cv_work.notify_one();
    e->cv_done.notify_all();
    run_hooks(e, notes);
    return RR_OK;
}
void engine_set_done_hook(rr_engine* e, EngineDoneHook fn, void* ctx) {
    std::lock_guard<std::mutex> lk(e->mu);
    e->hook = fn; e->hook_ctx = ctx;
}
int engine_limits(const rr_engine* e, int* ctx_max, int* max_prefill, int* vocab) {
    if (!e) return RR_INVALID_ARGUMENT;
    if (ctx_max) *ctx_max = e->o.ctx_max;
    if (max_prefill) *max_prefill = e->Tmax;
    if (vocab) *vocab = e->d.vocab;
    return RR_OK;
}
}  // namespace rr

RR_API int rr_engine_submit(rr_engine* e, const int32_t* prompt_ids, int n_prompt, int max_new_tokens,
                            uint64_t* ticket) {
    return rr::engine_submit_tagged(e, prompt_ids, n_prompt, max_new_tokens, 0, ticket);
}

// Abandon a request (client gone / timed out): a queued request is dropped, a running one gives up its decode row at the
// next step; a finished one is just freed.  The ticket is consumed: do not wait on it afterwards.
RR_API int rr_engine_cancel(rr_engine* e, uint64_t ticket) {
    if (!e) return RR_INVALID_ARGUMENT;
    std::vector<DoneNote> notes;
    {
        std::lock_guard<std::mutex> lk(e->mu);
        auto it = e->table.find(ticket);
        if (it == e->table.end()) return RR_INVALID_ARGUMENT;
        Request* r = it->second;
        if (r->done) {
            e->table.erase(it);
            delete r;
        } else {
            r->detached = true;
            bool queued = false;
            for (auto q = e->waiting.begin(); q != e->waiting.end(); ++q)
                if (*q == r) { e->waiting.erase(q); queued = true; break; }
            if (queued) finish_request(e, r, RR_CANCELLED, &notes);      // frees it (detached)
            else r->cancel = true;                                       // active row: the worker drops it
        }
    }
    e->cv_work.notify_one();
    e->cv_done.notify_all();
    run_hooks(e, notes);
    return RR_OK;
}

// Streaming support: block until the request has more than `have` tokens (or is done / the wait times out), then
// copy the tokens generated so far.  Does not consume the request; finish with rr_engine_wait.
RR_API int rr_engine_peek(rr_engine* e, uint64_t ticket, int have, double timeout_s, int32_t* tokens_out,
                          int max_tokens_out, int32_t* n_generated, int32_t* done, double* t_first_token_s) {
    if (!e || !n_generated || !done) return RR_INVALID_ARGUMENT;
    std::unique_lock<std::mutex> lk(e->mu);
    const auto deadline = std::chrono::steady_clock::now() +
                          std::chrono::duration<double>(timeout_s > 0 ? timeout_s : 1e9);
    Request* r = nullptr;
    for (;;) {
        // looked up again after every wake-up: another thread may have consumed (wait) or cancelled the ticket meanwhile
        auto it = e->table.find(ticket);
        if (it == e->table.end()) return RR_INVALID_ARGUMENT;
        r = it->second;
        if (r->done || (int)r->out.size() > have) break;
        if (e->cv_done.wait_until(lk, deadline) == std::cv_status::timeout) {
            it = e->table.find(ticket);
            if (it == e->table.end()) return RR_INVALID_ARGUMENT;
            r = it->second;
            break;
        }
    }
    const int n = (int)r->out.size();
    *n_generated = n;
    *done = r->done ? 1 : 0;
    if (t_first_token_s) *t_first_token_s = r->t_first - r->t_submit;
    if (tokens_out) {
        const int m = n < max_tokens_out ? n : max_tokens_out;
        memcpy(tokens_out, r->out.data(), sizeof(int32_t) * m);
    }
    return RR_OK;
}

RR_API int rr_engine_wait(rr_engine* e, uint64_t ticket, double timeout_s, rr_completion* out, int32_t* tokens_out,
                          int max_tokens_out) {
    if (!e || !out) return RR_INVALID_ARGUMENT;
    std::unique_lock<std::mutex> lk(e->mu);
    const auto deadline = std::chrono::steady_clock::now() +
                          std::chrono::duration<double>(timeout_s > 0 ? timeout_s : 1e9);
    Request* r = nullptr;
    for (;;) {
        auto it = e->table.find(ticket);
        if (it == e->table.end()) return RR_INVALID_ARGUMENT;      // unknown, already consumed, or cancelled
        r = it->second;
        if (r->done) break;
        if (e->cv_done.wait_until(lk, deadline) == std::cv_status::timeout) {
            it = e->table.find(ticket);
            if (it == e->table.end()) return RR_INVALID_ARGUMENT;
            if (it->second->done) { r = it->second; break; }
            out->ticket = ticket; out->status = RR_TIMEOUT;
            return RR_TIMEOUT;   // the request stays in flight: wait again, or rr_engine_cancel
        }
    }
    out->ticket = ticket; out->status = r->status; out->n_prompt = (int)r->prompt.size();
    out->n_generated = (int)r->out.size(); out->reserved = 0;
    out->t_submit_s = r->t_submit; out->t_first_token_s = r->t_first; out->t_done_s = r->t_done;
    if (tokens_out) {
        const int n = (int)r->out.size() < max_tokens_out ? (int)r->out.size() : max_tokens_out;
        memcpy(tokens_out, r->out.data(), sizeof(int32_t) * n);
    }
    const int status = r->status;
    e->table.erase(ticket);
    delete r;
    return status == RR_OK ? RR_OK : status;
}

RR_API int rr_engine_run_batch(rr_engine* e, const int32_t* prompt_ids, const int32_t* prompt_start, int n_requests,
                               int max_new_tokens, rr_completion* out, int32_t* tokens_out) {
    if (!e || !prompt_ids || !prompt_start || n_requests < 1 || !out) return RR_INVALID_ARGUMENT;
    std::vector<uint64_t> tk(n_requests);
    for (int i = 0; i < n_requests; ++i) {
        int rc = rr_engine_submit(e, prompt_ids + prompt_start[i], prompt_start[i + 1] - prompt_start[i],
                                  max_new_tokens, &tk[i]);
        if (rc != RR_OK) return rc;
    }
    int worst = RR_OK;
    for (int i = 0; i < n_requests; ++i) {
        int rc = rr_engine_wait(e, tk[i], 0, &out[i], tokens_out ? tokens_out + (size_t)i * max_new_tokens : nullptr,
                                max_new_tokens);
        if (rc != RR_OK) worst = rc;
    }
    return worst;
}

RR_API double rr_engine_now(rr_engine* e) { return e ? now_s(e) : 0.0; }

RR_API int rr_engine_get_stats(rr_engine* e, rr_engine_stats* out) {
    if (!e || !out) return RR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> gl(e->gpu_mu);      // the worker updates the counters while it holds gpu_mu (then mu)
    std::lock_guard<std::mutex> lk(e->mu);
    *out = e->st;
    return RR_OK;
}

RR_API int rr_engine_reset_stats(rr_engine* e) {
    if (!e) return RR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> gl(e->gpu_mu);
    std::lock_guard<std::mutex> lk(e->mu);
    memset(&e->st, 0, sizeof(e->st));
    return RR_OK;
}
