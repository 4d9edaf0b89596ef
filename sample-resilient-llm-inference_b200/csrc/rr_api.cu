// rr_api.cu — extern "C" surface of librr_b200.so for the kernel-level entry points
// (include/rr_b200.h §2, §3).  Router: rr_router.cu.  Engine: rr_engine.cu.
#include "rr_kernels.h"
#include <vector>

#include <string.h>

#define RR_API extern "C" __attribute__((visibility("default")))

#include <stdlib.h>

namespace rr {
int g_use_pdl = getenv("RR_NO_PDL") ? 0 : 1;
thread_local char g_last_cuda_error[256] = "";
void note_cuda_error(cudaError_t e) {
    if (e != cudaSuccess) {
        strncpy(g_last_cuda_error, cudaGetErrorString(e), sizeof(g_last_cuda_error) - 1);
    }
}
int check_last(void) {
    cudaError_t e = cudaGetLastError();
    note_cuda_error(e);
    return e == cudaSuccess ? RR_OK : RR_CUDA_ERROR;
}
}  // namespace rr

using namespace rr;

RR_API const char* rr_version(void) { return "rr_b200 0.1 (sm_100a)"; }

RR_API const char* rr_strerror(int rc) {
    switch (rc) {
        case RR_OK: return "ok";
        case RR_RATE_LIMITED: return "rate limited (429)";
        case RR_NO_GROUP: return "unknown model group";
        case RR_INTERNAL: return "internal error";
        case RR_INVALID_ARGUMENT: return "invalid argument";
        case RR_CUDA_ERROR: return "CUDA error";
        case RR_TIMEOUT: return "timeout";
        case RR_BACKEND_FAILED: return "backend failed";
        case RR_CANCELLED: return "cancelled";
    }
    return "unknown";
}

RR_API const char* rr_last_cuda_error(void) { return g_last_cuda_error; }

namespace rr {
void rr_trace_set_gemm(unsigned long long*);
void rr_trace_set_attn_decode(unsigned long long*);
void rr_trace_set_attn_tc(unsigned long long*);
void rr_trace_set_elementwise(unsigned long long*);
void rr_trace_set_gemm_detail(int);
void rr_trace_set_attn_decode_detail(int);
}
static unsigned long long* g_trace_dev = nullptr;
static int g_trace_cap = 0;
static int g_trace_detail_on = 0;

// Debug timeline: (kernel id, start ns, dependency-resolved ns, end ns) of CTA 0 of every library kernel (globaltimer).
RR_API int rr_debug_trace_start(int max_entries) {
    if (max_entries < 1) return RR_INVALID_ARGUMENT;
    if (g_trace_dev) cudaFree(g_trace_dev);
    const size_t n = 2 + 4 * (size_t)max_entries;
    if (cudaMalloc(&g_trace_dev, n * 8) != cudaSuccess) return RR_CUDA_ERROR;
    cudaMemset(g_trace_dev, 0, n * 8);
    unsigned long long cap = (unsigned long long)max_entries;
    cudaMemcpy(g_trace_dev + 1, &cap, 8, cudaMemcpyHostToDevice);
    g_trace_cap = max_entries;
    rr_trace_set_gemm(g_trace_dev); rr_trace_set_attn_decode(g_trace_dev);
    rr_trace_set_attn_tc(g_trace_dev);
    rr_trace_set_elementwise(g_trace_dev);
    return check_last();
}
// Stops tracing and copies up to max_entries (id, start, dep, end) records; returns the number recorded via *n.
RR_API int rr_debug_trace_stop(unsigned long long* out, int max_entries, int* n) {
    if (!g_trace_dev || !out || !n) return RR_INVALID_ARGUMENT;
    cudaDeviceSynchronize();
    rr_trace_set_gemm(nullptr); rr_trace_set_attn_decode(nullptr);
    rr_trace_set_attn_tc(nullptr);
    rr_trace_set_elementwise(nullptr);
    unsigned long long cnt = 0;
    cudaMemcpy(&cnt, g_trace_dev, 8, cudaMemcpyDeviceToHost);
    int m = (int)(cnt < (unsigned long long)g_trace_cap ? cnt : g_trace_cap);
    if (g_trace_detail_on) m = g_trace_cap;       // fixed-slot detail marks live at the end of the buffer; empty rows are zero
    if (m > max_entries) m = max_entries;
    cudaMemcpy(out, g_trace_dev + 2, (size_t)m * 32, cudaMemcpyDeviceToHost);
    *n = m;
    cudaFree(g_trace_dev);
    g_trace_dev = nullptr;
    return check_last();
}

// Fixed-slot marks of sample CTAs inside the fused MLP / decode attention / plain decode projection kernels; off by default.
RR_API int rr_debug_trace_detail(int on) {
    g_trace_detail_on = on ? 1 : 0;
    rr_trace_set_gemm_detail(on);      // 1: fused MLP kernel; 10 + s: the plain decode projection with split-K factor s
    rr_trace_set_attn_decode_detail(on ? 1 : 0);
    return check_last();
}

RR_API int rr_set_pdl(int enabled) {
    int old = g_use_pdl;
    g_use_pdl = enabled ? 1 : 0;
    return old;
}

// ---------------------------------------------------------------- tokenizer (K2)
// Byte-level: id 1 = BOS, then 3 + byte value (0/1/2 reserved: pad/bos/eos), folded into the
// model's vocabulary by modulo when vocab < 259.
RR_API int rr_count_tokens(const uint8_t* text, size_t n_bytes, int32_t* n_tokens) {
    if (!n_tokens || (!text && n_bytes)) return RR_INVALID_ARGUMENT;
    *n_tokens = (int32_t)n_bytes + 1;
    return RR_OK;
}

RR_API int rr_tokenize(const uint8_t* text, size_t n_bytes, int32_t vocab, int32_t* ids,
                       int32_t max_ids, int32_t* n_ids) {
    if (!ids || !n_ids || vocab < 4 || (!text && n_bytes)) return RR_INVALID_ARGUMENT;
    if ((size_t)max_ids < n_bytes + 1) return RR_INVALID_ARGUMENT;
    ids[0] = 1;
    for (size_t i = 0; i < n_bytes; ++i) {
        int32_t t = 3 + (int32_t)text[i];
        ids[i + 1] = t < vocab ? t : 3 + (t - 3) % (vocab - 3);
    }
    *n_ids = (int32_t)n_bytes + 1;
    return RR_OK;
}

// ---------------------------------------------------------------- kernels
RR_API int rr_gemm_bf16(const void* A, int rowsA, int ldA, const void* B, int rowsB, int ldB, int K,
                        void* out, int ldo, int ld_rows, int splits, int mode, int bn,
                        void* stream) {
    GemmPlan p;
    int rc = gemm_plan_init(&p, A, rowsA, ldA, B, rowsB, ldB, K, out, ldo, ld_rows, splits, mode, bn);
    if (rc != RR_OK) return rc;
    rc = gemm_launch(p, (cudaStream_t)stream);
    if (rc != RR_OK) note_cuda_error(cudaPeekAtLastError());
    return rc;
}

static PartIn mk_part(const void* p, int is_bf16, int n_splits, long long split_stride, int ld) {
    PartIn r;
    r.ptr = p; r.is_bf16 = is_bf16; r.n_splits = n_splits < 1 ? 1 : n_splits;
    r.split_stride = split_stride; r.ld = ld;
    return r;
}

RR_API int rr_op_embed(const int32_t* ids, const void* table, float* x, int rows, int hidden,
                       const int32_t* row_active, void* stream) {
    if (!ids || !table || !x || hidden % 8) return RR_INVALID_ARGUMENT;
    launch_embed(ids, (const __nv_bfloat16*)table, x, rows, hidden, row_active, (cudaStream_t)stream);
    return check_last();
}

RR_API int rr_op_add_rmsnorm(float* x, const void* part, int part_is_bf16, int n_splits,
                             long long split_stride, int part_ld, const void* w, void* xn, int rows,
                             int hidden, float eps, void* stream) {
    if (!x || !w || !xn || hidden % 4) return RR_INVALID_ARGUMENT;
    launch_add_rmsnorm(x, mk_part(part, part_is_bf16, n_splits, split_stride, part_ld),
                       (const __nv_bfloat16*)w, (__nv_bfloat16*)xn, rows, hidden, eps, (cudaStream_t)stream);
    return check_last();
}

RR_API int rr_op_silu_mul(const void* gu, int is_bf16, int n_splits, long long split_stride, int ld,
                          void* act, int rows, int inter, void* stream) {
    if (!gu || !act || inter % 4) return RR_INVALID_ARGUMENT;
    launch_silu_mul(mk_part(gu, is_bf16, n_splits, split_stride, ld), (__nv_bfloat16*)act, rows, inter,
                    (cudaStream_t)stream);
    return check_last();
}

RR_API int rr_op_rope_kv(const void* qkv, int is_bf16, int n_splits, long long split_stride, int ld,
                         void* q_out, void* k_cache, void* v_cache, const int32_t* slot,
                         const int32_t* pos, int rows, int n_heads, int n_kv_heads, int ctx_max,
                         float theta, void* stream) {
    if (!qkv || !q_out || !k_cache || !v_cache || !slot || !pos) return RR_INVALID_ARGUMENT;
    RopeArgs a;
    a.qkv = mk_part(qkv, is_bf16, n_splits, split_stride, ld);
    a.q_out = (__nv_bfloat16*)q_out; a.k_cache = (__nv_bfloat16*)k_cache; a.v_cache = (__nv_bfloat16*)v_cache;
    a.slot = slot; a.pos = pos; a.rows = rows; a.n_heads = n_heads; a.n_kv_heads = n_kv_heads;
    a.ctx_max = ctx_max; a.theta = theta; a.table = nullptr; a.head_dim = 128;
    launch_rope_kv(a, (cudaStream_t)stream);
    return check_last();
}

RR_API int rr_op_argmax(const float* logits, int ld, int rows, int vocab, int32_t* out_tok,
                        float* out_val, const int32_t* row_active, int32_t* pos_inc, void* stream) {
    if (!logits || !out_tok || ld % 4) return RR_INVALID_ARGUMENT;
    launch_argmax(mk_part(logits, 0, 1, 0, ld), rows, vocab, out_tok, out_val, row_active, pos_inc,
                  (cudaStream_t)stream);
    return check_last();
}

RR_API int rr_op_decode_attn(const void* q, const void* k_cache, const void* v_cache, void* out,
                             const int32_t* slot, const int32_t* pos, int rows, int n_heads,
                             int n_kv_heads, int ctx_max, int n_slots, float scale, int kv_splits, void* stream) {
    if (!q || !k_cache || !v_cache || !out || !slot || !pos || n_slots < 1) return RR_INVALID_ARGUMENT;
    if (n_kv_heads <= 0 || n_heads % n_kv_heads) return RR_INVALID_ARGUMENT;
    const int G = n_heads / n_kv_heads;
    if (!(G == 1 || G == 2 || G == 4 || G == 8)) return RR_INVALID_ARGUMENT;
    DecodeAttnArgs a;
    a.q = (const __nv_bfloat16*)q; a.k_cache = (const __nv_bfloat16*)k_cache;
    a.v_cache = (const __nv_bfloat16*)v_cache; a.out = (__nv_bfloat16*)out; a.slot = slot; a.pos = pos;
    a.rows = rows; a.n_heads = n_heads; a.n_kv_heads = n_kv_heads; a.ctx_max = ctx_max; a.scale = scale;
    a.kv_splits = kv_splits < 1 ? 1 : kv_splits; a.ws = nullptr;
    a.fuse_rope = 0; a.qkv.ptr = nullptr; a.rope_table = nullptr; a.head_dim = 128;
    { int rcm = decode_attn_make_maps(&a, n_slots); if (rcm != RR_OK) return rcm; }
    float* ws = nullptr;
    if (a.kv_splits > 1) {
        cudaError_t e = cudaMallocAsync(&ws, decode_attn_ws_bytes(rows, n_heads, a.kv_splits), (cudaStream_t)stream);
        if (e != cudaSuccess) { note_cuda_error(e); return RR_CUDA_ERROR; }
        a.ws = ws;
    }
    launch_decode_attn(a, (cudaStream_t)stream);
    if (ws) cudaFreeAsync(ws, (cudaStream_t)stream);
    return check_last();
}

RR_API int rr_debug_mlp_schedule(int grid, int inter, int hidden, int slice_kb, int32_t* items_out, int capacity,
                                 int* max_items) {
    if (grid < 1 || inter < 64 || inter % 64 || hidden < 8 || slice_kb < 1 || !max_items) return RR_INVALID_ARGUMENT;
    std::vector<MlpItem> items;
    *max_items = mlp_schedule(grid, inter, hidden, slice_kb, &items);
    if (!items_out || (size_t)capacity < items.size()) return RR_INVALID_ARGUMENT;
    static_assert(sizeof(MlpItem) == 4 * sizeof(int32_t), "MlpItem layout");
    memcpy(items_out, items.data(), items.size() * sizeof(MlpItem));
    return RR_OK;
}

RR_API int rr_op_prefill_attn(const void* q, const void* k_cache, const void* v_cache, void* out,
                              const int32_t* seq_start, const int32_t* seq_slot, int n_seqs,
                              int max_len, int n_heads, int n_kv_heads, int ctx_max, float scale,
                              void* stream) {
    if (!q || !k_cache || !v_cache || !out || !seq_start || !seq_slot) return RR_INVALID_ARGUMENT;
    if (n_kv_heads <= 0 || n_heads % n_kv_heads) return RR_INVALID_ARGUMENT;
    PrefillAttnArgs a;
    a.q = (const __nv_bfloat16*)q; a.k_cache = (const __nv_bfloat16*)k_cache;
    a.v_cache = (const __nv_bfloat16*)v_cache; a.out = (__nv_bfloat16*)out; a.seq_start = seq_start;
    a.seq_slot = seq_slot; a.n_seqs = n_seqs; a.max_len = max_len; a.n_heads = n_heads;
    a.n_kv_heads = n_kv_heads; a.ctx_max = ctx_max; a.scale = scale; a.head_dim = 128;
    if (n_seqs > 0) {
        // the TMA maps need the extents of q and of the caches, which this entry point
        // does not take -- read them back from the caller's index arrays (standalone op, not the engine path).
        std::vector<int32_t> h(n_seqs + 1);
        cudaError_t e = cudaMemcpyAsync(h.data(), seq_slot, sizeof(int32_t) * n_seqs, cudaMemcpyDeviceToHost, (cudaStream_t)stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(&h[n_seqs], seq_start + n_seqs, sizeof(int32_t), cudaMemcpyDeviceToHost, (cudaStream_t)stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize((cudaStream_t)stream);
        if (e != cudaSuccess) { note_cuda_error(e); return RR_CUDA_ERROR; }
        int max_slot = 0;
        for (int i = 0; i < n_seqs; ++i) max_slot = h[i] > max_slot ? h[i] : max_slot;
        (void)prefill_attn_make_maps(&a, h[n_seqs], (long long)(max_slot + 1) * n_kv_heads * ctx_max);
    }
    const int rcl = launch_prefill_attn(a, (cudaStream_t)stream);
    if (rcl != RR_OK) return rcl;
    return check_last();
}
