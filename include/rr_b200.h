/* rr_b200.h — public C-ABI of librr_b200.so, the B200-native replacement for the request-router
 * hot path of aws-samples/sample-resilient-llm-inference.
 *
 * The reference has NO native/FFI boundary: its hot path is `litellm.Router` (un-vendored
 * dependency, reference pyproject.toml:8) configured by reference config/config.yaml:35-108,
 * launched by reference bin/start-gateway.sh:54 and called over HTTP from
 * reference src/demo_load_balancing.py:106-110, src/demo_fallback.py:143-147 and
 * src/demo_quota_isolation.py:52-56; tokens are produced by the remote bedrock:InvokeModel call
 * (reference iam/policy.json:8, src/demo_cris.py:233-238).  Every entry point below names the
 * reference interface it replaces.  INTEGRATION.md shows the ctypes binding a maintainer of the
 * reference would add.
 *
 * Conventions: plain C types only; integer return codes (no exceptions cross the ABI);
 * caller-owned buffers; `stream` arguments are cudaStream_t passed as void* (NULL = legacy
 * default stream).  All functions return RR_OK (0) on success.
 */
#ifndef RR_B200_H
#define RR_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------------------------------
 * Return codes.  RR_RATE_LIMITED is what the Python host maps to HTTP 429 / RateLimitError
 * (reference src/demo_quota_isolation.py:80, src/demo_fallback.py:184). */
enum {
    RR_OK = 0,
    RR_RATE_LIMITED = 1,      /* no deployment admitted the request (rpm/tpm/cooldown) -> 429 */
    RR_NO_GROUP = 2,          /* unknown model group -> 400 */
    RR_INTERNAL = 3,          /* -> 500 */
    RR_INVALID_ARGUMENT = 4,
    RR_CUDA_ERROR = 5,
    RR_TIMEOUT = 6,
    RR_BACKEND_FAILED = 7,    /* injected/real backend failure with no fallback left -> 500 */
    RR_CANCELLED = 8          /* the request was abandoned by its owner (rr_engine_cancel / rr_gateway_cancel) */
};

const char* rr_version(void);
const char* rr_strerror(int rc);
/* Last CUDA error string seen by the library on this thread (diagnostics). */
const char* rr_last_cuda_error(void);
/* Programmatic dependent launch between the library's kernels (default on; env RR_NO_PDL=1 turns it
 * off).  Returns the previous setting.  Must not change between capture and replay of an engine graph. */
int rr_set_pdl(int enabled);
/* Debug timeline: CTA 0 of every library kernel records (kernel id, start ns, ns when griddepcontrol.wait
 * returned, end ns) with %globaltimer.  start allocates a device buffer; stop copies `*n` records
 * (4 x uint64 each) to `out`. */
int rr_debug_trace_start(int max_entries);
int rr_debug_trace_stop(unsigned long long* out, int max_entries, int* n);
/* on = 1: sample CTAs of the fused decode MLP kernel (kernel ids 50 + k) and of the decode attention kernel (80 + k) also
 * record fixed-slot marks at the end of the trace buffer; on = 10 + s: also those of the plain decode projection with
 * split-K factor s (100 + k).  on = 0 turns them off. */
int rr_debug_trace_detail(int on);
/* Host-side work schedule of the fused decode MLP kernel (gate/up + down GEMMs in one launch, DESIGN.md section 3), for
 * inspection and tests; no device is touched.  items_out receives grid * (*max_items) entries of 4 x int32
 * {tile | phase << 16 (phase 0 gate/up, 1 down; -1 = end of the CTA's list), kb0, kb1, slice}, CTA-major;
 * returns RR_INVALID_ARGUMENT when `capacity` (in entries) is too small (*max_items is still set). */
int rr_debug_mlp_schedule(int grid, int inter, int hidden, int slice_kb, int32_t* items_out, int capacity,
                          int* max_items);

/* ================================================================================================
 * 1. Router: admission + rpm/tpm bucket debit + backend pick + cooldown + fallback chain (K1).
 *    Replaces litellm.Router as configured by reference config/config.yaml:35-108
 *    (model_list[].{model_name,litellm_params,rpm,tpm}; router_settings.{routing_strategy,
 *    enable_pre_call_checks,allowed_fails,cooldown_time,fallbacks}).
 *    State lives in HBM; one kernel launch processes an ordered trace of events with the same
 *    result as processing them one at a time (serialised-trace semantics, DESIGN.md §router). */

enum {                       /* router_settings.routing_strategy (reference config.yaml:101) */
    RR_STRATEGY_SIMPLE_SHUFFLE = 0,
    RR_STRATEGY_LEAST_BUSY = 1,
    /* client-side distribution strategies of reference src/demo_account_sharding.py:335-343: */
    RR_STRATEGY_ROUND_ROBIN = 2,  /* req_id % n */
    RR_STRATEGY_SPLIT = 3,        /* first share of the burst to backend 0, next to backend 1, ... (req_id < N / 2) */
    RR_STRATEGY_RANDOM = 4        /* random.choice, weights ignored */
};

/* RR_EV_BURST(target = group, tokens = N) declares the size of the next burst for RR_STRATEGY_SPLIT. */
enum { RR_EV_ADMIT = 0, RR_EV_DONE = 1, RR_EV_FAIL = 2, RR_EV_BURST = 3 };

typedef struct rr_deployment_desc {
    int32_t group;           /* index of model_name (reference config.yaml:36,44,...) */
    int32_t rpm;             /* requests / minute, <0 = unlimited (config.yaml:41) */
    int32_t tpm;             /* tokens / minute, <0 = unlimited (config.yaml:42) */
    int32_t weight;          /* simple-shuffle weight, <0 = unset */
    int32_t replica;         /* GPU / engine index that serves this deployment */
    int32_t reserved;
} rr_deployment_desc;

typedef struct rr_router_settings {
    int32_t strategy;               /* RR_STRATEGY_* */
    int32_t enable_pre_call_checks; /* config.yaml:102 */
    int32_t allowed_fails;          /* config.yaml:103 */
    int32_t cooldown_ms;            /* config.yaml:104 (seconds * 1000) */
    int32_t weight_by;              /* 0 = uniform, 1 = weight, 2 = rpm, 3 = tpm (simple-shuffle) */
    int32_t reserved[3];
} rr_router_settings;

typedef struct rr_event {
    int32_t type;            /* RR_EV_* */
    int32_t target;          /* ADMIT: group index; DONE/FAIL: deployment index */
    int32_t tokens;          /* ADMIT: prompt tokens; DONE: completion tokens */
    int32_t chain_start;     /* ADMIT: 0 = try the group itself first, k = start at k-th fallback */
    int64_t now_ms;          /* injectable clock, milliseconds */
} rr_event;

typedef struct rr_decision {
    int32_t status;          /* RR_OK / RR_RATE_LIMITED / RR_NO_GROUP */
    int32_t deployment;      /* picked deployment, -1 if none */
    int32_t served_group;    /* group that served (differs from target when fell back) */
    int32_t chain_pos;       /* 0 = primary, k = k-th fallback */
} rr_decision;

typedef struct rr_deployment_state {
    int64_t window;          /* minute index of the rpm/tpm window */
    int32_t req_count;
    int32_t tok_count;
    int64_t fail_window;
    int32_t fail_count;
    int32_t inflight;
    int64_t cooldown_until_ms;
    int64_t total_admitted;
} rr_deployment_state;

typedef struct rr_router rr_router;

/* fallback chains in CSR form: group g falls back to fb_groups[fb_offsets[g] .. fb_offsets[g+1])
 * (reference config.yaml:105-108). */
int rr_router_create(const rr_deployment_desc* deployments, int n_deployments, int n_groups,
                     const int32_t* fb_offsets, const int32_t* fb_groups,
                     const rr_router_settings* settings, uint64_t seed, int device,
                     rr_router** out);
void rr_router_destroy(rr_router* r);
/* Host buffers: copies events H2D, runs the admission kernel, copies decisions D2H. Thread-safe. */
int rr_router_process(rr_router* r, const rr_event* events, int n_events, rr_decision* decisions);
/* Device buffers already resident in HBM; asynchronous on `stream`. */
int rr_router_process_device(rr_router* r, const rr_event* d_events, int n_events,
                             rr_decision* d_decisions, void* stream);
int rr_router_snapshot(rr_router* r, rr_deployment_state* out /* [n_deployments] */);
/* Re-seed the MT19937 stream exactly like CPython random.seed(int). */
int rr_router_seed(rr_router* r, uint64_t seed);
/* Host-only: the MT19937 state (624 words + index) CPython's random.seed(seed) produces. */
int rr_mt_seed_state(uint64_t seed, uint32_t* out625);

/* ================================================================================================
 * 2. Prompt token count (K2).  Replaces litellm.token_counter as used for tpm accounting
 *    (no call site in the reference tree; tpm values at reference config.yaml:42).
 *    Counts tokens of the library's byte-level tokenizer: n_tokens = n_utf8_bytes + 1 (BOS).
 *    rr_count_tokens / rr_tokenize are the host forms (one message); the request path uses the batch kernel below. */
int rr_count_tokens(const uint8_t* text, size_t n_bytes, int32_t* n_tokens);
int rr_tokenize(const uint8_t* text, size_t n_bytes, int32_t vocab, int32_t* ids, int32_t max_ids,
                int32_t* n_ids);
/* The same tokenizer as a CUDA kernel over a batch of messages (csrc/rr_tokenizer.cu): n_texts messages back to back in
 * `text`, text_off[n_texts + 1] byte offsets.  counts[i] = tokens of message i (what an ADMIT event carries into the tpm
 * check); ids (optional) = the packed token ids, message i at ids_off[i] = text_off[i] - text_off[0] + i.
 * rr_tokenize_batch: host buffers (H2D copy, kernel, D2H copies inside; thread-safe).
 * rr_tokenize_batch_device: device buffers, asynchronous on `stream`; max_text_bytes bounds the longest message. */
int rr_tokenize_batch(const uint8_t* text, const int64_t* text_off, int n_texts, int32_t vocab, int32_t* counts_out,
                      int32_t* ids_out, int64_t ids_capacity, int64_t* ids_off_out);
int rr_tokenize_batch_device(const uint8_t* d_text, const int64_t* d_text_off, int n_texts, int64_t max_text_bytes,
                             int32_t vocab, int32_t* d_counts, int32_t* d_ids, int64_t* d_ids_off, void* stream);

/* ================================================================================================
 * 3. Kernel-level entry points (used by the parity tests and the engine).
 *    Replaces the remote bedrock:InvokeModel prefill/decode (reference iam/policy.json:8,
 *    src/demo_cris.py:233-238).  All pointers are device pointers. */

enum { RR_OUT_ROWMAJOR_BF16 = 0, RR_OUT_TRANSPOSED_F32 = 1,
       /* fused SiLU(gate)*up epilogues; the weight operand holds gate/up rows interleaved in 64-row blocks
        * [g0..g63, u0..u63, g64..g127, u64..u127, ...] and the output is bf16 act[.., inter]: */
       RR_OUT_TRANSPOSED_SILU = 2,   /* decode: A = interleaved weight [2*inter, K], out[b*ldo + n], splits = 1 */
       RR_OUT_ROWMAJOR_SILU = 3,     /* prefill: B = interleaved weight, bn = 256, out[a*ldo + n] */
       RR_OUT_ROWMAJOR_ROPE = 4,     /* engine-internal (prefill QKV epilogue with RoPE + KV scatter) */
       RR_OUT_ROWMAJOR_RESID = 5 };  /* out = fp32 residual [rowsA, ldo]: out[a*ldo + b] += acc (bn >= 128) */

/* D[a,b] = sum_k A[a,k] B[b,k] on tcgen05 tensor cores (bf16 in, fp32 accumulate).
 * mode RR_OUT_ROWMAJOR_BF16:  out bf16 [rowsA, ldo], out[a*ldo + b]         (splits must be 1)
 * mode RR_OUT_TRANSPOSED_F32: out fp32 [splits, ld_rows, ldo], out[(z*ld_rows + b)*ldo + a]
 * bn = tile width along B rows: 16/32/64/128/256.  splits >= 1. */
int rr_gemm_bf16(const void* A, int rowsA, int ldA, const void* B, int rowsB, int ldB, int K,
                 void* out, int ldo, int ld_rows, int splits, int mode, int bn, void* stream);

int rr_op_embed(const int32_t* ids, const void* table, float* x, int rows, int hidden,
                const int32_t* row_active, void* stream);
int rr_op_add_rmsnorm(float* x, const void* part, int part_is_bf16, int n_splits,
                      long long split_stride, int part_ld, const void* w, void* xn, int rows,
                      int hidden, float eps, void* stream);
int rr_op_silu_mul(const void* gu, int is_bf16, int n_splits, long long split_stride, int ld,
                   void* act, int rows, int inter, void* stream);
int rr_op_rope_kv(const void* qkv, int is_bf16, int n_splits, long long split_stride, int ld,
                  void* q_out, void* k_cache, void* v_cache, const int32_t* slot,
                  const int32_t* pos, int rows, int n_heads, int n_kv_heads, int ctx_max,
                  float theta, void* stream);
int rr_op_argmax(const float* logits, int ld, int rows, int vocab, int32_t* out_tok,
                 float* out_val, const int32_t* row_active, int32_t* pos_inc, void* stream);
int rr_op_decode_attn(const void* q, const void* k_cache, const void* v_cache, void* out,
                      const int32_t* slot, const int32_t* pos, int rows, int n_heads,
                      int n_kv_heads, int ctx_max /* % 64 == 0 */, int n_slots, float scale,
                      int kv_splits, void* stream);
int rr_op_prefill_attn(const void* q, const void* k_cache, const void* v_cache, void* out,
                       const int32_t* seq_start, const int32_t* seq_slot, int n_seqs, int max_len,
                       int n_heads, int n_kv_heads, int ctx_max, float scale, void* stream);

/* ================================================================================================
 * 4. Engine: one model replica on one GPU (prefill + continuous-batching greedy decode).
 *    Replaces one `litellm_params.model: bedrock/...` deployment (reference config.yaml:39,47,54,
 *    62,69,77,84,91). */

typedef struct rr_model_desc {
    int32_t vocab, hidden, inter, n_layers, n_heads, n_kv_heads, head_dim;
    float rope_theta, rms_eps;
} rr_model_desc;

/* Device pointers to bf16 weights, row-major [out_features, in_features] like torch nn.Linear.
 * wqkv = concat(q_proj, k_proj, v_proj) rows; wgu = concat(gate_proj, up_proj) rows. */
typedef struct rr_model_weights {
    const void* embed;            /* [vocab, hidden] */
    const void* lm_head;          /* [vocab, hidden] */
    const void* final_norm;       /* [hidden] */
    const void* const* wqkv;      /* n_layers x [(n_heads + 2 n_kv_heads) * head_dim, hidden] */
    const void* const* wo;        /* n_layers x [hidden, n_heads * head_dim] */
    const void* const* wgu;       /* n_layers x [2 * inter, hidden] */
    const void* const* wdown;     /* n_layers x [hidden, inter] */
    const void* const* norm_attn; /* n_layers x [hidden] */
    const void* const* norm_mlp;  /* n_layers x [hidden] */
    int32_t flags;                /* RR_WEIGHTS_* */
    int32_t reserved;
} rr_model_weights;
/* wgu rows are interleaved in 64-row gate/up blocks [g0..g63, u0..u63, g64.., u64.., ...] instead of
 * [gate; up]: enables the fused SiLU*mul GEMM epilogues (no separate activation kernel). */
#define RR_WEIGHTS_WGU_INTERLEAVED64 1

typedef struct rr_engine rr_engine;

typedef struct rr_engine_opts {
    int32_t device;
    int32_t max_batch;            /* decode rows / KV slots (<= 256) */
    int32_t ctx_max;              /* tokens per KV slot */
    int32_t max_prefill_tokens;   /* tokens per prefill chunk */
    int32_t use_cuda_graph;       /* capture the decode step */
    int32_t fail_seed;            /* fault injection: seed of the Bernoulli failure mask */
    float fail_prob;              /* fault injection: P(request fails) (BASELINE config #4) */
    int32_t reserved[4];          /* A/B switches: [0] unused, ignored; [1] = 1 no RoPE fusion in the prefill
                                     QKV epilogue; [2] = 1 no fused decode MLP kernel; [3] = 1 prefill RMSNorm as separate kernels instead of deferred into the GEMM epilogues */
} rr_engine_opts;

int rr_engine_create(const rr_model_desc* desc, const rr_model_weights* w,
                     const rr_engine_opts* opts, rr_engine** out);
void rr_engine_destroy(rr_engine* e);

/* Low-level synchronous steps (parity tests).  Host buffers.
 * prefill: n_seqs prompts concatenated in `ids`; seq_start[n_seqs+1]; slots[n_seqs] = KV slots.
 *          Writes first generated token per prompt to first_tok[n_seqs].
 *          If logits_out != NULL: fp32 [n_seqs, vocab] last-position logits. */
int rr_engine_prefill(rr_engine* e, const int32_t* ids, const int32_t* seq_start,
                      const int32_t* slots, int n_seqs, int32_t* first_tok, float* logits_out);
/* One decode step for the given slots, feeding tok[i] at position pos[i]; returns next tokens and
 * optionally fp32 logits [n, vocab]. */
int rr_engine_decode_step(rr_engine* e, const int32_t* slots, const int32_t* tok,
                          const int32_t* pos, int n, int32_t* next_tok, float* logits_out);

/* Asynchronous serving interface (the call shape of chat.completions.create: reference
 * src/demo_load_balancing.py:106-110).  submit is thread-safe and non-blocking; wait blocks
 * (release the GIL around it). */
typedef struct rr_completion {
    uint64_t ticket;
    int32_t status;               /* RR_OK / RR_BACKEND_FAILED / RR_TIMEOUT */
    int32_t n_prompt;
    int32_t n_generated;
    int32_t reserved;
    double t_submit_s, t_first_token_s, t_done_s;   /* engine monotonic clock */
} rr_completion;

int rr_engine_submit(rr_engine* e, const int32_t* prompt_ids, int n_prompt, int max_new_tokens,
                     uint64_t* ticket);
int rr_engine_wait(rr_engine* e, uint64_t ticket, double timeout_s, rr_completion* out,
                   int32_t* tokens_out, int max_tokens_out);
/* Abandon a request: queued -> dropped; running -> its decode row is freed at the next step; finished -> freed.
 * Consumes the ticket (do not wait on it afterwards).  Replaces the client-side `timeout=` of the reference's
 * chat.completions.create calls (reference src/demo_fallback.py:146) as seen from the backend. */
int rr_engine_cancel(rr_engine* e, uint64_t ticket);
/* Streaming (SSE): block until the request holds more than `have` tokens, is done, or `timeout_s` elapses;
 * copies the tokens generated so far.  Does not consume the request — finish with rr_engine_wait. */
int rr_engine_peek(rr_engine* e, uint64_t ticket, int have, double timeout_s, int32_t* tokens_out,
                   int max_tokens_out, int32_t* n_generated, int32_t* done, double* t_first_token_s);
/* Closed-batch convenience used by bench.py: submit all, wait all. prompts are host buffers
 * (pinned or pageable); the H2D copies happen inside. */
int rr_engine_run_batch(rr_engine* e, const int32_t* prompt_ids, const int32_t* prompt_start,
                        int n_requests, int max_new_tokens, rr_completion* out,
                        int32_t* tokens_out /* [n_requests, max_new_tokens] */);
double rr_engine_now(rr_engine* e);

typedef struct rr_engine_stats {
    uint64_t kernel_launches;     /* library kernels launched (graph replays count their nodes) */
    uint64_t decode_steps, prefill_chunks, prefill_tokens, generated_tokens;
    double decode_ms_total, prefill_ms_total;   /* CUDA-event time on the engine stream */
    int32_t active_rows, queued;
    uint64_t h2d_bytes, d2h_bytes;
} rr_engine_stats;
int rr_engine_get_stats(rr_engine* e, rr_engine_stats* out);
int rr_engine_reset_stats(rr_engine* e);

/* ================================================================================================
 * 5. Gateway: the whole per-request path behind one submit / wait pair, in native code.
 *    Replaces the reference's gateway process as its clients see it: N concurrent blocking
 *    chat.completions.create calls (reference src/demo_load_balancing.py:195-203,
 *    src/demo_quota_isolation.py:135-139) into litellm's single worker (reference bin/start-gateway.sh:54).
 *    rr_gateway_submit is thread-safe and non-blocking: the request enters an admission queue; a dispatcher
 *    thread coalesces everything pending (ADMIT / DONE / FAIL / fallback re-ADMIT) into ONE ordered trace per
 *    K1 launch (rr_router_process) and hands admitted prompts straight to the engine of the picked
 *    deployment.  A backend failure walks the fallback chain inside the library. */

typedef struct rr_gateway rr_gateway;

typedef struct rr_gateway_opts {
    int32_t manual_clock;      /* 0: events are stamped with the wall clock (ms); 1: with rr_gateway_set_now() */
    int32_t record_trace;      /* keep the last N (event, decision) pairs for replay through an oracle; 0 = off */
    int32_t max_batch_events;  /* events per K1 launch, 0 = 4096 */
    int32_t reserved[5];
} rr_gateway_opts;

typedef struct rr_gateway_result {
    uint64_t ticket;
    int32_t status;            /* RR_OK / RR_RATE_LIMITED (429) / RR_NO_GROUP / RR_BACKEND_FAILED / RR_TIMEOUT / RR_CANCELLED / ...;
                                  -1 while in flight (rr_gateway_peek) */
    int32_t deployment, served_group, chain_pos, replica;   /* the admission decision (valid once admitted) */
    int32_t n_prompt, n_generated;
    int32_t attempts;          /* admissions this request went through (1 + backends that failed under it) */
    double t_submit_s, t_admit_s, t_first_token_s, t_done_s;   /* gateway monotonic clock, seconds */
} rr_gateway_result;

typedef struct rr_gateway_stats {
    uint64_t submitted, admitted, completed, rate_limited, failed, failed_over;
    uint64_t launches;         /* K1 launches */
    uint64_t events;           /* events those launches processed */
    uint64_t max_batch;        /* largest trace of one launch */
    uint64_t in_flight;
    double admit_wait_s;       /* sum over admissions of (decision time - submit time) */
} rr_gateway_stats;

/* engines[i] serves the deployments whose rr_deployment_desc.replica == replica_ids[i].  The router and the engines
 * must outlive the gateway; the engines' completion hooks are taken by the gateway until it is destroyed. */
int rr_gateway_create(rr_router* router, rr_engine* const* engines, const int32_t* replica_ids, int n_engines,
                      const rr_gateway_opts* opts, rr_gateway** out);
void rr_gateway_destroy(rr_gateway* g);
int rr_gateway_set_now(rr_gateway* g, int64_t now_ms);
/* group = index of the model group (model_name) the client asked for.  Returns RR_NO_GROUP / RR_INVALID_ARGUMENT
 * (prompt + max_new_tokens beyond a replica's context, bad token id: HTTP 400) before anything is debited. */
int rr_gateway_submit(rr_gateway* g, int group, const int32_t* prompt_ids, int n_prompt, int max_new_tokens,
                      uint64_t* ticket);
/* A closed burst as one contiguous block of the admission trace (declare_burst != 0 prepends RR_EV_BURST). */
int rr_gateway_submit_batch(rr_gateway* g, int group, const int32_t* prompt_ids, const int32_t* prompt_start, int n,
                            int max_new_tokens, int declare_burst, uint64_t* tickets);
/* Blocks (release the GIL) until the request is finished; returns its status and consumes the ticket.
 * RR_TIMEOUT: still in flight -- wait again or rr_gateway_cancel. */
int rr_gateway_wait(rr_gateway* g, uint64_t ticket, double timeout_s, rr_gateway_result* out, int32_t* tokens_out,
                    int max_tokens_out);
/* Streaming: returns once more than `have` tokens exist, the request is finished, or timeout_s elapsed. */
int rr_gateway_peek(rr_gateway* g, uint64_t ticket, int have, double timeout_s, int32_t* tokens_out, int max_tokens_out,
                    int32_t* n_generated, int32_t* done, rr_gateway_result* out);
/* Abandon a request (consumes the ticket).  count_as_failure != 0: a client-side timeout -- the deployment gets a FAIL
 * event (allowed_fails / cooldown, reference config/config.yaml:103-104); 0: a disconnect -- a DONE event. */
int rr_gateway_cancel(rr_gateway* g, uint64_t ticket, int count_as_failure);
/* Block until every event queued so far (the DONE / FAIL reports of finished requests included) has been through K1:
 * call before rr_router_snapshot when the counters must reflect all completed requests. */
int rr_gateway_quiesce(rr_gateway* g, double timeout_s);
int rr_gateway_get_stats(rr_gateway* g, rr_gateway_stats* out);
/* The recorded trace (opts.record_trace): *n pairs, oldest first. */
int rr_gateway_trace(rr_gateway* g, rr_event* events, rr_decision* decisions, int capacity, int* n);

#ifdef __cplusplus
}
#endif
#endif /* RR_B200_H */
