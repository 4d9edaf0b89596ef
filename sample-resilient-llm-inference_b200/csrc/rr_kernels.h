// rr_kernels.h — internal (C++) declarations shared by the .cu files of librr_b200.so.
// The public C-ABI is include/rr_b200.h; nothing here crosses the library boundary.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <vector>

#include "../../include/rr_b200.h"

namespace rr {

#define RR_ERR_ARG RR_INVALID_ARGUMENT
#define RR_ERR_CUDA RR_CUDA_ERROR

enum GemmOutMode { OUT_ROWMAJOR_BF16 = 0, OUT_TRANSPOSED_F32 = 1, OUT_TRANSPOSED_SILU = 2, OUT_ROWMAJOR_SILU = 3,
                   OUT_ROWMAJOR_ROPE = 4, OUT_ROWMAJOR_RESID = 5 };
// OUT_ROWMAJOR_RESID (prefill O / down projections): out is the fp32 residual stream, out[a*ldo + b] += acc —
// the following norm kernel then only reads x and writes xn (half its bytes).

// OUT_ROWMAJOR_ROPE (prefill QKV projection, head_dim 128): the epilogue rotates q and k (RoPE table), writes q to q_out
// and appends k / v to the KV cache — no intermediate qkv matrix, no separate rope_kv launch.
struct RopeEpi {
    __nv_bfloat16* q_out;     // [T, n_heads*128]
    __nv_bfloat16* k_cache;   // [slot][kv_head][ctx_max][128]
    __nv_bfloat16* v_cache;
    const int32_t* slot;      // per token row
    const int32_t* pos;
    const float2* table;      // [ctx_max][64] (cos, sin)
    int n_heads, n_kv_heads, ctx_max;
    // ---- deferred RMSNorm (prefill): the GEMM that writes the residual also emits the next GEMM's operand
    // xhat = bf16(x * gamma) (NOT normalised) and per-row partial sums of squares; the next GEMM scales its
    // accumulators by rsqrt(mean(x^2) + eps) of the row in its epilogue (the projection is linear).  No norm kernel,
    // no second pass over the fp32 residual.
    // consumer side (OUT_ROWMAJOR_ROPE / _SILU / _BF16):
    const float* rowss;       // [rowsA][n_part] partial sum(x^2) of the operand rows; n_part = 0: operand is normalised
    int n_part;
    float inv_hidden, eps;
    // producer side (OUT_ROWMAJOR_RESID): xhat = nullptr -> plain residual add
    const __nv_bfloat16* gamma;   // [rowsB] norm weight of the NEXT norm
    __nv_bfloat16* xhat;          // [rowsA][ldo]
    float* rowss_out;             // [rowsA][n_part_out], column = this item's b_tile
    int n_part_out;
};

struct GemmPlan {
    CUtensorMap tmA, tmB;
    void* out;
    int rowsA, rowsB, K, splits, ldo, ld_rows, mode, bn, max_ctas;
    RopeEpi rope;             // OUT_ROWMAJOR_ROPE only
    CUtensorMap tmB2;         // 2-CTA kernel: B with a 128-row box (each CTA of the pair stages half of the 256 rows)
    int two_cta;
    CUtensorMap tmOut;        // OUT_TRANSPOSED_F32: planes [splits][rowsB][rowsA] (3-D, box {128, bn, 1}) for the TMA-store epilogue
    int tma_epi;              // 1: the epilogue stages the tile in shared memory and issues ONE TMA store per item
};

int num_sms();

// ---- engine / router internals used by the native gateway (rr_gateway.cu)
typedef void (*EngineDoneHook)(void* ctx, uint64_t tag, uint64_t ticket, int status, int n_generated);
int engine_submit_tagged(rr_engine* e, const int32_t* prompt_ids, int n_prompt, int max_new_tokens, uint64_t tag,
                         uint64_t* ticket);
void engine_set_done_hook(rr_engine* e, EngineDoneHook fn, void* ctx);
int engine_limits(const rr_engine* e, int* ctx_max, int* max_prefill, int* vocab);
int router_shape(const rr_router* r, int* n_deployments, int* n_groups);
int router_dep_replica(const rr_router* r, int deployment);
int make_tmap_bf16_2d(CUtensorMap* map, const void* base, int rows, int K, int ld, int box_rows);
int gemm_plan_init(GemmPlan* p, const void* A, int rowsA, int ldA, const void* B, int rowsB, int ldB,
                   int K, void* out, int ldo, int ld_rows, int splits, int mode, int bn);
int gemm_launch(const GemmPlan& p, cudaStream_t st);

// ---- fused decode MLP (rr_gemm.cu): gate/up GEMM (+SiLU*mul) and down GEMM in one persistent launch.
// Per-CTA work lists (built once on the host) replace the kernel boundary: a down item covers one K-slice of
// `slice_kb` k-blocks = the act columns written by `slice_kb` gate/up tiles, and waits for `ready[slice]` to reach
// that count instead of for the whole gate/up grid.
struct MlpItem {             // 16 bytes, read as int4
    int tile_phase;           // a_tile | phase << 16 (phase 0 = gate/up, 1 = down); -1 terminates the list
    int kb0, kb1;             // k-block range
    int z;                    // down: output plane = K-slice index (also the index into `ready`)
};
struct MlpArgs {
    CUtensorMap tmA0, tmB0;   // gate/up: weights [2*inter, hidden] (64-row interleaved), activations xn [rows, hidden]
    CUtensorMap tmA1, tmB1;   // down: weights [hidden, inter], activations act [rows, inter]
    __nv_bfloat16* act;       // [rows, inter]
    float* out1;              // planes [n_slices][ld_rows][hidden]
    int inter, hidden, rows, ld_rows;
    const MlpItem* items;     // [grid][max_items]
    int max_items;
    unsigned* ready;          // [n_slices + 1], zero at launch; the last word is the dynamic down-item counter
    int slice_kb;
    int dyn, n_down, tiles1, kb1n, n_slices;   // dyn: down items drawn from ready[n_slices] in slice-major order (not in `items`)
    CUtensorMap tmAct, tmPlanes;   // TMA-store epilogues: act [rows][inter] bf16 (box {64, bn}), planes (3-D, box {128, bn, 1})
    int tma_epi;
};
struct MlpPlan {
    MlpArgs args;
    int grid, bn, n_slices;
};
// Host schedule: `items` gets grid * max_items entries (CTA-major); returns max_items.
int mlp_schedule(int grid, int inter, int hidden, int slice_kb, std::vector<MlpItem>* items, int dynamic = 0);
int mlp_plan_init(MlpPlan* p, const void* Wgu, const void* Wd, int inter, int hidden, const void* xn, int rows,
                  void* act, void* planes, int ld_rows, int bn, const MlpItem* items_dev, int max_items, int grid,
                  unsigned* ready, int slice_kb, int dynamic = 0);
int mlp_launch(const MlpPlan& p, cudaStream_t st);

// ---- elementwise / normalisation (rr_elementwise.cu) -------------------------------------------
// `part` inputs are the GEMM outputs: either fp32 split-K partials P[z][row][col] (n_splits >= 1,
// part_is_bf16 = 0, split stride = split_stride elements) or a single bf16 matrix.
struct PartIn {
    const void* ptr;
    int is_bf16;
    int n_splits;
    long long split_stride;   // elements between split planes
    int ld;                   // row pitch in elements
};

void launch_embed(const int32_t* ids, const __nv_bfloat16* table, float* x, int rows, int hidden,
                  const int32_t* row_active, cudaStream_t st);
// x[row] (+)= sum_z part[z][row]; xn[row] = rmsnorm(x[row]) * w   (part.ptr may be null: norm only)
// `zero` (optional): zero_n dependency counters reset by the kernel (the fused MLP kernel that follows it).
// `rowss_out` (optional, deferred norm): write xn = bf16(x * w) UN-normalised and rowss_out[row][0] = sum(x^2),
// rowss_out[row][1 .. n_part_out) = 0 -- the layout the OUT_ROWMAJOR_RESID epilogue produces (RopeEpi).
void launch_add_rmsnorm(float* x, PartIn part, const __nv_bfloat16* w, __nv_bfloat16* xn, int rows,
                        int hidden, float eps, cudaStream_t st, unsigned* zero = nullptr, int zero_n = 0,
                        float* rowss_out = nullptr, int n_part_out = 0);
// act[row, j] = silu(gate[row, j]) * up[row, j]; gate = cols [0, inter), up = cols [inter, 2*inter)
void launch_silu_mul(PartIn gu, __nv_bfloat16* act, int rows, int inter, cudaStream_t st);
// qkv (partials) -> RoPE(q), RoPE(k); q -> q_out [rows, n_heads*128] bf16; k, v -> KV cache.
struct RopeArgs {
    PartIn qkv;
    __nv_bfloat16* q_out;
    __nv_bfloat16* k_cache;   // [slot][kv_head][ctx_max][128]
    __nv_bfloat16* v_cache;
    const int32_t* slot;      // per row: KV slot (or -1 = skip)
    const int32_t* pos;       // per row: position
    int rows, n_heads, n_kv_heads, ctx_max;
    float theta;
    const float2* table;      // [ctx_max][64] (cos, sin) or null: compute inline
    int head_dim;             // true head dim (<= 128, % 8 == 0): column stride inside qkv; q_out / caches are padded to 128
};
void launch_rope_kv(const RopeArgs& a, cudaStream_t st);
void launch_rope_table(float2* table, int ctx_max, float theta, int head_dim, cudaStream_t st);
// argmax over fp32 logits [rows, vocab] (partials with n_splits = 1); writes next token, and if
// advance != 0: pos[row]++ (decode bookkeeping folded into the same launch).
void launch_argmax(PartIn logits, int rows, int vocab, int32_t* out_tok, float* out_val,
                   const int32_t* row_active, int32_t* pos_inc, cudaStream_t st);

// ---- attention (rr_attn_decode.cu, rr_attn_tc.cu) ---------------------------------------------------
struct DecodeAttnArgs {
    const __nv_bfloat16* q;   // [rows, n_heads*128]
    const __nv_bfloat16* k_cache;
    const __nv_bfloat16* v_cache;
    __nv_bfloat16* out;       // [rows, n_heads*128]
    const int32_t* slot;      // per row
    const int32_t* pos;       // per row: position of the current token (ctx = pos + 1)
    int rows, n_heads, n_kv_heads, ctx_max;
    float scale;
    float* ws;                // split-KV workspace (may be null when kv_splits == 1)
    int kv_splits;
    CUtensorMap tmK, tmV;     // [n_slots*n_kv_heads*ctx_max, 128] views of the caches, box {64, 64}, SW128
    CUtensorMap tmK16, tmV16; // same views, box {64, 16}: the last tile of a row is requested in 16-row pieces
    int trim_tail;
    // fused RoPE + KV append (decode): q/k/v of the current token come straight from the QKV GEMM's
    // split-K planes; q is rotated into the MMA fragments, k/v are rotated, appended to the cache and
    // patched into the staged tile.  fuse_rope == 0: `q` holds rotated bf16 queries (rope_kv_kernel ran).
    int fuse_rope;
    PartIn qkv;
    const float2* rope_table;
    int head_dim;             // true head dim: qkv column stride and `out` head stride; q / caches padded to 128
};
int decode_attn_make_maps(DecodeAttnArgs* a, int n_slots);   // fills tmK / tmV (ctx_max % 64 == 0)
void launch_decode_attn(const DecodeAttnArgs& a, cudaStream_t st);
size_t decode_attn_ws_bytes(int rows, int n_heads, int kv_splits);

struct PrefillAttnArgs {
    const __nv_bfloat16* q;   // [T, n_heads*128] (RoPE applied)
    const __nv_bfloat16* k_cache;
    const __nv_bfloat16* v_cache;
    __nv_bfloat16* out;       // [T, n_heads*128]
    const int32_t* seq_start; // [n_seqs+1] token offsets into T
    const int32_t* seq_slot;  // [n_seqs]
    int n_seqs, max_len, n_heads, n_kv_heads, ctx_max;
    float scale;
    int head_dim;             // true head dim: `out` head stride; q / caches padded to 128
    int has_maps = 0;         // tmQ/tmK/tmV valid (prefill_attn_make_maps): required
    CUtensorMap tmQ, tmK, tmV;
};
int launch_prefill_attn(const PrefillAttnArgs& a, cudaStream_t st);   // RR_ERR_ARG when the maps are missing / shape unsupported
// tcgen05 kernel (rr_attn_tc.cu): head pairs for even GQA group sizes, one head per item otherwise (MHA).
int prefill_attn_make_maps(PrefillAttnArgs* a, long long q_rows, long long kv_rows);
bool prefill_attn_tc_eligible(const PrefillAttnArgs& a);
int launch_prefill_attn_tc(const PrefillAttnArgs& a, cudaStream_t st);

}  // namespace rr
