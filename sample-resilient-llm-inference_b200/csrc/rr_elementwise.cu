// rr_elementwise.cu — the HBM-bound glue between the projections: embedding gather (K3),
// split-K reduce + residual add + RMSNorm (K4), RoPE + KV-cache append (K6), SiLU*mul,
// greedy argmax (K11 tail).  All are row-parallel, 16-byte vectorised, fp32 math.
// Each consumer reads the producing GEMM's output either as fp32 split-K partials
// P[z][row][col] (decode orientation) or as one bf16 matrix (prefill orientation).
// Every kernel is PDL-aware (rr_launch.cuh): constants may be touched before griddep_wait().
//
// Replaces (together with rr_gemm.cu / rr_attn_tc.cu / rr_attn_decode.cu) the remote bedrock:InvokeModel call
// (reference iam/policy.json:8; src/demo_cris.py:233-238).
#include <stdlib.h>
#include "rr_ptx.cuh"
#include "rr_launch.cuh"
#include "rr_kernels.h"

namespace rr {

// ---- reading a GEMM output ---------------------------------------------------------------------
// 4 consecutive columns of one row, summed over split planes.
__device__ __forceinline__ float4 part_load4(const PartIn& p, int row, int col) {
    if (p.is_bf16) {
        const uint2 v = *reinterpret_cast<const uint2*>(
            reinterpret_cast<const __nv_bfloat16*>(p.ptr) + (size_t)row * p.ld + col);
        return make_float4(bf16_lo(v.x), bf16_hi(v.x), bf16_lo(v.y), bf16_hi(v.y));
    }
    const float* base = reinterpret_cast<const float*>(p.ptr) + (size_t)row * p.ld + col;
    float4 acc = *reinterpret_cast<const float4*>(base);
#pragma unroll 8
    for (int z = 1; z < p.n_splits; ++z) {
        const float4 t = *reinterpret_cast<const float4*>(base + (size_t)z * p.split_stride);
        acc.x += t.x; acc.y += t.y; acc.z += t.z; acc.w += t.w;
    }
    return acc;
}

__device__ __forceinline__ float block_sum(float v, float* red) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    if (lane == 0) red[warp] = v;
    __syncthreads();
    float t = (lane < nw) ? red[lane] : 0.f;
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    __syncthreads();
    return t;
}

// ---- K3 embedding gather -----------------------------------------------------------------------
__global__ void embed_kernel(const int32_t* __restrict__ ids, const __nv_bfloat16* __restrict__ table,
                             float* __restrict__ x, int hidden, const int32_t* __restrict__ row_active) {
    griddep_launch();
    const int tr_slot = trace_begin(TR_EMBED);
    griddep_wait();
    trace_dep(tr_slot);
    const int row = blockIdx.x;
    if (row_active && row_active[row] < 0) return;
    const int id = ids[row];
    const __nv_bfloat16* src = table + (size_t)id * hidden;
    float* dst = x + (size_t)row * hidden;
    for (int c = threadIdx.x * 8; c < hidden; c += blockDim.x * 8) {
        const uint4 v = ldg_nc_v4(src + c);
        float4 a = make_float4(bf16_lo(v.x), bf16_hi(v.x), bf16_lo(v.y), bf16_hi(v.y));
        float4 b = make_float4(bf16_lo(v.z), bf16_hi(v.z), bf16_lo(v.w), bf16_hi(v.w));
        *reinterpret_cast<float4*>(dst + c) = a;
        *reinterpret_cast<float4*>(dst + c + 4) = b;
    }
    trace_end(tr_slot);
}

void launch_embed(const int32_t* ids, const __nv_bfloat16* table, float* x, int rows, int hidden,
                  const int32_t* row_active, cudaStream_t st) {
    if (rows <= 0) return;
    launch_pdl(embed_kernel, dim3(rows), dim3(256), 0, st, ids, table, x, hidden, row_active);
}

// ---- K4 residual add + RMSNorm (+ split-K reduce) ------------------------------------------------
// One CTA per row; the row (hidden <= 8192) stays in registers between the sum-of-squares pass and
// the normalise pass: x and the split planes are read exactly once.
// Decode (few rows, latency-bound): 1024 threads, one float4 each, so every load of a thread is independent.
// Prefill (thousands of rows, bandwidth-bound): 256 threads, 4 float4 each.

template <int THREADS, int MAXV>
__global__ void __launch_bounds__(THREADS)
add_rmsnorm_kernel(float* __restrict__ x, PartIn part, const __nv_bfloat16* __restrict__ w,
                   __nv_bfloat16* __restrict__ xn, int hidden, float eps, unsigned* __restrict__ zero, int zero_n,
                   float* __restrict__ rowss_out, int n_part_out) {
    __shared__ float red[32];
    griddep_launch();
    const int tr_slot = trace_begin(TR_NORM);
    const int row = blockIdx.x;
    float* xr = x + (size_t)row * hidden;
    // norm weights are constants: fetch them before waiting for the producer
    uint2 wv[MAXV];
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
        const int c = (threadIdx.x + i * THREADS) * 4;
        if (c < hidden) wv[i] = *reinterpret_cast<const uint2*>(w + c);
    }
    griddep_wait();
    trace_dep(tr_slot);
    // optional: reset the dependency counters of the fused MLP kernel that follows (its previous user has completed)
    // (grid-stride: the layer-kernel path resets every counter of the step here)
    for (int i = blockIdx.x * THREADS + threadIdx.x; i < zero_n; i += gridDim.x * THREADS) zero[i] = 0u;
    float4 v[MAXV];
    float ss = 0.f;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
        const int c = (threadIdx.x + i * THREADS) * 4;
        if (c < hidden) {
            v[i] = *reinterpret_cast<float4*>(xr + c);
            if (part.ptr) {
                const float4 p = part_load4(part, row, c);
                v[i].x += p.x; v[i].y += p.y; v[i].z += p.z; v[i].w += p.w;
            }
            ss += v[i].x * v[i].x + v[i].y * v[i].y + v[i].z * v[i].z + v[i].w * v[i].w;
        }
    }
    // the residual is written back only after every load of this thread has been issued: a store inside the load
    // loop would fence the following loads (possible aliasing) and turn them into a latency chain
    if (part.ptr) {
#pragma unroll
        for (int i = 0; i < MAXV; ++i) {
            const int c = (threadIdx.x + i * THREADS) * 4;
            if (c < hidden) *reinterpret_cast<float4*>(xr + c) = v[i];
        }
    }
    ss = block_sum(ss, red);
    // deferred norm: hand sum(x^2) to the consuming GEMM's epilogue and leave the operand un-normalised
    if (rowss_out != nullptr && (int)threadIdx.x < n_part_out)
        rowss_out[(size_t)row * n_part_out + threadIdx.x] = threadIdx.x == 0 ? ss : 0.f;
    const float inv = rowss_out != nullptr ? 1.f : rsqrtf(ss / (float)hidden + eps);
    __nv_bfloat16* out = xn + (size_t)row * hidden;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
        const int c = (threadIdx.x + i * THREADS) * 4;
        if (c < hidden) {
            uint2 o;
            o.x = pack_bf16(v[i].x * inv * bf16_lo(wv[i].x), v[i].y * inv * bf16_hi(wv[i].x));
            o.y = pack_bf16(v[i].z * inv * bf16_lo(wv[i].y), v[i].w * inv * bf16_hi(wv[i].y));
            *reinterpret_cast<uint2*>(out + c) = o;
        }
    }
    trace_end(tr_slot);
}

// Decode variant (<= 256 rows, fp32 planes, <= 8 of them, hidden <= 4096): one memory round trip and a register budget that
// leaves room for the next kernel's CTA.
//  * every load of a thread -- x and ALL split planes of both of its column groups -- is issued before the first add.  The
//    generic kernel sums the planes in a loop whose trip count is a run-time value: the compiler keeps it rolled, the add of
//    plane z stalls on its load and the load of plane z + 1 is only issued after it, i.e. n_splits dependent L2 round trips.
//  * 512 threads x 88 registers: 4 warps x 88 x 32 = 11 K of the 16 K registers of each SM sub-partition, which leaves room for
//    the 2 warps x 80 registers the next GEMM's CTA (6 warps) puts on a sub-partition.  The generic kernel runs 1024 threads x
//    64 registers = the whole register file: on the 64 SMs that host a row, the next GEMM's CTA could not start until the norm
//    had finished, and its weight prefetch before the PDL wait was lost on 43 % of the SMs (tools/trace_gemm.py).
// predicated 16-byte load as a volatile asm: volatile asm statements keep their program order, so a block of these followed by
// pin4() on every result forces "all loads issued, then one wait" (nvcc otherwise sinks each load next to its add to save
// registers, which re-creates the dependent-round-trip chain)
__device__ __forceinline__ float4 ldg_f4_pred(const float* p, bool pred) {
    float4 r = make_float4(0.f, 0.f, 0.f, 0.f);
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %5, 0;\n\t@q ld.global.v4.f32 {%0, %1, %2, %3}, [%4];\n\t}"
                 : "+f"(r.x), "+f"(r.y), "+f"(r.z), "+f"(r.w) : "l"(p), "r"((int)pred) : "memory");
    return r;
}
__device__ __forceinline__ void pin4(float4& v) { asm volatile("" : "+f"(v.x), "+f"(v.y), "+f"(v.z), "+f"(v.w)); }

template <int MAXV>
__global__ void __maxnreg__(88)
add_rmsnorm_dec_kernel(float* __restrict__ x, PartIn part, const __nv_bfloat16* __restrict__ w,
                       __nv_bfloat16* __restrict__ xn, int hidden, float eps, unsigned* __restrict__ zero, int zero_n,
                       float* __restrict__ rowss_out, int n_part_out) {
    constexpr int THREADS = 512, NP = 8;
    __shared__ float red[32];
    __shared__ float one_s;
    if (threadIdx.x == 0) one_s = 1.f;
    griddep_launch();
    const int tr_slot = trace_begin(TR_NORM);
    const int row = blockIdx.x;
    float* xr = x + (size_t)row * hidden;
    uint2 wv[MAXV];
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
        const int c = (threadIdx.x + i * THREADS) * 4;
        wv[i] = c < hidden ? *reinterpret_cast<const uint2*>(w + c) : make_uint2(0u, 0u);
    }
    griddep_wait();
    trace_dep(tr_slot);
    for (int i = blockIdx.x * THREADS + threadIdx.x; i < zero_n; i += gridDim.x * THREADS) zero[i] = 0u;
    const int ns = part.ptr ? part.n_splits : 0;
    float4 v[MAXV], t[MAXV][NP];
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
        const int c = (threadIdx.x + i * THREADS) * 4;
        const bool on = c < hidden;
        v[i] = ldg_f4_pred(xr + c, on);
        const float* base = reinterpret_cast<const float*>(part.ptr) + (size_t)row * part.ld + c;
#pragma unroll
        for (int z = 0; z < NP; ++z) t[i][z] = ldg_f4_pred(base + (size_t)z * part.split_stride, on && z < ns);
    }
    // ptxas re-interleaves loads and adds to save registers (even across a barrier or an empty asm), which re-creates the chain.
    // What it cannot move: every add below is an FMA with a factor 1.0f that is read from shared memory AFTER a block barrier
    // that follows the loads -- fma(t, 1, acc) == acc + t exactly, and no add can issue before all 18 loads have.
    __syncthreads();
    const float one = *reinterpret_cast<volatile float*>(&one_s);
    float ss = 0.f;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
        // same association as part_load4: (((p0 + p1) + p2) + ...) first, then x + that sum
        float4 acc = t[i][0];
#pragma unroll
        for (int z = 1; z < NP; ++z) {
            acc.x = fmaf(t[i][z].x, one, acc.x); acc.y = fmaf(t[i][z].y, one, acc.y);
            acc.z = fmaf(t[i][z].z, one, acc.z); acc.w = fmaf(t[i][z].w, one, acc.w);
        }
        v[i].x += acc.x; v[i].y += acc.y; v[i].z += acc.z; v[i].w += acc.w;
        ss += v[i].x * v[i].x + v[i].y * v[i].y + v[i].z * v[i].z + v[i].w * v[i].w;
    }
    if (ns > 0) {
#pragma unroll
        for (int i = 0; i < MAXV; ++i) {
            const int c = (threadIdx.x + i * THREADS) * 4;
            if (c < hidden) *reinterpret_cast<float4*>(xr + c) = v[i];
        }
    }
    ss = block_sum(ss, red);
    if (rowss_out != nullptr && (int)threadIdx.x < n_part_out)
        rowss_out[(size_t)row * n_part_out + threadIdx.x] = threadIdx.x == 0 ? ss : 0.f;
    const float inv = rowss_out != nullptr ? 1.f : rsqrtf(ss / (float)hidden + eps);
    __nv_bfloat16* out = xn + (size_t)row * hidden;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
        const int c = (threadIdx.x + i * THREADS) * 4;
        if (c < hidden) {
            uint2 o;
            o.x = pack_bf16(v[i].x * inv * bf16_lo(wv[i].x), v[i].y * inv * bf16_hi(wv[i].x));
            o.y = pack_bf16(v[i].z * inv * bf16_lo(wv[i].y), v[i].w * inv * bf16_hi(wv[i].y));
            *reinterpret_cast<uint2*>(out + c) = o;
        }
    }
    trace_end(tr_slot);
}

void launch_add_rmsnorm(float* x, PartIn part, const __nv_bfloat16* w, __nv_bfloat16* xn, int rows,
                        int hidden, float eps, cudaStream_t st, unsigned* zero, int zero_n, float* rowss_out, int n_part_out) {
    if (rows <= 0 || hidden > 8192) return;
    const bool no_dec = getenv("RR_NO_DEC_NORM") != nullptr;     // A/B switch (tools/decode_ab.py); launches are graph-captured
    if (rows <= 256 && hidden <= 4096 && !no_dec && (part.ptr == nullptr || (!part.is_bf16 && part.n_splits <= 8)))
        launch_pdl(add_rmsnorm_dec_kernel<2>, dim3(rows), dim3(512), 0, st, x, part, w, xn, hidden, eps, zero, zero_n,
                   rowss_out, n_part_out);
    else if (rows <= 256)
        launch_pdl(add_rmsnorm_kernel<1024, 2>, dim3(rows), dim3(1024), 0, st, x, part, w, xn, hidden, eps, zero, zero_n,
                   rowss_out, n_part_out);
    else if (hidden <= 4096)      // fewer registers -> more rows in flight per SM (HBM-bound at thousands of rows)
        launch_pdl(add_rmsnorm_kernel<256, 4>, dim3(rows), dim3(256), 0, st, x, part, w, xn, hidden, eps, zero, zero_n,
                   rowss_out, n_part_out);
    else
        launch_pdl(add_rmsnorm_kernel<256, 8>, dim3(rows), dim3(256), 0, st, x, part, w, xn, hidden, eps, zero, zero_n,
                   rowss_out, n_part_out);
}

// ---- SiLU(gate) * up -----------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
silu_mul_kernel(PartIn gu, __nv_bfloat16* __restrict__ act, int inter) {
    griddep_launch();
    const int tr_slot = trace_begin(TR_SILU);
    griddep_wait();
    trace_dep(tr_slot);
    const int row = blockIdx.y;
    const int c = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (c >= inter) return;
    const float4 g = part_load4(gu, row, c);
    const float4 u = part_load4(gu, row, inter + c);
    auto f = [](float a, float b) { return __fdividef(a, 1.f + __expf(-a)) * b; };   // same formula as silu_mul (rr_gemm.cu)
    uint2 o;
    o.x = pack_bf16(f(g.x, u.x), f(g.y, u.y));
    o.y = pack_bf16(f(g.z, u.z), f(g.w, u.w));
    *reinterpret_cast<uint2*>(act + (size_t)row * inter + c) = o;
    trace_end(tr_slot);
}

void launch_silu_mul(PartIn gu, __nv_bfloat16* act, int rows, int inter, cudaStream_t st) {
    if (rows <= 0) return;
    dim3 grid((inter / 4 + 255) / 256, rows);
    launch_pdl(silu_mul_kernel, grid, dim3(256), 0, st, gu, act, inter);
}

// ---- K6 RoPE + KV-cache append --------------------------------------------------------------------
// head_dim = 128, HF "rotate_half" convention: pairs (i, i + 64), inv_freq_i = theta^(-i/64).
// cos/sin come from a table [ctx_max][64] (float2) built once per engine in double precision;
// without a table (kernel-level tests) they are computed inline.
__global__ void rope_table_kernel(float2* __restrict__ table, int ctx_max, double theta, int half) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= ctx_max * 64) return;
    const int pos = idx >> 6, i = idx & 63;
    if (i >= half) { table[idx] = make_float2(1.f, 0.f); return; }
    const double inv_freq = pow(theta, -(double)i / (double)half);
    // the oracle (and HF) form the angle in fp32: pos * float(inv_freq)
    const float ang = (float)pos * (float)inv_freq;
    table[idx] = make_float2((float)cos((double)ang), (float)sin((double)ang));
}

void launch_rope_table(float2* table, int ctx_max, float theta, int head_dim, cudaStream_t st) {
    const int n = ctx_max * 64;
    rope_table_kernel<<<(n + 255) / 256, 256, 0, st>>>(table, ctx_max, (double)theta, head_dim / 2);
}

__device__ __forceinline__ float2 part_load2(const PartIn& p, int row, int col) {   // 2 consecutive columns
    if (p.is_bf16) {
        const uint32_t v = *reinterpret_cast<const uint32_t*>(
            reinterpret_cast<const __nv_bfloat16*>(p.ptr) + (size_t)row * p.ld + col);
        return make_float2(bf16_lo(v), bf16_hi(v));
    }
    const float* base = reinterpret_cast<const float*>(p.ptr) + (size_t)row * p.ld + col;
    float2 acc = *reinterpret_cast<const float2*>(base);
    for (int z = 1; z < p.n_splits; ++z) {
        const float2 t = *reinterpret_cast<const float2*>(base + (size_t)z * p.split_stride);
        acc.x += t.x; acc.y += t.y;
    }
    return acc;
}

__global__ void __launch_bounds__(256)
rope_kv_kernel(RopeArgs a) {
    griddep_launch();
    const int tr_slot = trace_begin(TR_ROPE);
    griddep_wait();
    trace_dep(tr_slot);
    const int row = blockIdx.x;
    const int slot = a.slot[row];
    if (slot < 0) return;
    const int pos = a.pos[row];
    // work items of 2 rotation pairs: (head, i..i+1) for q heads then k heads, then v copies (4 elements).
    // hd = true head dim: rotation pairs (i, i + hd/2); destination rows are padded to 128 (pad stays zero).
    const int hd = a.head_dim, half = hd >> 1, ipw = half >> 1, vpw = hd >> 2;      // items per head
    const int n_q = a.n_heads * ipw, n_k = a.n_kv_heads * ipw;
    const int total = n_q + n_k + a.n_kv_heads * vpw;
    const float l2t = a.table ? 0.f : log2f(a.theta);
    for (int it = threadIdx.x; it < total; it += blockDim.x) {
        if (it < n_q + n_k) {
            const bool is_q = it < n_q;
            const int j = is_q ? it : it - n_q;
            const int head = j / ipw, i = (j % ipw) * 2;
            const int col = (is_q ? 0 : a.n_heads * hd) + head * hd + i;
            const float2 lo = part_load2(a.qkv, row, col);
            const float2 hi = part_load2(a.qkv, row, col + half);
            float c0, s0, c1, s1;
            if (a.table) {
                const float4 t = *reinterpret_cast<const float4*>(a.table + (size_t)pos * 64 + i);
                c0 = t.x; s0 = t.y; c1 = t.z; s1 = t.w;
            } else {
                sincosf((float)pos * exp2f(-l2t * (float)i / (float)half), &s0, &c0);
                sincosf((float)pos * exp2f(-l2t * (float)(i + 1) / (float)half), &s1, &c1);
            }
            const uint32_t o_lo = pack_bf16(lo.x * c0 - hi.x * s0, lo.y * c1 - hi.y * s1);
            const uint32_t o_hi = pack_bf16(hi.x * c0 + lo.x * s0, hi.y * c1 + lo.y * s1);
            __nv_bfloat16* dst = is_q
                ? a.q_out + (size_t)row * (a.n_heads * 128) + head * 128 + i
                : a.k_cache + (((size_t)slot * a.n_kv_heads + head) * a.ctx_max + pos) * 128 + i;
            *reinterpret_cast<uint32_t*>(dst) = o_lo;
            *reinterpret_cast<uint32_t*>(dst + half) = o_hi;
        } else {
            const int j = it - n_q - n_k;            // 4 elements each
            const int head = j / vpw, i4 = (j % vpw) * 4;
            const int col = (a.n_heads + a.n_kv_heads) * hd + head * hd + i4;
            const float4 v = part_load4(a.qkv, row, col);
            __nv_bfloat16* dst = a.v_cache + (((size_t)slot * a.n_kv_heads + head) * a.ctx_max + pos) * 128 + i4;
            uint2 o;
            o.x = pack_bf16(v.x, v.y);
            o.y = pack_bf16(v.z, v.w);
            *reinterpret_cast<uint2*>(dst) = o;
        }
    }
    trace_end(tr_slot);
}

void launch_rope_kv(const RopeArgs& a, cudaStream_t st) {
    if (a.rows <= 0) return;
    launch_pdl(rope_kv_kernel, dim3(a.rows), dim3(256), 0, st, a);
}

// ---- greedy argmax (lowest index wins ties) ------------------------------------------------------
__global__ void __launch_bounds__(1024)
argmax_kernel(PartIn logits, int vocab, int32_t* __restrict__ out_tok, float* __restrict__ out_val,
              const int32_t* __restrict__ row_active, int32_t* __restrict__ pos_inc) {
    __shared__ float s_v[32];
    __shared__ int s_i[32];
    griddep_launch();
    const int tr_slot = trace_begin(TR_ARGMAX);
    griddep_wait();
    trace_dep(tr_slot);
    const int row = blockIdx.x;
    if (row_active && row_active[row] < 0) return;
    const float* r = reinterpret_cast<const float*>(logits.ptr) + (size_t)row * logits.ld;
    float best = -INFINITY;
    int bi = 0x7fffffff;
    const int v4 = vocab & ~3;
    // 8 independent 16-byte loads per round: the compare chain is loop-carried, and with one load per iteration the 31
    // iterations of a 128 k vocabulary were 31 dependent memory round trips (51 us per step; now ~4 rounds)
    constexpr int U = 8;
    const int stride = blockDim.x * 4;
    for (int c0 = threadIdx.x * 4; c0 < v4; c0 += stride * U) {
        float4 v[U];
#pragma unroll
        for (int k = 0; k < U; ++k) {
            const int c = c0 + k * stride;
            v[k] = c < v4 ? *reinterpret_cast<const float4*>(r + c) : make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
        }
#pragma unroll
        for (int k = 0; k < U; ++k) {                      // increasing index order: the lowest index wins ties
            const int c = c0 + k * stride;
            if (v[k].x > best) { best = v[k].x; bi = c; }
            if (v[k].y > best) { best = v[k].y; bi = c + 1; }
            if (v[k].z > best) { best = v[k].z; bi = c + 2; }
            if (v[k].w > best) { best = v[k].w; bi = c + 3; }
        }
    }
    for (int c = v4 + threadIdx.x; c < vocab; c += blockDim.x) {
        const float v = r[c];
        if (v > best) { best = v; bi = c; }
    }
    auto better = [](float v, int i, float bv, int bi_) { return v > bv || (v == bv && i < bi_); };
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (better(ov, oi, best, bi)) { best = ov; bi = oi; }
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) { s_v[warp] = best; s_i[warp] = bi; }
    __syncthreads();
    if (warp == 0) {
        const int nw = blockDim.x >> 5;
        best = lane < nw ? s_v[lane] : -INFINITY;
        bi = lane < nw ? s_i[lane] : 0x7fffffff;
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, best, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (better(ov, oi, best, bi)) { best = ov; bi = oi; }
        }
        if (lane == 0) {
            out_tok[row] = bi;
            if (out_val) out_val[row] = best;
            if (pos_inc) pos_inc[row] += 1;
        }
    }
    trace_end(tr_slot);
}

void launch_argmax(PartIn logits, int rows, int vocab, int32_t* out_tok, float* out_val,
                   const int32_t* row_active, int32_t* pos_inc, cudaStream_t st) {
    if (rows <= 0) return;
    launch_pdl(argmax_kernel, dim3(rows), dim3(1024), 0, st, logits, vocab, out_tok, out_val, row_active, pos_inc);
}

void rr_trace_set_elementwise(unsigned long long* p) { rr_trace_set_local(p); }

}  // namespace rr
