// rr_gemm.cu — the path's one dense contraction (QKV / O / gate-up / down / lm_head projections)
// on 5th-generation tensor cores: tcgen05.mma (UTCHMMA) with fp32 accumulators in TMEM,
// operands staged by TMA (UTMALDG) into 128B-swizzled shared memory, persistent
// warp-specialised CTAs (1 TMA warp, 1 MMA warp, 4 epilogue warps), double-buffered TMEM.
//
//   D[a, b] = sum_k A[a, k] * B[b, k]          A: [rowsA, K] bf16, B: [rowsB, K] bf16 (both K-major)
//
// Two orientations of the same kernel:
//   * prefill  (OUT_ROWMAJOR_BF16):  A = activations [T, K], B = weight [N, K]  -> C[T, N] bf16
//   * decode   (OUT_TRANSPOSED_F32): A = weight [N, K] (UMMA M side, streamed once from HBM),
//                                    B = activations [batch<=BN, K]; fp32 partial planes
//                                    P[z][b][n] reduced by the consumer kernel (rr_elementwise.cu).
//     Work split for decode: uniform split-K (splits planes); the wave-quantisation tail of the big gate/up
//     projection is removed by the fused MLP kernel below (per-slice dataflow), not by a stream-K split.
//
// PDL: the weight operand is constant, its first pipeline stages are requested before
// griddepcontrol.wait; only the activation operand and the output wait for the preceding kernel.
//
// Replaces: the remote bedrock:InvokeModel call (reference iam/policy.json:8,
// src/demo_cris.py:233-238) — there is no reference kernel; see DESIGN.md §kernels.
#include "rr_ptx.cuh"
#include "rr_launch.cuh"
#include "rr_kernels.h"

#include <mutex>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

namespace rr {

constexpr int BLOCK_A = 128;   // UMMA M
constexpr int BLOCK_K = 64;    // 64 bf16 = 128 B = one swizzle row
constexpr int UMMA_K = 16;
constexpr int GEMM_THREADS = 192;
constexpr int GROUP_A = 16;    // raster group: 16 A tiles share the streamed B tiles through L2

// CAP bounds the smem ring.
template <int BN, int CAP = 8>
struct GemmCfg {
    static constexpr int kStageBytesA = BLOCK_A * BLOCK_K * 2;
    static constexpr int kStageBytesB = BN * BLOCK_K * 2;
    static constexpr int kStageBytes = kStageBytesA + kStageBytesB;
    static constexpr int kStagesRaw = (200 * 1024) / kStageBytes;
    static constexpr int kStages = kStagesRaw > CAP ? CAP : kStagesRaw;
    static constexpr uint32_t kTmemCols =
        (2 * BN <= 32) ? 32 : (2 * BN <= 64) ? 64 : (2 * BN <= 128) ? 128 : (2 * BN <= 256) ? 256 : 512;
    static constexpr int kSmemBytes = kStages * kStageBytes + 1024 /*align slack*/ + 256 /*barriers*/;
    static constexpr int kSiluStageBytes = 2 * 32 * 64 * 4;   // OUT_TRANSPOSED_SILU: up-row exchange, 2 x [32 cols][64 rows] fp32
};
// TMA-store epilogues of the decode orientation (BN <= 64): the planes tile [BN][128] fp32 (one 3-D TMA store per item); the
// fused MLP kernel aliases it with the up-row exchange (16 KB) + the act tile [BN][64] bf16 of the SiLU epilogue.
template <int BN>
constexpr int planes_stage_bytes() { return BN <= 64 ? BN * 128 * 4 : 0; }
template <int BN>
constexpr int mlp_stage_bytes() {
    constexpr int a = planes_stage_bytes<BN>(), b = GemmCfg<BN>::kSiluStageBytes + (BN <= 64 ? BN * 64 * 2 : 0);
    return a > b ? a : b;
}
template <int MODE>
__host__ __device__ constexpr bool decode_orient() { return MODE == OUT_TRANSPOSED_F32 || MODE == OUT_TRANSPOSED_SILU; }
template <int BN, int MODE, int CAP = 8>
constexpr int gemm_smem_bytes() {
    // SILU (decode): up-row exchange; RESID (prefill): per-warp 32 x 36 fp32 transpose tiles (18 KB) -- same slot
    return GemmCfg<BN, CAP>::kSmemBytes +
           (MODE == OUT_TRANSPOSED_SILU ? GemmCfg<BN, CAP>::kSiluStageBytes : MODE == OUT_ROWMAJOR_RESID ? 4 * 32 * 36 * 4 :
            MODE == OUT_TRANSPOSED_F32 ? planes_stage_bytes<BN>() : 0);
}
// SiLU(g) * u.  __fdividef, not `/`: the IEEE division compiles to a convergence-barrier region with a slow-path CALL per element,
// which serialises the unrolled epilogue loops (2 ulp of fp32 before the bf16 rounding; 0 instead of -1e-36 for g < -87).
__device__ __forceinline__ float silu_mul(float g, float u) { return __fdividef(g, 1.f + __expf(-g)) * u; }

struct WorkItem {
    int a_tile, b_tile, z, kb0, kb1;
};

// Deterministic per-CTA sequence of work items (uniform split-K); every warp role walks the same sequence.
// (A stream-K split -- k-block units dealt evenly to the SMs regardless of tile boundaries -- was measured in round 1:
// 4.55 -> 4.92 ms per decode step, the consumers read more planes than the better balance returns; removed.)
struct WorkSched {
    int tilesA, tilesB, splits, kblocks, n_work, w;

    __device__ __forceinline__ void init(int rowsA, int rowsB, int K, int splits_, int BN) {
        tilesA = (rowsA + BLOCK_A - 1) / BLOCK_A;
        tilesB = (rowsB + BN - 1) / BN;
        kblocks = (K + BLOCK_K - 1) / BLOCK_K;
        splits = splits_;
        n_work = tilesA * tilesB * splits;
        w = blockIdx.x;
    }
    __device__ __forceinline__ bool next(WorkItem& it) {
        if (w >= n_work) return false;
        it.z = w % splits;
        const int q = w / splits;
        const int per_group = GROUP_A * tilesB;
        const int g = q / per_group;
        const int r = q - g * per_group;
        const int a0 = g * GROUP_A;
        const int ga = min(GROUP_A, tilesA - a0);
        it.a_tile = a0 + r % ga;
        it.b_tile = r / ga;
        it.kb0 = (int)(((long long)kblocks * it.z) / splits);
        it.kb1 = (int)(((long long)kblocks * (it.z + 1)) / splits);
        w += gridDim.x;
        return true;
    }
};

// Epilogue of one work item: TMEM accumulator (this warp's 32 lanes x BN columns at taddr0) -> global memory, in the
// layout / fusion selected by MODE.  Shared by the 1-CTA kernel, the 2-CTA kernel and (by copy) the chain kernel.
template <int BN, int MODE>
__device__ __forceinline__ void epilogue_item(uint32_t taddr0, int a_row, const WorkItem& t, int quarter, int lane,
                                              void* __restrict__ out, int rowsA, int rowsB, int ldo, int ld_rows,
                                              const RopeEpi& rope, float* silu_stage) {
    constexpr int CH = (BN >= 32) ? 32 : 16;
    // deferred RMSNorm, consumer side: this thread's row of the A operand was bf16(x * gamma); scale by 1 / rms(x)
    float rinv = 1.f;
    if constexpr (MODE == OUT_ROWMAJOR_ROPE || MODE == OUT_ROWMAJOR_SILU || MODE == OUT_ROWMAJOR_BF16) {
        if (rope.n_part > 0 && a_row < rowsA) {
            const float* ps = rope.rowss + (size_t)a_row * rope.n_part;
            float ss = 0.f;
            for (int j = 0; j < rope.n_part; ++j) ss += ps[j];
            rinv = rsqrtf(ss * rope.inv_hidden + rope.eps);
        }
    }
    if constexpr (MODE == OUT_TRANSPOSED_SILU) {
        // gate/up rows are interleaved in blocks of 64: lanes 0..63 of the tile hold gate rows, lanes 64..127 the
        // matching up rows.  The up warps hand their values over through smem ([col][row] -> conflict-free), the
        // gate warps write act[b][n] = silu(g) * u as bf16.  rowsA = 2 * inter (interleaved), ldo = inter.
        float* stage = silu_stage;
        const bool is_up = quarter >= 2;
        const int r64 = (quarter & 1) * 32 + lane;
        const int n = t.a_tile * 64 + r64;
        __nv_bfloat16* act = reinterpret_cast<__nv_bfloat16*>(out);
#pragma unroll 1
        for (int c = 0; c < BN; c += 32) {
            float* buf = stage + ((c >> 5) & 1) * (32 * 64);
            uint32_t v[32];
            tmem_ld_32x32b_x32(taddr0 + c, v);
            tmem_ld_wait();
            if (is_up) {
#pragma unroll
                for (int j = 0; j < 32; ++j) buf[j * 64 + r64] = __uint_as_float(v[j]);
            }
            asm volatile("bar.sync 2, 128;" ::: "memory");
            if (!is_up && 2 * n < rowsA) {
                const int b0 = t.b_tile * BN + c;
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const int b = b0 + j;
                    if (b < rowsB)
                        act[(size_t)b * ldo + n] = __float2bfloat16(silu_mul(__uint_as_float(v[j]), buf[j * 64 + r64]));
                }
            }
        }
    } else if constexpr (MODE == OUT_ROWMAJOR_ROPE) {
        // 256 columns = two 128-wide heads of the fused qkv projection; thread = token row.
        const bool row_ok = a_row < rowsA;
        const int slot = row_ok ? rope.slot[a_row] : -1;
        const int pos = row_ok ? rope.pos[a_row] : 0;
        const bool live = slot >= 0;
        const float2* tab = rope.table + (size_t)pos * 64;
#pragma unroll 1
        for (int hb = 0; hb < BN / 128; ++hb) {
            const int H = t.b_tile * (BN / 128) + hb;                  // head index in [q heads | k heads | v heads]
            if (H * 128 >= rowsB) break;
            const uint32_t tcol = taddr0 + hb * 128;
            if (H < rope.n_heads + rope.n_kv_heads) {
                __nv_bfloat16* dst = H < rope.n_heads
                    ? rope.q_out + (size_t)a_row * (rope.n_heads * 128) + H * 128
                    : rope.k_cache + (((size_t)slot * rope.n_kv_heads + (H - rope.n_heads)) * rope.ctx_max + pos) * 128;
#pragma unroll 1
                for (int c = 0; c < 64; c += 32) {
                    uint32_t lo[32], hi[32];
                    tmem_ld_32x32b_x32(tcol + c, lo);
                    tmem_ld_32x32b_x32(tcol + 64 + c, hi);
                    tmem_ld_wait();
                    if (live) {
#pragma unroll
                        for (int j = 0; j < 32; j += 8) {
                            uint4 plo, phi;
                            uint32_t* wl = reinterpret_cast<uint32_t*>(&plo);
                            uint32_t* wh = reinterpret_cast<uint32_t*>(&phi);
#pragma unroll
                            for (int q = 0; q < 4; ++q) {
                                const float4 cs = *reinterpret_cast<const float4*>(tab + c + j + 2 * q);   // 2 pairs
                                const float l0 = __uint_as_float(lo[j + 2 * q]) * rinv, l1 = __uint_as_float(lo[j + 2 * q + 1]) * rinv;
                                const float h0 = __uint_as_float(hi[j + 2 * q]) * rinv, h1 = __uint_as_float(hi[j + 2 * q + 1]) * rinv;
                                wl[q] = pack_bf16(l0 * cs.x - h0 * cs.y, l1 * cs.z - h1 * cs.w);
                                wh[q] = pack_bf16(h0 * cs.x + l0 * cs.y, h1 * cs.z + l1 * cs.w);
                            }
                            *reinterpret_cast<uint4*>(dst + c + j) = plo;
                            *reinterpret_cast<uint4*>(dst + 64 + c + j) = phi;
                        }
                    }
                }
            } else {
                __nv_bfloat16* dst = rope.v_cache +
                    (((size_t)slot * rope.n_kv_heads + (H - rope.n_heads - rope.n_kv_heads)) * rope.ctx_max + pos) * 128;
#pragma unroll 1
                for (int c = 0; c < 128; c += 32) {
                    uint32_t v[32];
                    tmem_ld_32x32b_x32(tcol + c, v);
                    tmem_ld_wait();
                    if (live) {
#pragma unroll
                        for (int j = 0; j < 32; j += 8) {
                            uint4 pk;
                            pk.x = pack_bf16(__uint_as_float(v[j + 0]) * rinv, __uint_as_float(v[j + 1]) * rinv);
                            pk.y = pack_bf16(__uint_as_float(v[j + 2]) * rinv, __uint_as_float(v[j + 3]) * rinv);
                            pk.z = pack_bf16(__uint_as_float(v[j + 4]) * rinv, __uint_as_float(v[j + 5]) * rinv);
                            pk.w = pack_bf16(__uint_as_float(v[j + 6]) * rinv, __uint_as_float(v[j + 7]) * rinv);
                            *reinterpret_cast<uint4*>(dst + c + j) = pk;
                        }
                    }
                }
            }
        }
    } else if constexpr (MODE == OUT_ROWMAJOR_RESID) {
        float* xres = reinterpret_cast<float*>(out);
        const bool defer = rope.xhat != nullptr;       // also emit bf16(x * gamma) and sum(x^2) of this row over the tile
        if (silu_stage != nullptr) {
            // Coalesced residual add.  TMEM hands every thread one ROW (32 consecutive columns = one 128-byte line per
            // chunk), so a direct read-modify-write issues 16-byte pieces of 32 different lines per instruction: 32 LSU
            // wavefronts and half-used sectors.  Each warp instead transposes its 32 x 32 chunk through 4.5 KB of shared
            // memory (row pitch 36 floats: conflict-free both ways) and lets 8 lanes cover one line: 4 full lines per
            // instruction.
            float* stg = silu_stage + (quarter * 32) * 36;              // this warp's [32][36] tile
            const int sub_row = lane >> 3, sub_col = (lane & 7) * 4;
            const int row0 = t.a_tile * BLOCK_A + quarter * 32;         // first of this warp's 32 rows
            float ssr[8];                                               // deferred norm: sum(x^2) pieces of rows 4i + sub_row
#pragma unroll
            for (int i = 0; i < 8; ++i) ssr[i] = 0.f;
#pragma unroll 1
            for (int c = 0; c < BN; c += 32) {
                uint32_t v[32];
                tmem_ld_32x32b_x32(taddr0 + c, v);
                tmem_ld_wait();
                const int b0 = t.b_tile * BN + c;
                if (b0 + 32 <= rowsB) {
#pragma unroll
                    for (int j = 0; j < 32; j += 4)
                        *reinterpret_cast<float4*>(stg + lane * 36 + j) =
                            make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
                    __syncwarp();
                    // all eight loads first: a store between them would fence the later loads (possible aliasing) and
                    // turn eight independent L2 round trips into a chain
                    float4 xs[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const int r = 4 * i + sub_row;
                        xs[i] = (row0 + r < rowsA) ? *reinterpret_cast<const float4*>(xres + (size_t)(row0 + r) * ldo + b0 + sub_col)
                                                   : make_float4(0.f, 0.f, 0.f, 0.f);
                    }
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const int r = 4 * i + sub_row;
                        if (row0 + r < rowsA) {
                            const float4 a4 = *reinterpret_cast<const float4*>(stg + r * 36 + sub_col);
                            float4 x4 = xs[i];
                            x4.x += a4.x; x4.y += a4.y; x4.z += a4.z; x4.w += a4.w;
                            *reinterpret_cast<float4*>(xres + (size_t)(row0 + r) * ldo + b0 + sub_col) = x4;
                            if (defer) {
                                const uint2 gw = *reinterpret_cast<const uint2*>(rope.gamma + b0 + sub_col);
                                ssr[i] += x4.x * x4.x + x4.y * x4.y + x4.z * x4.z + x4.w * x4.w;
                                uint2 pk;
                                pk.x = pack_bf16(x4.x * bf16_lo(gw.x), x4.y * bf16_hi(gw.x));
                                pk.y = pack_bf16(x4.z * bf16_lo(gw.y), x4.w * bf16_hi(gw.y));
                                *reinterpret_cast<uint2*>(rope.xhat + (size_t)(row0 + r) * ldo + b0 + sub_col) = pk;
                            }
                        }
                    }
                    __syncwarp();
                } else {
                    // ragged last chunk: thread = row, scalar; its sum(x^2) joins the row's lane group through smem
                    float ss_tail = 0.f;
                    if (a_row < rowsA) {
                        float* dst = xres + (size_t)a_row * ldo + b0;
                        for (int j = 0; j < 32; ++j)
                            if (b0 + j < rowsB) {
                                const float xv = dst[j] + __uint_as_float(v[j]);
                                dst[j] = xv;
                                if (defer) {
                                    ss_tail += xv * xv;
                                    rope.xhat[(size_t)a_row * ldo + b0 + j] = __float2bfloat16(xv * __bfloat162float(rope.gamma[b0 + j]));
                                }
                            }
                    }
                    if (defer) {
                        stg[lane * 36] = ss_tail;                     // row `lane` of this warp
                        __syncwarp();
#pragma unroll
                        for (int i = 0; i < 8; ++i)
                            if ((lane & 7) == 0) ssr[i] += stg[(4 * i + sub_row) * 36];
                        __syncwarp();
                    }
                }
            }
            if (defer) {
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    float v2 = ssr[i];
                    v2 += __shfl_xor_sync(0xffffffffu, v2, 1);
                    v2 += __shfl_xor_sync(0xffffffffu, v2, 2);
                    v2 += __shfl_xor_sync(0xffffffffu, v2, 4);
                    const int r = row0 + 4 * i + sub_row;
                    if ((lane & 7) == 0 && r < rowsA) rope.rowss_out[(size_t)r * rope.n_part_out + t.b_tile] = v2;
                }
            }
        } else {
            float ss = 0.f;
    #pragma unroll 1
            for (int c = 0; c < BN; c += 32) {
                uint32_t v[32];
                tmem_ld_32x32b_x32(taddr0 + c, v);
                tmem_ld_wait();
                const int b0 = t.b_tile * BN + c;
                if (a_row < rowsA) {
                    float* dst = xres + (size_t)a_row * ldo + b0;
                    if (b0 + 32 <= rowsB) {
                        __nv_bfloat16* hdst = defer ? rope.xhat + (size_t)a_row * ldo + b0 : nullptr;
    #pragma unroll
                        for (int j = 0; j < 32; j += 8) {
                            float4 x4 = *reinterpret_cast<const float4*>(dst + j);
                            float4 y4 = *reinterpret_cast<const float4*>(dst + j + 4);
                            x4.x += __uint_as_float(v[j + 0]); x4.y += __uint_as_float(v[j + 1]);
                            x4.z += __uint_as_float(v[j + 2]); x4.w += __uint_as_float(v[j + 3]);
                            y4.x += __uint_as_float(v[j + 4]); y4.y += __uint_as_float(v[j + 5]);
                            y4.z += __uint_as_float(v[j + 6]); y4.w += __uint_as_float(v[j + 7]);
                            *reinterpret_cast<float4*>(dst + j) = x4;
                            *reinterpret_cast<float4*>(dst + j + 4) = y4;
                            if (defer) {
                                const uint4 gw = *reinterpret_cast<const uint4*>(rope.gamma + b0 + j);
                                ss += x4.x * x4.x + x4.y * x4.y + x4.z * x4.z + x4.w * x4.w
                                    + y4.x * y4.x + y4.y * y4.y + y4.z * y4.z + y4.w * y4.w;
                                uint4 pk;
                                pk.x = pack_bf16(x4.x * bf16_lo(gw.x), x4.y * bf16_hi(gw.x));
                                pk.y = pack_bf16(x4.z * bf16_lo(gw.y), x4.w * bf16_hi(gw.y));
                                pk.z = pack_bf16(y4.x * bf16_lo(gw.z), y4.y * bf16_hi(gw.z));
                                pk.w = pack_bf16(y4.z * bf16_lo(gw.w), y4.w * bf16_hi(gw.w));
                                *reinterpret_cast<uint4*>(hdst + j) = pk;
                            }
                        }
                    } else {
                        for (int j = 0; j < 32; ++j)
                            if (b0 + j < rowsB) {
                                const float xv = dst[j] + __uint_as_float(v[j]);
                                dst[j] = xv;
                                if (defer) {
                                    ss += xv * xv;
                                    rope.xhat[(size_t)a_row * ldo + b0 + j] = __float2bfloat16(xv * __bfloat162float(rope.gamma[b0 + j]));
                                }
                            }
                    }
                }
            }
            if (defer && a_row < rowsA) rope.rowss_out[(size_t)a_row * rope.n_part_out + t.b_tile] = ss;
        }
    } else if constexpr (MODE == OUT_ROWMAJOR_SILU) {
        // BN == 256 weight rows = [gate 64 | up 64 | gate 64 | up 64]: a token's gate and up values sit in the same
        // TMEM lane, so silu(g) * u needs no exchange; 128 output columns per tile, ldo = inter.
        __nv_bfloat16* act = reinterpret_cast<__nv_bfloat16*>(out);
        const int n_out = rowsB >> 1;
#pragma unroll 1
        for (int hb = 0; hb < BN / 128; ++hb) {
#pragma unroll 1
            for (int c = 0; c < 64; c += 32) {
                uint32_t vg[32], vu[32];
                tmem_ld_32x32b_x32(taddr0 + hb * 128 + c, vg);
                tmem_ld_32x32b_x32(taddr0 + hb * 128 + 64 + c, vu);
                tmem_ld_wait();
                if (rope.n_part > 0) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        vg[j] = __float_as_uint(__uint_as_float(vg[j]) * rinv);
                        vu[j] = __float_as_uint(__uint_as_float(vu[j]) * rinv);
                    }
                }
                const int col = t.b_tile * (BN / 2) + hb * 64 + c;
                if (a_row < rowsA) {
                    __nv_bfloat16* dst = act + (size_t)a_row * ldo + col;
                    if (col + 32 <= n_out) {
#pragma unroll
                        for (int j = 0; j < 32; j += 8) {
                            uint4 pk;
                            pk.x = pack_bf16(silu_mul(__uint_as_float(vg[j + 0]), __uint_as_float(vu[j + 0])),
                                             silu_mul(__uint_as_float(vg[j + 1]), __uint_as_float(vu[j + 1])));
                            pk.y = pack_bf16(silu_mul(__uint_as_float(vg[j + 2]), __uint_as_float(vu[j + 2])),
                                             silu_mul(__uint_as_float(vg[j + 3]), __uint_as_float(vu[j + 3])));
                            pk.z = pack_bf16(silu_mul(__uint_as_float(vg[j + 4]), __uint_as_float(vu[j + 4])),
                                             silu_mul(__uint_as_float(vg[j + 5]), __uint_as_float(vu[j + 5])));
                            pk.w = pack_bf16(silu_mul(__uint_as_float(vg[j + 6]), __uint_as_float(vu[j + 6])),
                                             silu_mul(__uint_as_float(vg[j + 7]), __uint_as_float(vu[j + 7])));
                            *reinterpret_cast<uint4*>(dst + j) = pk;
                        }
                    } else {
                        for (int j = 0; j < 32; ++j)
                            if (col + j < n_out)
                                dst[j] = __float2bfloat16(silu_mul(__uint_as_float(vg[j]), __uint_as_float(vu[j])));
                    }
                }
            }
        }
    } else {
#pragma unroll 1
    for (int c = 0; c < BN; c += CH) {
        uint32_t v[32];
        if constexpr (CH == 32) {
            tmem_ld_32x32b_x32(taddr0 + c, v);
        } else {
            uint32_t v16[16];
            tmem_ld_32x32b_x16(taddr0 + c, v16);
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] = v16[j];
        }
        tmem_ld_wait();
        const int b0 = t.b_tile * BN + c;
        if constexpr (MODE == OUT_ROWMAJOR_BF16) {
            if (rope.n_part > 0) {
#pragma unroll
                for (int j = 0; j < CH; ++j) v[j] = __float_as_uint(__uint_as_float(v[j]) * rinv);
            }
            if (a_row < rowsA) {
                __nv_bfloat16* dst =
                    reinterpret_cast<__nv_bfloat16*>(out) + (size_t)a_row * ldo + b0;
                if (b0 + CH <= rowsB) {
#pragma unroll
                    for (int j = 0; j < CH; j += 8) {
                        uint4 pk;
                        pk.x = pack_bf16(__uint_as_float(v[j + 0]), __uint_as_float(v[j + 1]));
                        pk.y = pack_bf16(__uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
                        pk.z = pack_bf16(__uint_as_float(v[j + 4]), __uint_as_float(v[j + 5]));
                        pk.w = pack_bf16(__uint_as_float(v[j + 6]), __uint_as_float(v[j + 7]));
                        *reinterpret_cast<uint4*>(dst + j) = pk;
                    }
                } else {
                    for (int j = 0; j < CH; ++j)
                        if (b0 + j < rowsB) dst[j] = __float2bfloat16(__uint_as_float(v[j]));
                }
            }
        } else {
            float* dst = reinterpret_cast<float*>(out);
            if (a_row < rowsA) {
#pragma unroll
                for (int j = 0; j < CH; ++j) {
                    const int b = b0 + j;
                    if (b < rowsB)
                        dst[((size_t)t.z * ld_rows + b) * ldo + a_row] = __uint_as_float(v[j]);
                }
            }
        }
    }
    }
}

// ---- TMA-store epilogues (decode orientation, BN <= 64) ---------------------------------------------------------------------
// Under a saturated weight stream an LSU store costs the issuing warp 75-170 ns (tools/trace_mlp.py: 64 four-byte stores
// per thread = 5 us per planes tile, the 2-byte act stores of the SiLU epilogue + the fence = 14 us from "accumulator
// ready" to "tile published", and the down items of the fused MLP kernel wait exactly for that).  Here the 128 epilogue
// threads transpose the tile through shared memory and ONE thread hands it to the TMA engine as a single bulk store.
__device__ __forceinline__ void epi_bar() { asm volatile("bar.sync 4, 128;" ::: "memory"); }

// planes tile: stage[b][n] fp32, b < BN, n < 128 (n = accumulator row = this thread)  ->  P[z][b][a_tile * 128 + n]
template <int BN>
__device__ __forceinline__ void epilogue_planes_tma(uint32_t taddr0, const WorkItem& t, int quarter, int lane, int etid,
                                                    const CUtensorMap* tmOut, float* stage) {
    constexpr int CH = (BN >= 32) ? 32 : 16;
    if (etid == 0) bulk_wait_read0();              // the previous item's store has read the staging tile
    epi_bar();
    float* col = stage + quarter * 32 + lane;
#pragma unroll 1
    for (int c = 0; c < BN; c += CH) {
        uint32_t v[32];
        if constexpr (CH == 32) {
            tmem_ld_32x32b_x32(taddr0 + c, v);
        } else {
            uint32_t v16[16];
            tmem_ld_32x32b_x16(taddr0 + c, v16);
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] = v16[j];
        }
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < CH; ++j) col[(c + j) * 128] = __uint_as_float(v[j]);      // lanes = consecutive n: conflict-free
    }
    fence_proxy_async();                           // generic-proxy smem writes -> the TMA engine's reads
    epi_bar();
    if (etid == 0) {
        tma_store_3d(tmOut, stage, t.a_tile * BLOCK_A, t.b_tile * BN, t.z);
        bulk_commit();
    }
}

// SiLU tile of the gate/up projection: lanes 0..63 of the accumulator = gate rows, 64..127 = the matching up rows.  ALL four
// warps compute: per 32-column chunk the gate thread of a feature hands its columns 16..31 to the up thread and receives the up
// values of columns 0..15 (exch: two [16][64] fp32 halves per chunk, double-buffered), so each thread evaluates 16 SiLUs per
// chunk instead of the gate threads 32.  act_stage[b][n64] bf16  ->  act[b][a_tile * 64 + n64]
template <int BN>
__device__ __forceinline__ void epilogue_silu_tma(uint32_t taddr0, const WorkItem& t, int quarter, int lane, int etid,
                                                  const CUtensorMap* tmAct, float* exch, __nv_bfloat16* act_stage) {
    const bool is_up = quarter >= 2;
    const int r64 = (quarter & 1) * 32 + lane;
    if (etid == 0) bulk_wait_read0();
    epi_bar();
#pragma unroll 1
    for (int c = 0; c < BN; c += 32) {
        float* buf = exch + ((c >> 5) & 1) * (32 * 64);     // [0, 16) rows: up values of cols 0..15; [16, 32): gate values of cols 16..31
        uint32_t v[32];
        tmem_ld_32x32b_x32(taddr0 + c, v);
        tmem_ld_wait();
        if (is_up) {
#pragma unroll
            for (int j = 0; j < 16; ++j) buf[j * 64 + r64] = __uint_as_float(v[j]);
        } else {
#pragma unroll
            for (int j = 16; j < 32; ++j) buf[j * 64 + r64] = __uint_as_float(v[j]);
        }
        asm volatile("bar.sync 2, 128;" ::: "memory");
        float o[16];
        if (is_up) {
#pragma unroll
            for (int j = 0; j < 16; ++j) o[j] = buf[(16 + j) * 64 + r64];          // gate values, cols 16..31
#pragma unroll
            for (int j = 0; j < 16; ++j)
                act_stage[(c + 16 + j) * 64 + r64] = __float2bfloat16(silu_mul(o[j], __uint_as_float(v[16 + j])));
        } else {
#pragma unroll
            for (int j = 0; j < 16; ++j) o[j] = buf[j * 64 + r64];                 // up values, cols 0..15
#pragma unroll
            for (int j = 0; j < 16; ++j)
                act_stage[(c + j) * 64 + r64] = __float2bfloat16(silu_mul(__uint_as_float(v[j]), o[j]));
        }
    }
    fence_proxy_async();
    epi_bar();
    if (etid == 0) {
        tma_store_2d(tmAct, act_stage, t.a_tile * 64, t.b_tile * BN);
        bulk_commit();
    }
}

template <int BN, int MODE, int CAP = 8>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_bf16_tcgen05(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                  void* __restrict__ out, int rowsA, int rowsB, int K, int splits, int ldo,
                  int ld_rows, const RopeEpi rope, const __grid_constant__ CUtensorMap tmOut, int tma_epi) {
    using Cfg = GemmCfg<BN, CAP>;
    constexpr int kStages = Cfg::kStages;

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = align_smem_1024(smem_raw);
    uint8_t* smemA = smem;
    uint8_t* smemB = smem + kStages * Cfg::kStageBytesA;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + kStages * Cfg::kStageBytes);
    uint64_t* empty_bar = full_bar + kStages;
    uint64_t* tmem_full = empty_bar + kStages;
    uint64_t* tmem_empty = tmem_full + 2;
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty + 2);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    griddep_launch();   // PDL: the next kernel may start its prologue now
    const int tr_slot = trace_begin(decode_orient<MODE>() ? TR_GEMM_DEC : TR_GEMM_PF);

    if (warp == 0 && elect_one()) {
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmB);
    }
    if (warp == 1) {
        if (elect_one()) {
            for (int s = 0; s < kStages; ++s) {
                mbar_init(&full_bar[s], 1);
                mbar_init(&empty_bar[s], 1);
            }
            for (int s = 0; s < 2; ++s) {
                mbar_init(&tmem_full[s], 1);
                mbar_init(&tmem_empty[s], 4);
            }
            fence_barrier_init();
        }
        __syncwarp();
        tmem_alloc<Cfg::kTmemCols>(tmem_ptr);
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_ptr;

    WorkSched sched;
    sched.init(rowsA, rowsB, K, splits, BN);
    WorkItem t;
    // detail trace of a plain decode projection: selected by its split-K factor (rr_debug_trace_detail(10 + splits)), CTAs 0 / 37 / 74 / 111
    const int tsm = (decode_orient<MODE>() && rr_trace_detail == 10 + splits && blockIdx.x % 37 == 0) ? 8 + (int)(blockIdx.x / 37) : -1;

    if (warp == 0) {
        // ===================== TMA producer =====================
        if (elect_one()) {
            // Streamed-once operand (decode weights) should not displace the KV cache in L2;
            // the small re-read operand is kept.
            const uint64_t polA = decode_orient<MODE>() ? l2_policy_evict_first()
                                                               : l2_policy_evict_last();
            const uint64_t polB = l2_policy_evict_last();
            int stage = 0;
            uint32_t phase = 0;
            bool have = sched.next(t);
            if (tsm >= 0) trace_mark_at(TR_GEMM_MARK + 0, tsm, 0);
            // PDL prefetch of the constant (weight) operand for the first `pre` k-blocks.
            // (An additional L2 prefetch of the panel behind the ring was measured in round 1: whole panel 5.12 -> 5.37 ms
            //  per decode step, bounded to 8 / 16 k-blocks no gain / slower; removed.)
            int pre = 0;
            if (have) {
                pre = min(kStages, t.kb1 - t.kb0);
                for (int i = 0; i < pre; ++i) {
                    mbar_arrive_expect_tx(&full_bar[i], Cfg::kStageBytes);
                    if (decode_orient<MODE>())
                        tma_load_2d_hint(smemA + i * Cfg::kStageBytesA, &tmA, &full_bar[i], (t.kb0 + i) * BLOCK_K,
                                         t.a_tile * BLOCK_A, polA);
                    else
                        tma_load_2d_hint(smemB + i * Cfg::kStageBytesB, &tmB, &full_bar[i], (t.kb0 + i) * BLOCK_K,
                                         t.b_tile * BN, polB);
                }
            }
            griddep_wait();
            trace_dep(tr_slot);
            if (tsm >= 0) trace_mark_at(TR_GEMM_MARK + 1, tsm, 1);
            if (have) {
                for (int i = 0; i < pre; ++i) {
                    if (decode_orient<MODE>())
                        tma_load_2d_hint(smemB + i * Cfg::kStageBytesB, &tmB, &full_bar[i], (t.kb0 + i) * BLOCK_K,
                                         t.b_tile * BN, polB);
                    else
                        tma_load_2d_hint(smemA + i * Cfg::kStageBytesA, &tmA, &full_bar[i], (t.kb0 + i) * BLOCK_K,
                                         t.a_tile * BLOCK_A, polA);
                }
                t.kb0 += pre;                          // already in flight
                stage = pre % kStages;
                phase = (pre == kStages) ? 1u : 0u;
            }
            while (have) {
                for (int kb = t.kb0; kb < t.kb1; ++kb) {
                    mbar_wait(&empty_bar[stage], phase ^ 1);
                    mbar_arrive_expect_tx(&full_bar[stage], Cfg::kStageBytes);
                    tma_load_2d_hint(smemA + stage * Cfg::kStageBytesA, &tmA, &full_bar[stage],
                                     kb * BLOCK_K, t.a_tile * BLOCK_A, polA);
                    tma_load_2d_hint(smemB + stage * Cfg::kStageBytesB, &tmB, &full_bar[stage],
                                     kb * BLOCK_K, t.b_tile * BN, polB);
                    if (++stage == kStages) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
                have = sched.next(t);
            }
            if (tsm >= 0) trace_mark_at(TR_GEMM_MARK + 2, tsm, 2);
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        if (elect_one()) {
            constexpr uint32_t idesc = umma_idesc_bf16_f32(BLOCK_A, BN);
            int stage = 0;
            uint32_t phase = 0;
            for (int it = 0; sched.next(t); ++it) {
                const int acc = it & 1;
                const uint32_t acc_phase = (it >> 1) & 1;
                mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
                tcgen05_fence_after();
                const uint32_t tmem_d = tmem_base + acc * BN;
                for (int kb = t.kb0; kb < t.kb1; ++kb) {
                    mbar_wait(&full_bar[stage], phase);
                    if (tsm >= 0 && kb == t.kb0) trace_mark_at(TR_GEMM_MARK + 3, tsm, 8 + it);
                    tcgen05_fence_after();
                    const uint64_t adesc =
                        umma_desc_sw128_kmajor(smem_u32(smemA + stage * Cfg::kStageBytesA));
                    const uint64_t bdesc =
                        umma_desc_sw128_kmajor(smem_u32(smemB + stage * Cfg::kStageBytesB));
#pragma unroll
                    for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
                        // advance 16 bf16 = 32 B inside the swizzle row: +2 in 16-byte units
                        umma_bf16_ss(tmem_d, adesc + 2 * k, bdesc + 2 * k, idesc,
                                     (kb > t.kb0 || k > 0) ? 1u : 0u);
                    }
                    umma_commit(&empty_bar[stage]);   // smem slot free once these MMAs retire
                    if (++stage == kStages) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
                umma_commit(&tmem_full[acc]);         // accumulator ready for the epilogue
            }
        }
    } else {
        // ===================== epilogue (warps 2..5) =====================
        const int quarter = warp & 3;                 // TMEM lane quarter this warp may access
        const int row_in_tile = quarter * 32 + lane;
        const int etid = (warp - 2) * 32 + lane;
        float* epi_stage = reinterpret_cast<float*>(smem + kStages * Cfg::kStageBytes + 256);
        if (MODE == OUT_TRANSPOSED_F32 && BN <= 64 && tma_epi && etid == 0) tma_prefetch_desc(&tmOut);
        griddep_wait();                               // `out` may still be read by the preceding kernel
        for (int it = 0; sched.next(t); ++it) {
            const int acc = it & 1;
            const uint32_t acc_phase = (it >> 1) & 1;
            mbar_wait(&tmem_full[acc], acc_phase);
            if (tsm >= 0 && etid == 0) trace_mark_at(TR_GEMM_MARK + 4, tsm, 16 + 2 * it);
            tcgen05_fence_after();
            const int a_row = t.a_tile * BLOCK_A + row_in_tile;
            const uint32_t taddr0 = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + acc * BN;
            bool done = false;
            if constexpr (MODE == OUT_TRANSPOSED_F32 && BN <= 64) {
                if (tma_epi) { epilogue_planes_tma<BN>(taddr0, t, quarter, lane, etid, &tmOut, epi_stage); done = true; }
            }
            if (!done)
                epilogue_item<BN, MODE>(taddr0, a_row, t, quarter, lane, out, rowsA, rowsB, ldo, ld_rows, rope, epi_stage);
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tmem_empty[acc]);
            if (tsm >= 0 && etid == 0) trace_mark_at(TR_GEMM_MARK + 5, tsm, 17 + 2 * it);
        }
        if constexpr (MODE == OUT_TRANSPOSED_F32 && BN <= 64) {
            if (tma_epi && etid == 0) bulk_wait_read0();   // the staging tile must outlive the reads of its stores; grid completion covers the writes
        }
    }

    tcgen05_fence_before();
    __syncthreads();
    if (tsm >= 0 && threadIdx.x == 0) trace_mark_at(TR_GEMM_MARK + 6, tsm, 3);
    trace_end(tr_slot);
    if (warp == 1) {
        tcgen05_fence_after();
        tmem_dealloc<Cfg::kTmemCols>(tmem_base);
    }
}

// =================================================================================================
// Fused decode MLP: act = SiLU(x Wg^T) * (x Wu^T), planes = act Wd^T in ONE persistent launch (decode orientation,
// weights on the UMMA M side).  Same warp roles, smem ring and TMEM double buffer as gemm_bf16_tcgen05; the pipeline
// state simply carries from item to item.  Each CTA runs its gate/up tiles from a host-built list, then its down items:
// drawn from a device counter (a.dyn, default) or from the same list (static schedule, RR_MLP_STATIC).
// A down item = (128 output features, one K-slice of `slice_kb` k-blocks); k-block kb of the down GEMM is
// exactly the 64 act columns gate/up tile kb writes, so the item only depends on the tiles of its slice: the gate/up
// epilogue (TMA store of the act tile, completion wait, fence) bumps ready[slice] and the producer of a down item requests
// the WEIGHT tiles of its first stages, then acquires ready[slice] == slice length, then requests the activation tiles.
// No kernel boundary,
// no wave-quantisation tail of the gate/up grid (224 tiles on 148 SMs): CTAs that own one gate/up tile start on the
// early slices while the others finish their second tile.
__device__ __forceinline__ unsigned ld_acquire_gpu_u32(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

template <int BN>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_mlp_tcgen05(const __grid_constant__ MlpArgs a) {
    using Cfg = GemmCfg<BN>;
    constexpr int kStages = Cfg::kStages;

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = align_smem_1024(smem_raw);
    uint8_t* smemA = smem;
    uint8_t* smemB = smem + kStages * Cfg::kStageBytesA;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + kStages * Cfg::kStageBytes);
    uint64_t* empty_bar = full_bar + kStages;
    uint64_t* tmem_full = empty_bar + kStages;
    uint64_t* tmem_empty = tmem_full + 2;
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty + 2);
    volatile int* dyn_q = reinterpret_cast<volatile int*>(smem + kStages * Cfg::kStageBytes + 176);   // [16] dynamic down items of this CTA
    float* silu_stage = reinterpret_cast<float*>(smem + kStages * Cfg::kStageBytes + 256);    // exchange; aliased by the planes tile
    __nv_bfloat16* act_stage = reinterpret_cast<__nv_bfloat16*>(smem + kStages * Cfg::kStageBytes + 256 + Cfg::kSiluStageBytes);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    griddep_launch();
    const int tr_slot = trace_begin(TR_GEMM_DEC);

    if (warp == 0 && elect_one()) {
        tma_prefetch_desc(&a.tmA0); tma_prefetch_desc(&a.tmB0);
        tma_prefetch_desc(&a.tmA1); tma_prefetch_desc(&a.tmB1);
        if (a.tma_epi) { tma_prefetch_desc(&a.tmAct); tma_prefetch_desc(&a.tmPlanes); }
    }
    if (warp == 1) {
        if (elect_one()) {
            for (int s = 0; s < kStages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
            for (int s = 0; s < 2; ++s) { mbar_init(&tmem_full[s], 1); mbar_init(&tmem_empty[s], 4); }
            for (int s = 0; s < 16; ++s) dyn_q[s] = -2;
            fence_barrier_init();
        }
        __syncwarp();
        tmem_alloc<Cfg::kTmemCols>(tmem_ptr);
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_ptr;

    const int4* my = reinterpret_cast<const int4*>(a.items) + (size_t)blockIdx.x * a.max_items;   // constant data
    auto get = [&](int i, WorkItem& t, int& ph) -> bool {
        if (i >= a.max_items) return false;
        const int4 v = __ldg(my + i);
        if (v.x < 0) return false;
        ph = v.x >> 16; t.a_tile = v.x & 0xffff; t.b_tile = 0; t.kb0 = v.y; t.kb1 = v.z; t.z = v.w;
        return true;
    };
    // Down items are not in the static lists when a.dyn: after its gate/up tiles a CTA takes the next item q of the slice-major
    // order (z = q / tiles1) from a global counter, so the split follows the real finishing order instead of a host-side time
    // model (the static list schedule left a 10 us tail: CTAs with three down items next to CTAs with one).  The producer thread
    // draws q -- when the last load of the current item is out, so the round trip of the atomic overlaps the drain of the ring and
    // no CTA sits on an item it cannot start -- and publishes it to the MMA / epilogue warps through dyn_q[] (-2 = not drawn yet,
    // -1 = no more work).  Which CTA computes an item does not change a single bit of its plane tile.
    auto dyn_decode = [&](int q, WorkItem& t, int& ph) {
        const int z = q / a.tiles1;
        t.a_tile = q - z * a.tiles1; t.b_tile = 0; t.kb0 = z * a.slice_kb;
        t.kb1 = min(t.kb0 + a.slice_kb, a.kb1n); t.z = z; ph = 1;
    };
    auto next_consumer = [&](int it, int& nstat, WorkItem& t, int& ph) -> bool {
        if (nstat < 0) {
            if (get(it, t, ph)) return true;
            nstat = it;
        }
        if (!a.dyn) return false;
        const int d = it - nstat;
        if (d >= 16) return false;
        int q;
        do { q = dyn_q[d]; } while (q == -2);
        if (q < 0) return false;
        dyn_decode(q, t, ph);
        return true;
    };
    WorkItem t;
    int ph = 0;

    if (warp == 0) {
        // ===================== TMA producer =====================
        if (elect_one()) {
            const uint64_t polA = l2_policy_evict_first(), polB = l2_policy_evict_last();
            int stage = 0;
            uint32_t phase = 0;
            bool first = true;
            int tm_i = 0;
            trace_mark_fixed(TR_MLP_MARK + 0, tm_i++);
            int nstat = -1;
            unsigned q_next = 0;
            bool have_next = false;
            for (int i = 0;; ++i) {
                if (nstat < 0 && !get(i, t, ph)) nstat = i;
                if (nstat >= 0) {
                    if (!a.dyn) break;
                    const int d = i - nstat;
                    if (d >= 16) break;
                    if (first) { griddep_wait(); trace_dep(tr_slot); first = false; }    // the counter is zeroed by the preceding kernel
                    const unsigned q = have_next ? q_next : atomicAdd(a.ready + a.n_slices, 1u);
                    have_next = false;
                    if (q >= (unsigned)a.n_down) { dyn_q[d] = -1; break; }
                    dyn_q[d] = (int)q;
                    dyn_decode((int)q, t, ph);
                }
                const CUtensorMap* tA = ph ? &a.tmA1 : &a.tmA0;
                const CUtensorMap* tB = ph ? &a.tmB1 : &a.tmB0;
                // weight tiles of the first stages go out before the activations are known to exist: at the start
                // of the kernel (PDL: the preceding kernel is still running) and for every down item (its slice of
                // act may still be in flight on other SMs)
                const int pre = (first || ph) ? min(kStages, t.kb1 - t.kb0) : 0;
                const int st0 = stage;
                for (int j = 0; j < pre; ++j) {
                    mbar_wait(&empty_bar[stage], phase ^ 1);
                    mbar_arrive_expect_tx(&full_bar[stage], Cfg::kStageBytes);
                    tma_load_2d_hint(smemA + stage * Cfg::kStageBytesA, tA, &full_bar[stage], (t.kb0 + j) * BLOCK_K,
                                     t.a_tile * BLOCK_A, polA);
                    if (++stage == kStages) { stage = 0; phase ^= 1; }
                }
                if (first) { griddep_wait(); trace_dep(tr_slot); first = false; trace_mark_fixed(TR_MLP_MARK + 1, tm_i++); }
                if (ph) {
                    const unsigned need = (unsigned)(t.kb1 - t.kb0);
                    trace_mark_fixed(TR_MLP_MARK + 2, tm_i++);
                    while (ld_acquire_gpu_u32(a.ready + t.z) < need) {
                    }
                    asm volatile("fence.proxy.async;" ::: "memory");   // other SMs' generic-proxy stores -> our TMA reads
                    trace_mark_fixed(TR_MLP_MARK + 3, tm_i++);
                }
                for (int j = 0, s2 = st0; j < pre; ++j) {
                    tma_load_2d_hint(smemB + s2 * Cfg::kStageBytesB, tB, &full_bar[s2], (t.kb0 + j) * BLOCK_K, 0, polB);
                    if (++s2 == kStages) s2 = 0;
                }
                for (int kb = t.kb0 + pre; kb < t.kb1; ++kb) {
                    mbar_wait(&empty_bar[stage], phase ^ 1);
                    mbar_arrive_expect_tx(&full_bar[stage], Cfg::kStageBytes);
                    tma_load_2d_hint(smemA + stage * Cfg::kStageBytesA, tA, &full_bar[stage], kb * BLOCK_K, t.a_tile * BLOCK_A, polA);
                    tma_load_2d_hint(smemB + stage * Cfg::kStageBytesB, tB, &full_bar[stage], kb * BLOCK_K, 0, polB);
                    if (++stage == kStages) { stage = 0; phase ^= 1; }
                }
                if (a.dyn) {                       // the next item is a dynamic one: draw it now
                    WorkItem tn; int pn;
                    const bool next_static = nstat < 0 && get(i + 1, tn, pn);
                    const int dn = nstat < 0 ? 0 : i + 1 - nstat;
                    if (!next_static && dn < 16) { q_next = atomicAdd(a.ready + a.n_slices, 1u); have_next = true; }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        if (elect_one()) {
            constexpr uint32_t idesc = umma_idesc_bf16_f32(BLOCK_A, BN);
            int stage = 0;
            uint32_t phase = 0;
            int nstat = -1;
            for (int it = 0; next_consumer(it, nstat, t, ph); ++it) {
                const int acc = it & 1;
                mbar_wait(&tmem_empty[acc], ((it >> 1) & 1) ^ 1);
                tcgen05_fence_after();
                const uint32_t tmem_d = tmem_base + acc * BN;
                for (int kb = t.kb0; kb < t.kb1; ++kb) {
                    mbar_wait(&full_bar[stage], phase);
                    if (kb == t.kb0) trace_mark_fixed(TR_MLP_MARK + 4 + ph, 64 + it);
                    tcgen05_fence_after();
                    const uint64_t adesc = umma_desc_sw128_kmajor(smem_u32(smemA + stage * Cfg::kStageBytesA));
                    const uint64_t bdesc = umma_desc_sw128_kmajor(smem_u32(smemB + stage * Cfg::kStageBytesB));
#pragma unroll
                    for (int k = 0; k < BLOCK_K / UMMA_K; ++k)
                        umma_bf16_ss(tmem_d, adesc + 2 * k, bdesc + 2 * k, idesc, (kb > t.kb0 || k > 0) ? 1u : 0u);
                    umma_commit(&empty_bar[stage]);
                    if (++stage == kStages) { stage = 0; phase ^= 1; }
                }
                umma_commit(&tmem_full[acc]);
            }
        }
    } else {
        // ===================== epilogue (warps 2..5) =====================
        const int quarter = warp & 3;
        const int row_in_tile = quarter * 32 + lane;
        const int etid = (warp - 2) * 32 + lane;
        RopeEpi no_rope;
        no_rope.q_out = nullptr; no_rope.k_cache = nullptr; no_rope.v_cache = nullptr; no_rope.slot = nullptr;
        no_rope.pos = nullptr; no_rope.table = nullptr; no_rope.n_heads = 0; no_rope.n_kv_heads = 0; no_rope.ctx_max = 0;
        griddep_wait();
        int nstat = -1;
        for (int it = 0; next_consumer(it, nstat, t, ph); ++it) {
            const int acc = it & 1;
            mbar_wait(&tmem_full[acc], (it >> 1) & 1);
            if (etid == 0) trace_mark_fixed(TR_MLP_MARK + 6 + ph, 128 + 4 * it);
            tcgen05_fence_after();
            const int a_row = t.a_tile * BLOCK_A + row_in_tile;
            const uint32_t taddr0 = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + acc * BN;
            bool tma_done = false;
            if constexpr (BN <= 64) {
                if (a.tma_epi) {
                    if (ph == 0) epilogue_silu_tma<BN>(taddr0, t, quarter, lane, etid, &a.tmAct, silu_stage, act_stage);
                    else epilogue_planes_tma<BN>(taddr0, t, quarter, lane, etid, &a.tmPlanes, silu_stage);
                    tma_done = true;
                }
            }
            if (tma_done) {
            } else if (ph == 0)
                epilogue_item<BN, OUT_TRANSPOSED_SILU>(taddr0, a_row, t, quarter, lane, a.act, 2 * a.inter, a.rows, a.inter, 0,
                                                       no_rope, silu_stage);
            else
                epilogue_item<BN, OUT_TRANSPOSED_F32>(taddr0, a_row, t, quarter, lane, a.out1, a.hidden, a.rows, a.hidden,
                                                      a.ld_rows, no_rope, nullptr);
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tmem_empty[acc]);
            if (etid == 0) trace_mark_fixed(TR_MLP_MARK + 10, 128 + 4 * it + 1);      // stores issued
            if (ph == 0) {
                // publish this tile's 64 act columns: every epilogue thread's stores, then one release-increment
                if (tma_done) {
                    if (etid == 0) {
                        bulk_wait0();                                                  // the bulk store's writes are performed
                        trace_mark_fixed(TR_MLP_MARK + 11, 128 + 4 * it + 2);
                        asm volatile("fence.proxy.async;" ::: "memory");
                        __threadfence();
                        atomicAdd(a.ready + t.a_tile / a.slice_kb, 1u);
                        trace_mark_fixed(TR_MLP_MARK + 8, 128 + 4 * it + 3);
                    }
                } else {
                    asm volatile("bar.sync 3, 128;" ::: "memory");
                    if (etid == 0) {
                        trace_mark_fixed(TR_MLP_MARK + 11, 128 + 4 * it + 2);          // all epilogue threads past their stores
                        __threadfence();
                        atomicAdd(a.ready + t.a_tile / a.slice_kb, 1u);
                        trace_mark_fixed(TR_MLP_MARK + 8, 128 + 4 * it + 3);
                    }
                }
            }
        }
    }

    if (a.tma_epi && threadIdx.x == 64) bulk_wait_read0();  // epilogue thread 0: the staging tile must outlive the reads of its stores
    tcgen05_fence_before();
    __syncthreads();
    trace_end(tr_slot);
    if (warp == 1) {
        tcgen05_fence_after();
        tmem_dealloc<Cfg::kTmemCols>(tmem_base);
    }
}

// =================================================================================================
// 2-CTA variant for the prefill orientation (tokens on M): a CTA pair (cluster of 2, same TPC) computes a
// 256 x 256 tile with tcgen05.mma.cta_group::2 (UMMA M = 256).  Each CTA stages its own 128 rows of A and only HALF of
// the 256 B rows per k-block (the tensor core reads the other half from the peer's shared memory), so the smem fill
// traffic per FLOP halves and the ring holds 6 stages of 32 KB instead of 4 of 48 KB.  The leader CTA (rank 0) issues
// the MMAs; both CTAs run a TMA producer (2SM TMA form: transaction bytes land on the leader's full barrier) and 4
// epilogue warps for their own 128 accumulator rows.  tcgen05.commit multicasts "slot free" / "accumulator ready" to
// both CTAs; the epilogue warps of both CTAs release the accumulator on the leader's barrier.
constexpr int K2_BN = 256;
constexpr int K2_STAGE_A = BLOCK_A * BLOCK_K * 2;          // 16 KB: this CTA's 128 rows of A
constexpr int K2_STAGE_B = 128 * BLOCK_K * 2;              // 16 KB: this CTA's half of the 256 B rows
constexpr int K2_STAGE = K2_STAGE_A + K2_STAGE_B;
constexpr int K2_STAGES = 6;
constexpr int K2_EPI_STAGE = 4 * 32 * 36 * 4;             // residual epilogue: per-warp 32 x 36 fp32 transpose tiles
constexpr int K2_SMEM = K2_STAGES * K2_STAGE + 1024 + 256 + K2_EPI_STAGE;
constexpr int GROUP_PAIRS = 8;

__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t cta) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(cta));
    return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tma_load_2d_2sm(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int32_t c0, int32_t c1,
                                                uint64_t policy) {
    // executed by both CTAs; peer bit cleared so the transaction bytes update the leader CTA's barrier
    const uint32_t mbar = smem_u32(bar) & 0xFEFFFFFFu;
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
        " [%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(mbar), "r"(c0), "r"(c1), "l"(policy)
        : "memory");
}
__device__ __forceinline__ void umma_bf16_ss_2sm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                                 uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}\n"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit_2sm(uint64_t* bar) {      // arrives on `bar` in BOTH CTAs of the pair
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"((uint16_t)3)
                 : "memory");
}

template <int MODE>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(GEMM_THREADS, 1)
gemm_bf16_tcgen05_2cta(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                       void* __restrict__ out, int rowsA, int rowsB, int K, int ldo, const RopeEpi rope) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = align_smem_1024(smem_raw);
    uint8_t* smemA = smem;
    uint8_t* smemB = smem + K2_STAGES * K2_STAGE_A;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + K2_STAGES * K2_STAGE);
    uint64_t* empty_bar = full_bar + K2_STAGES;
    uint64_t* tmem_full = empty_bar + K2_STAGES;
    uint64_t* tmem_empty = tmem_full + 2;
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const bool leader = rank == 0;
    griddep_launch();
    const int tr_slot = trace_begin(TR_GEMM_PF);

    if (warp == 0 && elect_one()) {
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmB);
    }
    if (warp == 1) {
        if (elect_one()) {
            for (int s = 0; s < K2_STAGES; ++s) {
                mbar_init(&full_bar[s], 1);        // leader's expect_tx arrive; both CTAs' TMA bytes complete on it
                mbar_init(&empty_bar[s], 1);       // multicast commit
            }
            for (int s = 0; s < 2; ++s) {
                mbar_init(&tmem_full[s], 1);       // multicast commit
                mbar_init(&tmem_empty[s], 8);      // 4 epilogue warps of each CTA (leader's instance is the one waited on)
            }
            fence_barrier_init();
        }
        __syncwarp();
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr)), "n"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tcgen05_fence_before();
    __syncthreads();
    cluster_sync_all();                            // peer barriers initialised before any remote arrive / multicast
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_ptr;

    const int pairsA = (rowsA + 255) / 256;
    const int tilesB = (rowsB + K2_BN - 1) / K2_BN;
    const int kblocks = (K + BLOCK_K - 1) / BLOCK_K;
    const int n_work = pairsA * tilesB;
    const int n_clusters = gridDim.x >> 1, cluster_id = blockIdx.x >> 1;
    auto decode = [&](int w, int& pa, int& tb) {
        const int per_group = GROUP_PAIRS * tilesB;
        const int g = w / per_group, r = w - g * per_group;
        const int a0 = g * GROUP_PAIRS, ga = min(GROUP_PAIRS, pairsA - a0);
        pa = a0 + r % ga;
        tb = r / ga;
    };

    if (warp == 0) {
        // ===================== TMA producer (both CTAs) =====================
        if (elect_one()) {
            const uint64_t polA = l2_policy_evict_last(), polB = l2_policy_evict_last();
            griddep_wait();
            trace_dep(tr_slot);
            int stage = 0;
            uint32_t phase = 0;
            for (int w = cluster_id; w < n_work; w += n_clusters) {
                int pa, tb;
                decode(w, pa, tb);
                for (int kb = 0; kb < kblocks; ++kb) {
                    mbar_wait(&empty_bar[stage], phase ^ 1);
                    // The peer needs no arrive of its own: its loads for the next phase are only issued after its
                    // empty barrier fired, i.e. after the leader consumed the previous phase.
                    if (leader) mbar_arrive_expect_tx(&full_bar[stage], 2 * K2_STAGE);
                    tma_load_2d_2sm(smemA + stage * K2_STAGE_A, &tmA, &full_bar[stage], kb * BLOCK_K,
                                    pa * 256 + (int)rank * 128, polA);
                    tma_load_2d_2sm(smemB + stage * K2_STAGE_B, &tmB, &full_bar[stage], kb * BLOCK_K,
                                    tb * K2_BN + (int)rank * 128, polB);
                    if (++stage == K2_STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer (leader CTA only) =====================
        if (leader && elect_one()) {
            constexpr uint32_t idesc = umma_idesc_bf16_f32(256, K2_BN);
            int stage = 0, it = 0;
            uint32_t phase = 0;
            for (int w = cluster_id; w < n_work; w += n_clusters, ++it) {
                const int acc = it & 1;
                mbar_wait(&tmem_empty[acc], ((it >> 1) & 1) ^ 1);
                tcgen05_fence_after();
                const uint32_t tmem_d = tmem_base + acc * K2_BN;
                for (int kb = 0; kb < kblocks; ++kb) {
                    mbar_wait(&full_bar[stage], phase);
                    tcgen05_fence_after();
                    const uint64_t adesc = umma_desc_sw128_kmajor(smem_u32(smemA + stage * K2_STAGE_A));
                    const uint64_t bdesc = umma_desc_sw128_kmajor(smem_u32(smemB + stage * K2_STAGE_B));
#pragma unroll
                    for (int k = 0; k < BLOCK_K / UMMA_K; ++k)
                        umma_bf16_ss_2sm(tmem_d, adesc + 2 * k, bdesc + 2 * k, idesc, (kb > 0 || k > 0) ? 1u : 0u);
                    umma_commit_2sm(&empty_bar[stage]);
                    if (++stage == K2_STAGES) { stage = 0; phase ^= 1; }
                }
                umma_commit_2sm(&tmem_full[acc]);
            }
        }
    } else {
        // ===================== epilogue (both CTAs: own 128 rows x 256 columns) =====================
        const int quarter = warp & 3;
        const int row_in_tile = quarter * 32 + lane;
        const uint32_t empty0_remote = mapa_u32(smem_u32(&tmem_empty[0]), 0);
        griddep_wait();
        int it = 0;
        for (int w = cluster_id; w < n_work; w += n_clusters, ++it) {
            int pa, tb;
            decode(w, pa, tb);
            const int acc = it & 1;
            mbar_wait(&tmem_full[acc], (it >> 1) & 1);
            tcgen05_fence_after();
            WorkItem t;
            t.a_tile = pa * 2 + (int)rank; t.b_tile = tb; t.z = 0; t.kb0 = 0; t.kb1 = kblocks;
            const int a_row = t.a_tile * BLOCK_A + row_in_tile;
            const uint32_t taddr0 = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + acc * K2_BN;
            epilogue_item<K2_BN, MODE>(taddr0, a_row, t, quarter, lane, out, rowsA, rowsB, ldo, 0, rope,
                                       reinterpret_cast<float*>(smem + K2_STAGES * K2_STAGE + 256));
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(empty0_remote + acc * 8);
        }
    }

    tcgen05_fence_before();
    __syncthreads();
    cluster_sync_all();                            // the peer's tensor core may still read this CTA's shared memory
    trace_end(tr_slot);
    if (warp == 1) {
        tcgen05_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(512) : "memory");
    }
}

// ---------------------------------------------------------------- host side
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                    const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                    const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode_fn() {
    static PFN_encodeTiled fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres);
        if (e == cudaSuccess && qres == cudaDriverEntryPointSuccess) fn = (PFN_encodeTiled)p;
    });
    return fn;
}

// [rows, K] bf16 row-major (K contiguous, row pitch ld elements) -> TMA map with box {64, box_rows}.
int make_tmap_bf16_2d(CUtensorMap* map, const void* base, int rows, int K, int ld, int box_rows) {
    PFN_encodeTiled enc = get_encode_fn();
    if (!enc) return RR_ERR_CUDA;
    cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
    cuuint32_t box[2] = {(cuuint32_t)BLOCK_K, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides,
                     box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? RR_OK : RR_ERR_CUDA;
}

// planes P[z][b][n] fp32 (n contiguous, row pitch ldo, plane pitch ld_rows * ldo), valid n < n_valid, b < rows_valid:
// 3-D map {n, b, z}, box {128, box_rows, 1}, no swizzle -- the destination of epilogue_planes_tma
int make_tmap_planes_f32(CUtensorMap* map, const void* base, int n_valid, int ldo, int rows_valid, int ld_rows, int splits, int box_rows) {
    PFN_encodeTiled enc = get_encode_fn();
    if (!enc) return RR_ERR_CUDA;
    cuuint64_t dims[3] = {(cuuint64_t)n_valid, (cuuint64_t)rows_valid, (cuuint64_t)splits};
    cuuint64_t strides[2] = {(cuuint64_t)ldo * 4, (cuuint64_t)ld_rows * ldo * 4};
    cuuint32_t box[3] = {128, (cuuint32_t)box_rows, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? RR_OK : RR_ERR_CUDA;
}
// act[b][n] bf16 (row pitch ld): 2-D map {n, b}, box {64, box_rows}, no swizzle -- the destination of epilogue_silu_tma
int make_tmap_act_store(CUtensorMap* map, const void* base, int rows, int n, int ld, int box_rows) {
    PFN_encodeTiled enc = get_encode_fn();
    if (!enc) return RR_ERR_CUDA;
    cuuint64_t dims[2] = {(cuuint64_t)n, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
    cuuint32_t box[2] = {64, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? RR_OK : RR_ERR_CUDA;
}

static std::atomic<int> g_num_sms[64];
int num_sms() {                         // of the current device (one process may drive several)
    int dev = 0;
    cudaGetDevice(&dev);
    int n = g_num_sms[dev & 63].load(std::memory_order_relaxed);
    if (!n) {
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        g_num_sms[dev & 63].store(n, std::memory_order_relaxed);
    }
    return n;
}

template <int BN, int MODE>
static int launch_one(const GemmPlan& p, cudaStream_t st) {
    constexpr int CAP = 8;
    auto kern = gemm_bf16_tcgen05<BN, MODE, CAP>;
    static std::atomic<uint64_t> attr_set{0};
    if (ensure_dyn_smem(kern, (int)gemm_smem_bytes<BN, MODE, CAP>(), attr_set) != cudaSuccess) return RR_ERR_CUDA;
    const int tilesA = (p.rowsA + BLOCK_A - 1) / BLOCK_A;
    const int tilesB = (p.rowsB + BN - 1) / BN;
    const int n_work = tilesA * tilesB * p.splits;
    const int grid = n_work < num_sms() ? n_work : num_sms();
    cudaError_t le = launch_pdl(kern, dim3(grid), dim3(GEMM_THREADS), (size_t)gemm_smem_bytes<BN, MODE, CAP>(), st, p.tmA, p.tmB,
                                p.out, p.rowsA, p.rowsB, p.K, p.splits, p.ldo, p.ld_rows, p.rope, p.tmOut, p.tma_epi);
    return (le == cudaSuccess && cudaGetLastError() == cudaSuccess) ? RR_OK : RR_ERR_CUDA;
}

static bool decode_orient_rt(int mode) { return mode == OUT_TRANSPOSED_F32 || mode == OUT_TRANSPOSED_SILU; }

// splits >= 1: uniform split-K with `splits` planes.
int gemm_plan_init(GemmPlan* p, const void* A, int rowsA, int ldA, const void* B, int rowsB, int ldB,
                   int K, void* out, int ldo, int ld_rows, int splits, int mode, int bn) {
    if (K % 8 != 0 || ldA % 8 != 0 || ldB % 8 != 0) return RR_ERR_ARG;
    if (!(bn == 16 || bn == 32 || bn == 64 || bn == 128 || bn == 256)) return RR_ERR_ARG;
    const int kblocks = (K + BLOCK_K - 1) / BLOCK_K;
    if (splits < 1) return RR_ERR_ARG;
    if (splits > kblocks) splits = kblocks;
    if (mode == OUT_ROWMAJOR_BF16 && (splits != 1 || ldo % 8 != 0)) return RR_ERR_ARG;
    // fused SiLU*mul epilogues: weights row-interleaved in 64-row gate/up blocks, one plane, bf16 act output
    if (mode == OUT_TRANSPOSED_SILU && (splits != 1 || bn < 32 || rowsA % 128 != 0)) return RR_ERR_ARG;
    if (mode == OUT_ROWMAJOR_SILU && (splits != 1 || bn != 256 || rowsB % 128 != 0 || ldo % 8 != 0)) return RR_ERR_ARG;
    if (mode == OUT_ROWMAJOR_ROPE && (splits != 1 || bn != 256 || rowsB % 128 != 0)) return RR_ERR_ARG;
    if (mode == OUT_ROWMAJOR_RESID && (splits != 1 || bn < 32 || ldo % 4 != 0)) return RR_ERR_ARG;
    if (mode < 0 || mode > OUT_ROWMAJOR_RESID) return RR_ERR_ARG;
    memset(&p->rope, 0, sizeof(p->rope));
    p->rowsA = rowsA; p->rowsB = rowsB; p->K = K; p->out = out; p->ldo = ldo; p->ld_rows = ld_rows;
    p->splits = splits; p->mode = mode; p->bn = bn; p->max_ctas = 0;
    int rc = make_tmap_bf16_2d(&p->tmA, A, rowsA, K, ldA, BLOCK_A);
    if (rc != RR_OK) return rc;
    // prefill orientation with 256-wide tiles and at least one full 256-row pair: 2-CTA kernel (B box = 128 rows)
    // decode planes through one TMA store per item: needs 16-byte pitches and at most 64 batch columns per tile
    p->tma_epi = 0;
    if (mode == OUT_TRANSPOSED_F32 && bn <= 64 && ldo % 4 == 0 && ((uintptr_t)out & 15) == 0 && !getenv("RR_NO_TMA_EPI")) {
        rc = make_tmap_planes_f32(&p->tmOut, out, rowsA, ldo, rowsB, ld_rows > 0 ? ld_rows : rowsB, splits, bn);
        if (rc != RR_OK) return rc;
        p->tma_epi = 1;
    }
    p->two_cta = (bn == 256 && !decode_orient_rt(mode) && rowsA >= 256) ? 1 : 0;
    if (p->two_cta) {
        rc = make_tmap_bf16_2d(&p->tmB2, B, rowsB, K, ldB, 128);
        if (rc != RR_OK) return rc;
    }
    return make_tmap_bf16_2d(&p->tmB, B, rowsB, K, ldB, bn);
}

template <int MODE>
static int launch_2cta(const GemmPlan& p, cudaStream_t st) {
    auto kern = gemm_bf16_tcgen05_2cta<MODE>;
    static std::atomic<uint64_t> attr_set{0};
    if (ensure_dyn_smem(kern, (int)K2_SMEM, attr_set) != cudaSuccess) return RR_ERR_CUDA;
    const int pairs = (p.rowsA + 255) / 256, tilesB = (p.rowsB + K2_BN - 1) / K2_BN;
    int clusters = pairs * tilesB;
    if (clusters > num_sms() / 2) clusters = num_sms() / 2;
    cudaError_t le = launch_pdl(kern, dim3(2 * clusters), dim3(GEMM_THREADS), (size_t)K2_SMEM, st, p.tmA, p.tmB2, p.out,
                                p.rowsA, p.rowsB, p.K, p.ldo, p.rope);
    return (le == cudaSuccess && cudaGetLastError() == cudaSuccess) ? RR_OK : RR_ERR_CUDA;
}

int g_use_2cta = getenv("RR_NO_2CTA") ? 0 : 1;

int gemm_launch(const GemmPlan& p, cudaStream_t st) {
    if (p.two_cta && g_use_2cta) {
        switch (p.mode) {
            case OUT_ROWMAJOR_BF16: return launch_2cta<OUT_ROWMAJOR_BF16>(p, st);
            case OUT_ROWMAJOR_SILU: return launch_2cta<OUT_ROWMAJOR_SILU>(p, st);
            case OUT_ROWMAJOR_ROPE: return launch_2cta<OUT_ROWMAJOR_ROPE>(p, st);
            case OUT_ROWMAJOR_RESID: return launch_2cta<OUT_ROWMAJOR_RESID>(p, st);
        }
    }
#define RR_CASE(BN_)                                                                                  \
    case BN_:                                                                                         \
        if (p.mode == OUT_ROWMAJOR_BF16) return launch_one<BN_, OUT_ROWMAJOR_BF16>(p, st);             \
        if (p.mode == OUT_TRANSPOSED_F32) return launch_one<BN_, OUT_TRANSPOSED_F32>(p, st);           \
        if constexpr (BN_ >= 32) {                                                                    \
            if (p.mode == OUT_TRANSPOSED_SILU) return launch_one<BN_, OUT_TRANSPOSED_SILU>(p, st);     \
        }                                                                                             \
        if constexpr (BN_ >= 128) {                                                                   \
            if (p.mode == OUT_ROWMAJOR_RESID) return launch_one<BN_, OUT_ROWMAJOR_RESID>(p, st);       \
        }                                                                                             \
        if constexpr (BN_ == 256) {                                                                   \
            if (p.mode == OUT_ROWMAJOR_SILU) return launch_one<BN_, OUT_ROWMAJOR_SILU>(p, st);         \
            if (p.mode == OUT_ROWMAJOR_ROPE) return launch_one<BN_, OUT_ROWMAJOR_ROPE>(p, st);         \
        }                                                                                             \
        return RR_ERR_ARG;
    switch (p.bn) {
        RR_CASE(16)
        RR_CASE(32)
        RR_CASE(64)
        RR_CASE(128)
        RR_CASE(256)
    }
#undef RR_CASE
    return RR_ERR_ARG;
}


// ---- fused decode MLP: host side ------------------------------------------------------------------
// List schedule on a time line in units of k-blocks (one 16 KB weight tile at a CTA's fair share of the HBM rate, 0.37 us;
// + a fixed per-item cost for pipeline refill / epilogue).  Gate/up tile t goes to CTA t % grid (wave order: tile t is
// finished before tile t + grid).  A slice becomes READY kPublish units after its last gate/up tile finished its mainloop --
// the measured epilogue -> TMA store -> fence -> counter -> acquire chain (tools/trace_mlp.py: ~10 us).  The down items, slice by
// slice, go to the CTA that can START them first, max(CTA free, slice ready); among CTAs that would all wait, the one that
// has been free for the shortest time (best fit).  With the earlier "least loaded CTA" rule every early slice went to the CTAs
// that own one gate/up tile, and the CTAs that own two found only late slices when they finished: they all stalled for one
// publish latency (RR_MLP_SCHED_P=0 restores that rule).
int mlp_schedule(int grid, int inter, int hidden, int slice_kb, std::vector<MlpItem>* items, int dynamic) {
    const int tiles0 = (2 * inter) / BLOCK_A, kb0n = (hidden + BLOCK_K - 1) / BLOCK_K;
    const int tiles1 = (hidden + BLOCK_A - 1) / BLOCK_A, kb1n = inter / BLOCK_K;
    const int n_slices = (kb1n + slice_kb - 1) / slice_kb;
    constexpr int kItemCost = 6;
    const char* pe = getenv("RR_MLP_SCHED_P");
    const long long kPublish = pe ? atoi(pe) : 27;
    std::vector<std::vector<MlpItem>> per(grid);
    std::vector<long long> load(grid, 0);
    std::vector<long long> tile_done(tiles0, 0);
    for (int t = 0; t < tiles0; ++t) {
        MlpItem it; it.tile_phase = t; it.kb0 = 0; it.kb1 = kb0n; it.z = 0;
        per[t % grid].push_back(it);
        load[t % grid] += kb0n + kItemCost;
        tile_done[t] = load[t % grid];
    }
    for (int z = 0; z < (dynamic ? 0 : n_slices); ++z) {          // dynamic: the kernel deals the down items itself
        const int k0 = z * slice_kb, k1 = (k0 + slice_kb < kb1n) ? k0 + slice_kb : kb1n;
        long long ready = 0;
        if (kPublish > 0) {
            for (int t = k0; t < k1 && t < tiles0; ++t) ready = tile_done[t] > ready ? tile_done[t] : ready;
            ready += kPublish;
        }
        for (int tl = 0; tl < tiles1; ++tl) {
            int best = 0;
            for (int c = 1; c < grid; ++c) {
                const long long sc = load[c] > ready ? load[c] : ready, sb = load[best] > ready ? load[best] : ready;
                if (sc < sb || (sc == sb && load[c] > load[best])) best = c;
            }
            MlpItem it; it.tile_phase = tl | (1 << 16); it.kb0 = k0; it.kb1 = k1; it.z = z;
            per[best].push_back(it);
            load[best] = (load[best] > ready ? load[best] : ready) + (k1 - k0) + kItemCost;
        }
    }
    size_t mx = 1;
    for (auto& v : per) mx = v.size() > mx ? v.size() : mx;
    items->assign((size_t)grid * mx, MlpItem{-1, 0, 0, 0});
    for (int c = 0; c < grid; ++c)
        for (size_t i = 0; i < per[c].size(); ++i) (*items)[(size_t)c * mx + i] = per[c][i];
    return (int)mx;
}

int mlp_plan_init(MlpPlan* p, const void* Wgu, const void* Wd, int inter, int hidden, const void* xn, int rows,
                  void* act, void* planes, int ld_rows, int bn, const MlpItem* items_dev, int max_items, int grid,
                  unsigned* ready, int slice_kb, int dynamic) {
    if (!p || !Wgu || !Wd || !xn || !act || !planes || !items_dev || !ready) return RR_ERR_ARG;
    if (inter % 64 || (2 * inter) % BLOCK_A || hidden % 8 || rows > bn || bn < 32 || slice_kb < 1) return RR_ERR_ARG;
    if ((2 * inter) / BLOCK_A > 0xffff || grid < 1 || grid > num_sms()) return RR_ERR_ARG;
    MlpArgs& a = p->args;
    int rc = make_tmap_bf16_2d(&a.tmA0, Wgu, 2 * inter, hidden, hidden, BLOCK_A);
    if (rc == RR_OK) rc = make_tmap_bf16_2d(&a.tmB0, xn, rows, hidden, hidden, bn);
    if (rc == RR_OK) rc = make_tmap_bf16_2d(&a.tmA1, Wd, hidden, inter, inter, BLOCK_A);
    if (rc == RR_OK) rc = make_tmap_bf16_2d(&a.tmB1, act, rows, inter, inter, bn);
    if (rc != RR_OK) return rc;
    a.act = (__nv_bfloat16*)act; a.out1 = (float*)planes; a.inter = inter; a.hidden = hidden; a.rows = rows;
    a.ld_rows = ld_rows; a.items = items_dev; a.max_items = max_items; a.ready = ready; a.slice_kb = slice_kb;
    a.kb1n = inter / BLOCK_K; a.tiles1 = (hidden + BLOCK_A - 1) / BLOCK_A;
    a.n_slices = (a.kb1n + slice_kb - 1) / slice_kb; a.n_down = a.n_slices * a.tiles1; a.dyn = dynamic ? 1 : 0;
    p->grid = grid; p->bn = bn; p->n_slices = (inter / BLOCK_K + slice_kb - 1) / slice_kb;
    a.tma_epi = 0;
    if (bn <= 64 && hidden % 4 == 0 && inter % 8 == 0 && ((uintptr_t)planes & 15) == 0 && ((uintptr_t)act & 15) == 0 &&
        !getenv("RR_NO_TMA_EPI")) {
        rc = make_tmap_act_store(&a.tmAct, act, rows, inter, inter, bn);
        if (rc == RR_OK) rc = make_tmap_planes_f32(&a.tmPlanes, planes, hidden, hidden, rows, ld_rows, p->n_slices, bn);
        if (rc != RR_OK) return rc;
        a.tma_epi = 1;
    }
    return RR_OK;
}

template <int BN>
static int launch_mlp_bn(const MlpPlan& p, cudaStream_t st) {
    auto kern = gemm_mlp_tcgen05<BN>;
    static std::atomic<uint64_t> attr_set{0};
    constexpr int smem = GemmCfg<BN>::kSmemBytes + mlp_stage_bytes<BN>();
    static_assert(smem <= 227 * 1024, "fused MLP kernel: shared memory budget");
    if (ensure_dyn_smem(kern, smem, attr_set) != cudaSuccess) return RR_ERR_CUDA;
    cudaError_t e = launch_pdl(kern, dim3(p.grid), dim3(GEMM_THREADS), (size_t)smem, st, p.args);
    return e == cudaSuccess ? RR_OK : RR_ERR_CUDA;
}
// Requires all CTAs co-resident (grid <= SM count; one CTA per SM by shared memory) and ready[] zero at launch.
int mlp_launch(const MlpPlan& p, cudaStream_t st) {
    switch (p.bn) {
        case 32: return launch_mlp_bn<32>(p, st);
        case 64: return launch_mlp_bn<64>(p, st);
        case 128: return launch_mlp_bn<128>(p, st);
        case 256: return launch_mlp_bn<256>(p, st);
    }
    return RR_ERR_ARG;
}

void rr_trace_set_gemm(unsigned long long* p) { rr_trace_set_local(p); }
void rr_trace_set_gemm_detail(int on) { rr_trace_set_detail_local(on); }

}  // namespace rr
