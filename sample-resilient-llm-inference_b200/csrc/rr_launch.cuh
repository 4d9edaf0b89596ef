// rr_launch.cuh — programmatic dependent launch (PDL) plumbing.
//
// Every kernel of the library calls griddep_launch() at its top (lets the next kernel in the stream
// start its prologue / constant-data prefetch early) and griddep_wait() before it touches anything
// the preceding kernel produced.  Launched through launch_pdl() the stream edge becomes a programmatic
// dependency (also inside CUDA-graph capture); launched normally both instructions are no-ops.
#pragma once
#include <cuda_runtime.h>
#include <atomic>
#include <cstdint>
#include <utility>

namespace rr {

__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void griddep_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ---- optional in-kernel timeline (debug): CTA (0,0,0) thread 0 of every kernel records
// (kernel id, globaltimer at start, after griddepcontrol.wait, at end) into a device buffer; rr_debug_trace_*.
// Each translation unit owns its copy of the pointer (no -rdc); rr_api.cu sets them all.
static __device__ unsigned long long* rr_trace_ptr = nullptr;
static __device__ int rr_trace_detail = 0;      // 1: also per-item marks of sample CTAs (trace_mark_fixed / trace_mark_at), a few % slower
static inline void rr_trace_set_local(unsigned long long* p) { cudaMemcpyToSymbol(rr_trace_ptr, &p, sizeof(p)); }
static inline void rr_trace_set_detail_local(int on) { cudaMemcpyToSymbol(rr_trace_detail, &on, sizeof(on)); }
enum TraceId { TR_GEMM_DEC = 1, TR_GEMM_PF = 2, TR_ATTN_DEC = 3, TR_ATTN_PF = 4, TR_NORM = 5, TR_ROPE = 6,
               TR_SILU = 7, TR_EMBED = 8, TR_ARGMAX = 9, TR_COMBINE = 10, TR_MISC = 11,
               TR_MLP_MARK = 50, TR_ATTN_MARK = 80, TR_GEMM_MARK = 100 };  // + k: sample CTAs of the fused MLP kernel (tools/trace_mlp.py)
__device__ __forceinline__ unsigned long long rr_gtimer() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ int trace_begin(int kid) {
    unsigned long long* p = rr_trace_ptr;
    if (p == nullptr || (blockIdx.x | blockIdx.y | blockIdx.z | threadIdx.x) != 0) return -1;
    const int slot = (int)atomicAdd(p, 1ull);
    if (slot >= (int)p[1]) return -1;
    p[2 + 4 * slot] = (unsigned long long)kid;
    p[3 + 4 * slot] = rr_gtimer();
    return slot;
}
// after griddepcontrol.wait returned: the preceding grid has completed and flushed
__device__ __forceinline__ void trace_dep(int slot) {
    if (slot >= 0) rr_trace_ptr[4 + 4 * slot] = rr_gtimer();
}
// Marker from a few sample CTAs (0, 37, 74, 111, ...): kid in the low byte, CTA index above it.  NO atomic: the slot is a
// fixed function of (sample CTA, idx) at the END of the buffer, so the marking thread never waits for a memory round trip
// (an atomicAdd with a result costs 2-4 us under a saturated weight stream and would distort exactly the latencies being
// measured).  idx < 192 per CTA; rr_debug_trace_stop returns the whole buffer while detail marks are on and the reader
// drops the empty rows.
__device__ __forceinline__ void trace_mark_fixed(int kid, int idx) {
    unsigned long long* p = rr_trace_ptr;
    if (p == nullptr || rr_trace_detail == 0 || blockIdx.x % 37 != 0 || idx >= 192) return;
    const unsigned long long t = rr_gtimer();
    const long long slot = (long long)p[1] - 1 - ((long long)(blockIdx.x / 37) * 192 + idx);
    if (slot < 0) return;
    p[2 + 4 * slot] = (unsigned long long)(kid | ((int)blockIdx.x << 8));
    p[3 + 4 * slot] = t; p[4 + 4 * slot] = t; p[5 + 4 * slot] = t;
}
// fixed-slot mark with an explicit sample index (kernels whose sample CTAs are not blockIdx.x % 37 == 0): sample < 4, idx < 192
__device__ __forceinline__ void trace_mark_at(int kid, int sample, int idx) {
    unsigned long long* p = rr_trace_ptr;
    if (p == nullptr || rr_trace_detail == 0 || idx >= 192) return;
    const unsigned long long t = rr_gtimer();
    const long long slot = (long long)p[1] - 1 - ((long long)sample * 192 + idx);
    if (slot < 0) return;
    p[2 + 4 * slot] = (unsigned long long)(kid | (sample << 8));
    p[3 + 4 * slot] = t; p[4 + 4 * slot] = t; p[5 + 4 * slot] = t;
}
__device__ __forceinline__ void trace_end(int slot) {
    if (slot >= 0) rr_trace_ptr[5 + 4 * slot] = rr_gtimer();
}

// cudaFuncSetAttribute applies to the current device only: one process may host several replicas (the HTTP gateway
// runs one engine per GPU), so "already raised" is tracked per device (bit = device ordinal), lock-free.
template <typename K>
inline cudaError_t ensure_dyn_smem(K kern, int bytes, std::atomic<uint64_t>& done) {
    int dev = 0;
    cudaGetDevice(&dev);
    const uint64_t bit = 1ull << (dev & 63);
    if (done.load(std::memory_order_acquire) & bit) return cudaSuccess;
    const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e == cudaSuccess) done.fetch_or(bit, std::memory_order_release);
    return e;
}

extern int g_use_pdl;   // rr_api.cu; env RR_NO_PDL=1 or rr_set_pdl(0) turns it off

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                              Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = g_use_pdl ? 1 : 0;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, KArgs(std::forward<Args>(args))...);
}

}  // namespace rr
