// rr_ptx.cuh — thin inline-PTX wrappers for sm_100a (Blackwell B200).
//
// mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit / ld)
// and a few cache-hinted vector loads. Nothing here is portable: this
// file only compiles for compute_100a.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda.h>
#include <stdint.h>

namespace rr {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// One lane of a fully-converged warp is elected; returns true in that lane.
__device__ __forceinline__ bool elect_one() {
    uint32_t pred = 0;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}\n"
        : "=r"(pred));
    return pred != 0;
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
// 1024-byte aligned start of the dynamic shared memory (128B-swizzled TMA tiles / UMMA descriptors need it).  Pointer
// arithmetic on the __shared__ array itself: rounding the pointer up through uintptr_t loses the address space and every access
// through the result becomes a GENERIC load / store (LD.E / ST.E instead of LDS / STS), which the compiler must also keep in
// program order against each other -- the SiLU epilogue of the decode MLP ran at 220 cycles per element because of that.
__device__ __forceinline__ uint8_t* align_smem_1024(uint8_t* raw) {
    return raw + ((1024u - (smem_u32(raw) & 1023u)) & 1023u);
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Spin (HW-assisted sleep inside try_wait) until the phase with `parity` completes.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {
    }
}

// ---------------------------------------------------------------- TMA
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// 2-D tiled load global -> shared, completion on mbarrier (complete_tx::bytes).
// c0 = innermost coordinate (elements), c1 = row coordinate.
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar,
                                            int32_t c0, int32_t c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)),
        "r"(c0), "r"(c1)
        : "memory");
}
// Same, with an L2 cache-policy operand (createpolicy result).
__device__ __forceinline__ void tma_load_2d_hint(void* smem_dst, const CUtensorMap* m,
                                                 uint64_t* bar, int32_t c0, int32_t c1,
                                                 uint64_t policy) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
        " [%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)),
        "r"(c0), "r"(c1), "l"(policy)
        : "memory");
}
// ---- TMA stores (shared -> global, bulk async-group completion)
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* smem_src, int32_t c0, int32_t c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                 ::"l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* m, const void* smem_src, int32_t c0, int32_t c1, int32_t c2) {
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
                 ::"l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// the committed bulk stores of this thread have READ their shared-memory source (it may be overwritten)
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// ... have completed (their global writes are performed)
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}

// ---------------------------------------------------------------- tcgen05 / TMEM
__device__ __forceinline__ void tcgen05_fence_before() {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tcgen05_fence_after() {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// Whole warp executes. Writes the TMEM base address (lane<<16 | column) to *smem_dst.
template <uint32_t kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst) {
    static_assert(kCols >= 32 && kCols <= 512 && (kCols & (kCols - 1)) == 0, "TMEM cols");
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(smem_dst)),
                 "n"(kCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols)
                 : "memory");
}

// D[tmem] (+)= A[smem desc] * B[smem desc]; bf16 x bf16 -> fp32 (kind::f16).
__device__ __forceinline__ void umma_bf16_ss(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                             uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}\n"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// All previously issued tcgen05.mma of this thread arrive (once) on `bar` when they complete.
// Implies tcgen05.fence::before_thread_sync.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                     smem_u32(bar))
                 : "memory");
}

// TMEM -> registers: this warp's 32 lanes x 32 consecutive fp32 columns.
// Thread i of the warp receives TMEM lane (taddr.lane + i), columns [col, col+32).
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
          "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
          "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]),
          "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]),
          "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
          "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
          "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// Shared-memory matrix descriptor for a K-major bf16 tile stored with the 128-byte swizzle
// (rows of 64 bf16 = 128 B, groups of 8 rows = 1024 B, exactly what a TMA box {64, rows}
// with CU_TENSOR_MAP_SWIZZLE_128B writes). Field layout: cute::UMMA::SmemDescriptor
// (start>>4 [0,14), LBO>>4 [16,30), SBO>>4 [32,46), version=1 [46,48), layout_type [61,64)).
__device__ __forceinline__ uint64_t umma_desc_sw128_kmajor(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);   // start address
    d |= static_cast<uint64_t>(1) << 16;                       // LBO (ignored for swizzled K-major)
    d |= static_cast<uint64_t>(1024 >> 4) << 32;               // SBO: 8 rows * 128 B
    d |= static_cast<uint64_t>(1) << 46;                       // descriptor version (sm_100)
    d |= static_cast<uint64_t>(2) << 61;                       // SWIZZLE_128B
    return d;
}
// Instruction descriptor (cute::UMMA::InstrDescriptor): bf16 A/B, fp32 D, both K-major.
__host__ __device__ constexpr uint32_t umma_idesc_bf16_f32(uint32_t M, uint32_t N) {
    return (1u << 4)                 // c_format  = F32
           | (1u << 7)               // a_format  = BF16
           | (1u << 10)              // b_format  = BF16
           | ((N >> 3) << 17)        // n_dim
           | ((M >> 4) << 24);       // m_dim
}

// ---------------------------------------------------------------- misc loads
__device__ __forceinline__ uint4 ldg_nc_v4(const void* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}

__device__ __forceinline__ float bf16_lo(uint32_t packed) { return __uint_as_float(packed << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t packed) {
    return __uint_as_float(packed & 0xFFFF0000u);
}
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
}

}  // namespace rr
