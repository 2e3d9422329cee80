// Thin inline-PTX layer for sm_100a: mbarrier, bulk async copy (TMA, 1-D), tcgen05 (TMEM alloc,
// MMA, commit, load) and the 128-byte swizzle used by every operand image in this library.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace stdadk {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// One arrival per WARP for barriers that collect the workers' shared-memory writes: every lane has fenced its own
// writes, the warp converges, one lane arrives.  An mbarrier is a word in shared memory and arrivals on it are
// serialised (a 256-thread CTA arriving thread by thread cost ~1.5 us per operand slab, measured with the phase timers
// of the profiling build); the barrier counts are therefore in warps.
__device__ __forceinline__ void mbar_arrive_warp(uint64_t* bar) {
    __syncwarp();
    if ((threadIdx.x & 31u) == 0u) mbar_arrive(bar);
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
// try_wait suspends the thread in hardware until the phase completes or `hint_ns` elapses: a waiting warp issues
// one instruction per time slice instead of spinning, so it does not take issue slots from the warps doing the work.
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity, uint32_t hint_ns = 20000u) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity), "r"(hint_ns)
        : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug traps (launch error) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > 4000000000LL) __trap();
    }
}

// ---------------------------------------------------------------- programmatic dependent launch
// The training step's kernels are launched with programmatic stream serialisation (api.cu, launch_chained): kernel
// N+1 may become resident while kernel N still runs, does its independent set-up, and blocks in pdl_wait() until N has
// completed and its writes are visible.  pdl_wait() returns at once when the kernel has no programmatic prerequisite
// (eager launches after a plain kernel, the first kernel of a graph).  Every kernel that uses them keeps these rules:
//  1. A CTA calls pdl_launch_dependents() only after it has passed its own pdl_wait() and its own tcgen05.alloc.  So
//     when kernel N+1 starts, kernel N-1 has completed: code before N+1's wait overlaps kernel N only, and a dependent
//     CTA that allocates tensor memory before its wait can only contend with CTAs that already hold theirs.
//  2. Code before the wait reads only data written before the step began or by kernels at least two launches back on
//     the same stream (parameters, knot tables, weight images, activations of earlier blocks), and writes only
//     shared and tensor memory.  Every thread that reads a predecessor's output or writes global memory waits first.
//     Epilogue inputs count too: where the caller states that an input is that old (stdadk_bwd_args.settled for the
//     dropout step counter and for a saved x image and its stats, stdadk_adamw_args.state_early for the fused tail's
//     optimizer state, hyper-parameters and step counter), the one-wave backward's keep bits, x^ and activation bits
//     and the tail's state are formed or loaded before the wait.
//  3. A grid-wide barrier (the fused step tail) sits after the wait, where the prerequisites have exited.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ---------------------------------------------------------------- proxies / fences
__device__ __forceinline__ void fence_proxy_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// ---------------------------------------------------------------- bulk async copy global -> shared (TMA 1-D)
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// ---------------------------------------------------------------- TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)),
                 "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// 32 lanes x 32 consecutive 32-bit columns: thread i of the warp receives lane (base_lane + i).
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// The accumulator of an M = 64 MMA (cta_group::1) fills lanes 0-15 of each warp's 32-lane quarter.  16 lanes x two
// runs of 32 consecutive 32-bit columns, the second `split` columns after the first: thread i of the warp receives lane
// (base_lane + i % 16), run i / 16.
template <int SPLIT>
__device__ __forceinline__ void tmem_ld16x2(uint32_t taddr, float (&v)[32]) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.16x32bx2.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32], %33;"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr), "n"(SPLIT)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// Issue only (no wait): several loads can be in flight before one tmem_ld_wait().
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, float (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=f"(r[0]), "=f"(r[1]), "=f"(r[2]), "=f"(r[3]), "=f"(r[4]), "=f"(r[5]), "=f"(r[6]), "=f"(r[7]),
          "=f"(r[8]), "=f"(r[9]), "=f"(r[10]), "=f"(r[11]), "=f"(r[12]), "=f"(r[13]), "=f"(r[14]), "=f"(r[15]),
          "=f"(r[16]), "=f"(r[17]), "=f"(r[18]), "=f"(r[19]), "=f"(r[20]), "=f"(r[21]), "=f"(r[22]), "=f"(r[23]),
          "=f"(r[24]), "=f"(r[25]), "=f"(r[26]), "=f"(r[27]), "=f"(r[28]), "=f"(r[29]), "=f"(r[30]), "=f"(r[31])
        : "r"(taddr)
        : "memory");
}
// The wait names every destination register as an in/out operand so that no use of the loaded values can be
// scheduled above it.
__device__ __forceinline__ void tmem_ld_wait(float (&r)[32]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+f"(r[0]), "+f"(r[1]), "+f"(r[2]), "+f"(r[3]), "+f"(r[4]), "+f"(r[5]), "+f"(r[6]), "+f"(r[7]),
                   "+f"(r[8]), "+f"(r[9]), "+f"(r[10]), "+f"(r[11]), "+f"(r[12]), "+f"(r[13]), "+f"(r[14]), "+f"(r[15]),
                   "+f"(r[16]), "+f"(r[17]), "+f"(r[18]), "+f"(r[19]), "+f"(r[20]), "+f"(r[21]), "+f"(r[22]), "+f"(r[23]),
                   "+f"(r[24]), "+f"(r[25]), "+f"(r[26]), "+f"(r[27]), "+f"(r[28]), "+f"(r[29]), "+f"(r[30]), "+f"(r[31])
                 :
                 : "memory");
}

// 32 lanes x 32 consecutive 32-bit columns, registers -> TMEM (thread i of the warp writes lane base_lane + i)
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const float (&v)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
        ::"r"(taddr), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]), "f"(v[8]),
          "f"(v[9]), "f"(v[10]), "f"(v[11]), "f"(v[12]), "f"(v[13]), "f"(v[14]), "f"(v[15]), "f"(v[16]), "f"(v[17]),
          "f"(v[18]), "f"(v[19]), "f"(v[20]), "f"(v[21]), "f"(v[22]), "f"(v[23]), "f"(v[24]), "f"(v[25]), "f"(v[26]),
          "f"(v[27]), "f"(v[28]), "f"(v[29]), "f"(v[30]), "f"(v[31])
        : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---------------------------------------------------------------- UMMA descriptors
// Shared-memory matrix descriptor, 128-byte swizzle (cute/arch/mma_sm100_desc.hpp field layout):
// [0,14) addr>>4 | [16,30) LBO>>4 | [32,46) SBO>>4 | [46,48) version=1 | [61,64) layout=2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46) | (2ull << 61);
}
// Instruction descriptor, kind::tf32, FP32 accumulate, M = 128 or 64 (cta_group::1).
// c_format[4,6)=1 (F32) a_format[7,10)=2 (TF32) b_format[10,13)=2 a_major[15] b_major[16] (1 = MN-major)
// n_dim[17,23)=N>>3 m_dim[24,29)=M>>4
__device__ __forceinline__ uint32_t umma_idesc_tf32(uint32_t n, uint32_t a_mn_major, uint32_t b_mn_major,
                                                    uint32_t m = 128) {
    return (1u << 4) | (2u << 7) | (2u << 10) | (a_mn_major << 15) | (b_mn_major << 16) | ((n >> 3) << 17) |
           ((m >> 4) << 24);
}
// D[tmem] (+)= A[smem] * B[smem]; issued by ONE thread.
__device__ __forceinline__ void umma_tf32(uint32_t taddr, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(taddr), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]: the A operand (M = 128 lanes x K 32-bit columns) is read from tensor memory, so
// neither writing it nor fetching it touches the shared-memory pipe.
__device__ __forceinline__ void umma_tf32_ts(uint32_t taddr, uint32_t a_taddr, uint64_t bdesc, uint32_t idesc,
                                             uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(taddr), "r"(a_taddr), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// mbarrier arrives when all previously issued MMAs of this thread have completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}

// ---------------------------------------------------------------- operand image addressing
// Every operand (activation tile, weight slab, generated basis slab) is stored as rows of 128 bytes
// whose eight 16-byte chunks are XOR-swizzled with (row & 7): exactly the SWIZZLE_128B pattern the
// tensor core applies to shared-memory addresses, so an image in HBM is a byte copy of its SMEM form.
__device__ __forceinline__ uint32_t swz_off(uint32_t row, uint32_t chunk) {
    return row * 128u + ((chunk ^ (row & 7u)) << 4);
}
// Round to TF32 (10-bit mantissa), nearest with ties away from zero: add half an ulp to the magnitude bits and
// truncate -- what cvt.rna.tf32.f32 computes for every finite input (the compiler expands that cvt into four
// instructions on sm_100 to also preserve NaN payloads; operands here are finite).
__device__ __forceinline__ float to_tf32(float x) {
    return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xFFFFE000u);
}
// tf32x3 operand split: a value is fed to the tensor cores as hi = tf32(x) and lo = tf32(x - hi) (x - hi is exact in
// FP32); hi*hi + hi*lo + lo*hi accumulated in FP32 reproduces the FP32 product to ~2^-21.  `lo` selects the part.
__device__ __forceinline__ float tf32_part(float x, bool lo) {
    const float hi = to_tf32(x);
    return lo ? to_tf32(x - hi) : hi;
}
// Packed FP32 (two lanes per instruction, FFMA2 / FADD2 on sm_100): same rounding as the scalar forms, half the
// issue slots.  ptxas pairs the registers without moves when the operands come from adjacent array elements.
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) {
    float2 d;
    asm("{\n\t.reg .b64 ra, rb, rc, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tmov.b64 rc, {%6, %7};\n\t"
        "fma.rn.f32x2 rd, ra, rb, rc;\n\tmov.b64 {%0, %1}, rd;\n\t}"
        : "=f"(d.x), "=f"(d.y)
        : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
    return d;
}
__device__ __forceinline__ float2 add2(float2 a, float2 b) {
    float2 d;
    asm("{\n\t.reg .b64 ra, rb, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\t"
        "add.rn.f32x2 rd, ra, rb;\n\tmov.b64 {%0, %1}, rd;\n\t}"
        : "=f"(d.x), "=f"(d.y)
        : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
    return d;
}
__device__ __forceinline__ float2 mul2(float2 a, float2 b) {
    float2 d;
    asm("{\n\t.reg .b64 ra, rb, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\t"
        "mul.rn.f32x2 rd, ra, rb;\n\tmov.b64 {%0, %1}, rd;\n\t}"
        : "=f"(d.x), "=f"(d.y)
        : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
    return d;
}
// a - b with the subtraction's own single rounding: b * (-1) is exact inside the fma
__device__ __forceinline__ float2 sub2(float2 a, float2 b) { return fma2(b, make_float2(-1.0f, -1.0f), a); }
__device__ __forceinline__ void st_shared_v4(uint32_t saddr, float a, float b, float c, float d) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(saddr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

}  // namespace stdadk
