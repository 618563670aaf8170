// slb_ptx.cuh -- the PTX and warp primitives every kernel of the library shares: warp reductions and broadcasts, the
// mbarrier, TMA bulk copies (global <-> shared, L2 prefetch), 8-byte cp.async (LDGSTS) and the m8n8k4 FP64 DMMA.
// Each is inline asm (or a shuffle intrinsic), so a -fmad=false translation unit emits the same instructions.
#pragma once
#include "slb_math.cuh"

namespace slbd {

constexpr unsigned FULL = 0xffffffffu;
SLB_DEV double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}
SLB_DEV double bcast(double v, int src) { return __shfl_sync(FULL, v, src); }

SLB_DEV unsigned saddr(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }

// ---- mbarrier and TMA bulk copies (global -> shared completes on an mbarrier; shared -> global on a bulk group) ----
SLB_DEV void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(saddr(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
}
SLB_DEV void mbar_expect_tx(uint64_t *bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(saddr(bar)), "r"(bytes) : "memory");
}
SLB_DEV void mbar_wait(uint64_t *bar, unsigned parity) {
    unsigned done = 0;
    while (!done) {
        asm volatile(
            "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
            : "=r"(done)
            : "r"(saddr(bar)), "r"(parity)
            : "memory");
    }
}
SLB_DEV void bulk_g2s(void *dst, const void *src, unsigned bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(saddr(dst)),
                 "l"(src), "r"(bytes), "r"(saddr(bar))
                 : "memory");
}
SLB_DEV void bulk_s2g(void *gdst, const void *ssrc, unsigned bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;\n cp.async.bulk.commit_group;\n" ::"l"(gdst),
                 "r"(saddr(ssrc)), "r"(bytes)
                 : "memory");
}
SLB_DEV void bulk_prefetch_l2(const void *gsrc, unsigned bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;\n" ::"l"(gsrc), "r"(bytes) : "memory");
}
SLB_DEV void bulk_store_wait() { asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory"); }
SLB_DEV void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory"); }

// ---- 8-byte cp.async (LDGSTS): every load of a lane is in flight before the first one lands ------------------------
SLB_DEV void cp_async8(double *smem_dst, const double *gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(saddr(smem_dst)), "l"(gsrc) : "memory");
}
SLB_DEV void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
SLB_DEV void cp_async_wait0() { asm volatile("cp.async.wait_group 0;\n" ::: "memory"); }
SLB_DEV void cp_async_wait_all() { asm volatile("cp.async.commit_group;\n cp.async.wait_group 0;\n" ::: "memory"); }

// D(8x8) += A(8x4) B(4x8) on the FP64 tensor path: lane holds a = A[lane>>2][lane&3], b = B[lane&3][lane>>2] and the
// accumulator pair d0 = D[lane>>2][2*(lane&3)], d1 = D[lane>>2][2*(lane&3)+1].
SLB_DEV void dmma884(double &d0, double &d1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(d0), "+d"(d1)
                 : "d"(a), "d"(b));
}

}  // namespace slbd
