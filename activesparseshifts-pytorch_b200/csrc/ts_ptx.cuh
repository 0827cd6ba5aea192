// ts_ptx.cuh -- mbarrier / TMA / bulk-copy / cp.async / named-barrier PTX wrappers and launch-invariant fast division
// shared by every kernel family.
#pragma once
#include "ts_common.cuh"

namespace ts {
namespace ptx {

TS_D void mbar_init(uint64_t* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(shared_addr(bar)), "r"(count) : "memory");
}
TS_D void mbar_expect_tx(uint64_t* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(shared_addr(bar)), "r"(bytes) : "memory");
}
TS_D void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(shared_addr(bar)) : "memory");
}
TS_D void mbar_wait(uint64_t* bar, unsigned parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred P1;\n\t"
        "LAB_WAIT:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
        "@P1 bra DONE;\n\t"
        "bra LAB_WAIT;\n\t"
        "DONE:\n\t"
        "}" ::"r"(shared_addr(bar)), "r"(parity) : "memory");
}
// Wait of the arithmetic warps: try_wait with a suspend-time hint -- the warp is parked by the hardware until the phase
// completes (or the hint expires) instead of re-issuing TRYWAIT / BRA every few cycles (ncu: the spin of 14 waiting
// warps was 18 % of all issued instructions of the 3-D backward and competed with the working warps for issue slots).
TS_D void mbar_wait_parked(uint64_t* bar, unsigned parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred P1;\n\t"
        "LAB_WAIT:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1, %2;\n\t"
        "@P1 bra DONE;\n\t"
        "bra LAB_WAIT;\n\t"
        "DONE:\n\t"
        "}" ::"r"(shared_addr(bar)), "r"(parity), "r"(20000u) : "memory");
}
// Wait of a thread that runs AHEAD of the arithmetic warps (producer, fixer): between polls it sleeps instead of
// competing with them for issue slots (ncu: the spin loops of these two warps were ~10 % of all issued instructions
// of the instruction-bound 3-D backward).
TS_D void mbar_wait_relaxed(uint64_t* bar, unsigned parity, unsigned sleep_ns) {
    for (;;) {
        unsigned ok;
        asm volatile(
            "{\n\t"
            ".reg .pred P1;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, P1;\n\t"
            "}" : "=r"(ok) : "r"(shared_addr(bar)), "r"(parity) : "memory");
        if (ok) return;
        __nanosleep(sleep_ns);
    }
}
TS_D void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
// generic-proxy writes to shared memory made visible to / ordered before later async-proxy (TMA) accesses
TS_D void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// tiled 5-D TMA load global -> shared; coordinates innermost first; out-of-tensor elements arrive as zero.
// c0 must be a multiple of 16 bytes worth of elements.
TS_D void tma_load_5d(void* dst, const void* map, int c0, int c1, int c2, int c3, int c4, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5, %6}], [%7];" ::"r"(
            shared_addr(dst)),
        "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4), "r"(shared_addr(bar))
        : "memory");
}
// 1-D bulk async copy global -> shared, completion reported to an mbarrier (SASS: UBLKCP)
TS_D void bulk_g2s(void* dst, const void* src, unsigned bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(shared_addr(dst)),
                 "l"(src), "r"(bytes), "r"(shared_addr(bar))
                 : "memory");
}
// 1-D bulk copy shared -> global (SASS UBLKCP / bulk store), tracked by the issuing thread's bulk async-group
TS_D void bulk_s2g(void* dst_global, const void* src_shared, unsigned bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_global), "r"(shared_addr(src_shared)), "r"(bytes)
                 : "memory");
}
TS_D void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N> TS_D void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
template <int N> TS_D void bulk_wait() { asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory"); }
// 16-byte cp.async global -> shared (L2 only), tracked by the issuing thread's cp.async groups; dst is a shared-window address
TS_D void cp_async16(unsigned dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
TS_D void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> TS_D void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
// barrier among `count` threads (a multiple of 32) of the CTA, id 1..15 (0 is __syncthreads)
TS_D void named_barrier(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }

}  // namespace ptx

// ---- exact division by a launch-invariant (n < 2^31; FastDiv: ts_common.cuh) -------------------
TS_D unsigned fdiv(unsigned n, const FastDiv& f) { return (__umulhi(n, f.m) + n) >> f.l; }

}  // namespace ts
