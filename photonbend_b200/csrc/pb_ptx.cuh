// pb_ptx.cuh -- thin inline-PTX wrappers (sm_100a): mbarrier, TMA bulk copies (cp.async.bulk,
// SASS UBLKCP), async-proxy fences.
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

namespace pb {
namespace ptx {

__device__ __forceinline__ uint32_t smem_addr(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbarrier_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count) : "memory");
}

// make mbarrier.init visible to the async proxy (TMA) before the first bulk copy targets it
__device__ __forceinline__ void fence_mbarrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

__device__ __forceinline__ void mbarrier_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes)
                 : "memory");
}

// a plain arrival (release: this thread's earlier shared-memory accesses are ordered before it)
__device__ __forceinline__ void mbarrier_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_addr(bar)) : "memory");
}
__device__ __forceinline__ void mbarrier_arrive_sa(uint32_t bar_sa) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar_sa) : "memory");
}

__device__ __forceinline__ bool mbarrier_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(ok)
        : "r"(smem_addr(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}

__device__ __forceinline__ void mbarrier_wait(uint64_t* bar, uint32_t parity) {
    while (!mbarrier_try_wait(bar, parity)) {
    }
}

// global -> shared bulk copy (TMA, 1-D): 16-byte aligned addresses, size a multiple of 16;
// completion is signalled on `bar` as a transaction of `bytes` bytes.
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_addr(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_addr(bar))
                 : "memory");
}

// shared -> global bulk copy (TMA, 1-D), tracked by the per-thread bulk async-group
__device__ __forceinline__ void bulk_s2g(void* gmem_dst, const void* smem_src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmem_dst),
                 "r"(smem_addr(smem_src)), "r"(bytes)
                 : "memory");
}

__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }

// wait until the bulk stores of this thread have finished READING shared memory
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }

// wait until at most one bulk store group of this thread is still reading shared memory
__device__ __forceinline__ void bulk_wait_read1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }

// TMA tensor-map (cuTensorMapEncodeTiled) 3-D box load: global -> shared, completion on `bar`.
// Coordinates are in elements of the map, innermost first; out-of-bounds parts of the box are
// zero-filled by the hardware.
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const void* tmap, int c0, int c1, int c2, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(
            smem_addr(smem_dst)),
        "l"(reinterpret_cast<uint64_t>(tmap)), "r"(c0), "r"(c1), "r"(c2), "r"(smem_addr(bar))
        : "memory");
}

// TMA tensor-map 3-D box store: shared -> global (clipped to the tensor's bounds), bulk async-group
__device__ __forceinline__ void tma_store_3d(const void* tmap, int c0, int c1, int c2, const void* smem_src) {
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.tile.bulk_group [%0, {%1, %2, %3}], [%4];" ::"l"(
                     reinterpret_cast<uint64_t>(tmap)),
                 "r"(c0), "r"(c1), "r"(c2), "r"(smem_addr(smem_src))
                 : "memory");
}

// L2 eviction-priority policies for bulk copies: the source is re-read by neighbouring tiles
// (keep it), the output is written once (let it go first)
__device__ __forceinline__ uint64_t policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t policy_evict_last() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}

__device__ __forceinline__ uint64_t policy_evict_normal() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(p));
    return p;
}
// 0 = evict_last, 1 = evict_normal, 2 = evict_first
__device__ __forceinline__ uint64_t policy_of(int k) {
    return k == 0 ? policy_evict_last() : k == 1 ? policy_evict_normal() : policy_evict_first();
}

__device__ __forceinline__ void tma_load_3d_hint(void* smem_dst, const void* tmap, int c0, int c1, int c2, uint64_t* bar,
                                                 uint64_t policy) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%2, %3, %4}], [%5], %6;" ::"r"(
            smem_addr(smem_dst)),
        "l"(reinterpret_cast<uint64_t>(tmap)), "r"(c0), "r"(c1), "r"(c2), "r"(smem_addr(bar)), "l"(policy)
        : "memory");
}

__device__ __forceinline__ void tma_store_3d_hint(const void* tmap, int c0, int c1, int c2, const void* smem_src,
                                                  uint64_t policy) {
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.tile.bulk_group.L2::cache_hint [%0, {%1, %2, %3}], [%4], %5;" ::"l"(
                     reinterpret_cast<uint64_t>(tmap)),
                 "r"(c0), "r"(c1), "r"(c2), "r"(smem_addr(smem_src)), "l"(policy)
                 : "memory");
}

// TMA tensor-map 3-D box prefetch: global -> L2 only (no shared memory, no completion to wait for)
__device__ __forceinline__ void tma_prefetch_l2_3d(const void* tmap, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global.tile [%0, {%1, %2, %3}];" ::"l"(
                     reinterpret_cast<uint64_t>(tmap)),
                 "r"(c0), "r"(c1), "r"(c2)
                 : "memory");
}

__device__ __forceinline__ void prefetch_tensormap(const void* tmap) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}

// shared-memory counter shared by the warps of a block: the add releases this warp's reads of a
// stage buffer and acquires those of the warps that counted before it
__device__ __forceinline__ unsigned atom_add_acq_rel_shared(unsigned* p, unsigned v) {
    unsigned old;
    asm volatile("atom.acq_rel.cta.shared::cta.add.u32 %0, [%1], %2;" : "=r"(old) : "r"(smem_addr(p)), "r"(v) : "memory");
    return old;
}

// the same on a shared-window address (saves the generic -> shared conversion in a hot loop)
__device__ __forceinline__ void mbarrier_wait_sa(uint32_t bar_sa, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t"
            "}"
            : "=r"(ok)
            : "r"(bar_sa), "r"(parity)
            : "memory");
    } while (!ok);
}

// The 3 bytes of a pixel that starts at byte (shift / 8) % 4 of the aligned shared-memory word at
// word_sa + offset (+ one byte of garbage on top): two words and a funnel shift (SHF takes its
// count modulo 32).
__device__ __forceinline__ uint32_t lds_pixel(uint32_t word_sa, uint32_t offset, uint32_t shift) {
    uint32_t lo, hi;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(lo) : "r"(word_sa + offset));
    asm volatile("ld.shared.b32 %0, [%1+4];" : "=r"(hi) : "r"(word_sa + offset));
    return __funnelshift_r(lo, hi, shift);
}

// The same with the second word loaded only by the lanes whose pixel runs into it (byte offset
// 2 or 3 within the word): half the lanes sit the second LDS out, which roughly halves its bank
// conflicts, at the price of one predicate-setting instruction.
__device__ __forceinline__ uint32_t lds_pixel_pred(uint32_t byte_sa) {
    uint32_t lo, hi;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        ".reg .b32 a, t;\n\t"
        "and.b32 a, %2, 0xfffffffc;\n\t"
        "and.b32 t, %2, 2;\n\t"
        "setp.ne.u32 p, t, 0;\n\t"
        "ld.shared.b32 %0, [a];\n\t"
        "mov.b32 %1, 0;\n\t"
        "@p ld.shared.b32 %1, [a+4];\n\t"
        "}"
        : "=r"(lo), "=r"(hi)
        : "r"(byte_sa));
    return __funnelshift_r(lo, hi, byte_sa << 3);
}

// lds_pixel with the second word loaded only where the pixel runs into it (shift = 16 or 24)
__device__ __forceinline__ uint32_t lds_pixel_sparse(uint32_t word_sa, uint32_t offset, uint32_t shift) {
    uint32_t lo, hi;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        ".reg .b32 t;\n\t"
        "and.b32 t, %3, 16;\n\t"
        "setp.ne.u32 p, t, 0;\n\t"
        "ld.shared.b32 %0, [%2];\n\t"
        "mov.b32 %1, 0;\n\t"
        "@p ld.shared.b32 %1, [%2+4];\n\t"
        "}"
        : "=r"(lo), "=r"(hi)
        : "r"(word_sa + offset), "r"(shift));
    return __funnelshift_r(lo, hi, shift);
}

__device__ __forceinline__ void sts32(uint32_t sa, uint32_t v) {
    asm volatile("st.shared.b32 [%0], %1;" ::"r"(sa), "r"(v) : "memory");
}

// generic-proxy writes to shared memory -> visible to the async proxy (before a bulk store)
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

}  // namespace ptx
}  // namespace pb
