// umma.cuh — thin inline-PTX layer for sm_100a: mbarrier, 1-D bulk async copy (TMA engine),
// TMEM allocation, tcgen05.mma / commit / ld, and the shared-memory matrix descriptors.
// Everything here is a direct PTX-ISA wrapper; the kernels built on it are in trunk_fused.cu
// and umma_selftest.cu.
#pragma once
#include <cuda_bf16.h>
#include <stdint.h>

namespace nsb {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}

// One lane of the (fully converged) warp; the blessed idiom for single-thread tcgen05 issue: the
// compiler keeps warp-uniform operands in uniform registers instead of waterfall-looping R2UR.
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred P1;\n\t"
        "elect.sync _|P1, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, P1;\n\t}"
        : "=r"(pred));
    return pred != 0;
}

// ---- mbarrier -------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    return done != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {
    }
}

// ---- proxies / fences -----------------------------------------------------------------------
// Generic-proxy smem writes must be fenced before the async proxy (tcgen05.mma, bulk copy) reads.
__device__ __forceinline__ void fence_proxy_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
// non-blocking arrival on a named barrier that other warps wait on with named_bar_sync
__device__ __forceinline__ void named_bar_arrive(uint32_t id, uint32_t nthreads) {
    asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ---- bulk async copy global -> shared (SASS: UBLKCP), completes on an mbarrier ---------------
__device__ __forceinline__ void bulk_g2s(uint32_t dst_smem, const void* src, uint32_t bytes,
                                         uint32_t bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
        ::"r"(dst_smem), "l"(src), "r"(bytes), "r"(bar)
        : "memory");
}

// ---- TMEM -----------------------------------------------------------------------------------
// One full warp allocates `ncols` (power of two >= 32) columns; base address lands in smem.
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem),
                 "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
                 : "memory");
}

// ---- descriptors ----------------------------------------------------------------------------
// Shared-memory matrix descriptor, K-major, SWIZZLE_NONE ("interleave") canonical layout:
//   element (row r, k) lives at  start + (r % 8) * 16 B + (r / 8) * SBO + (k / 8) * LBO + (k % 8) * 2 B
// i.e. 8x(16 B) core matrices; SBO strides 8-row groups, LBO strides the two 8-element K chunks
// of one K=16 MMA.  With SBO = 128 B every row sits at a uniform 16 B pitch, so a descriptor can
// start at ANY row: that is what makes the shifted 3x3 taps zero-copy (DESIGN.md §6).
// Bits: [0,14) addr>>4 | [16,30) LBO>>4 | [32,46) SBO>>4 | [46,48) version=1 | [61,64) layout=0.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr, uint32_t lbo_bytes,
                                                   uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
    d |= 1ull << 46;
    return d;
}

// The same descriptor split into its halves for issue loops: shared-memory addresses are below 256 KB,
// so (addr >> 4) needs no mask, and consecutive K steps differ by a constant in the low word only -
// one integer add per descriptor instead of a shift and two logic ops on the (narrow) uniform datapath.
__device__ __forceinline__ uint32_t smem_desc_lo(uint32_t smem_addr, uint32_t lbo_bytes) {
    // matrix-descriptor-encode(x) = (x & 0x3FFFF) >> 4: in a cluster launch (trunk_pair_kernel) the shared-window address
    // of a CTA of rank > 0 carries its rank above bit 18, which must not spill into the LBO field
    return ((smem_addr & 0x3FFFFu) >> 4) | ((lbo_bytes >> 4) << 16);
}
__device__ __forceinline__ uint64_t smem_desc_from(uint32_t lo, uint32_t sbo_bytes) {
    return ((uint64_t)(((sbo_bytes >> 4) & 0x3FFFu) | (1u << 14)) << 32) | lo;
}

// Instruction descriptor for kind::f16, A/B = bf16 K-major, D = fp32.
//   [4,6) c_format=1 (f32) | [7,10) a_format=1 (bf16) | [10,13) b_format=1 | [15] a_major=0 (K)
//   [16] b_major=0 (K) | [17,23) N>>3 | [24,29) M>>4
__host__ __device__ constexpr uint32_t make_idesc_bf16_f32(int m, int n) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) |
           ((uint32_t)(m >> 4) << 24);
}

// D[tmem] (+)= A[smem] * B[smem]^T, issued by ONE thread (SASS: UTCHMMA).
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                          uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// Same with the A operand in tensor memory (lane = row, 32-bit column = two consecutive K elements).
__device__ __forceinline__ void umma_bf16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                             uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// registers -> TMEM: this thread's lane (quadrant = warp_id % 4), 8 consecutive 32-bit columns
__device__ __forceinline__ void tmem_st_32x32b_x8(uint32_t taddr, const uint32_t (&v)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr),
                 "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
                 : "memory");
}
// Warpgroup register reallocation: every warp of a group of 4 consecutive warps executes it.
template <int N>
__device__ __forceinline__ void setmaxnreg_inc() {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N));
}
template <int N>
__device__ __forceinline__ void setmaxnreg_dec() {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N));
}
// Arrive on an mbarrier once all previously issued MMAs of this thread have completed
// (implies tcgen05.fence::before_thread_sync).
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar)
                 : "memory");
}

// TMEM -> registers: the warp's 32 lanes (quadrant = warp_id % 4) x 32 consecutive columns.
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
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
// TMEM -> registers, 16 lanes x 32 columns in the mma C-fragment layout (shape .16x256b, x4):
// for column group g (8 columns each), thread t holds
//   v[4g+0], v[4g+1] = (lane t/4    , columns 8g + 2(t%4), +1)
//   v[4g+2], v[4g+3] = (lane t/4 + 8, columns 8g + 2(t%4), +1)
// which is exactly the fragment stmatrix / ldmatrix (.trans) move to and from shared memory.
__device__ __forceinline__ void tmem_ld_16x256b_x4(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.16x256b.x4.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
          "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
          "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}
// Four 8x8 b16 matrices, transposed on the way: memory row i of matrix k is the 16-byte record
// at the address supplied by lane 8k+i and receives column i of the register fragment.
__device__ __forceinline__ void stmatrix_x4_trans(uint32_t addr, uint32_t r0, uint32_t r1, uint32_t r2,
                                                  uint32_t r3) {
    asm volatile("stmatrix.sync.aligned.m8n8.x4.trans.shared.b16 [%0], {%1, %2, %3, %4};" ::"r"(addr),
                 "r"(r0), "r"(r1), "r"(r2), "r"(r3)
                 : "memory");
}
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2,
                                                  uint32_t& r3) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3)
                 : "r"(addr)
                 : "memory");
}
// ReLU fused into the conversion: negative inputs (and NaN) become +0.
__device__ __forceinline__ uint32_t pack_relu_bf16x2(float lo, float hi) {
    uint32_t d;
    asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    return d;
}
// Packed fp32 pair arithmetic (SASS FADD2): one issue slot for two adds.
__device__ __forceinline__ uint64_t pack_f32x2(float lo, float hi) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ uint64_t pack_u32x2(uint32_t lo, uint32_t hi) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(lo), "r"(hi));
    return r;
}
__device__ __forceinline__ uint64_t add_f32x2(uint64_t a, uint64_t b) {
    uint64_t r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
// cvt.rn.relu.bf16x2 of a packed pair (low half of the result = low element)
__device__ __forceinline__ uint32_t pack_relu_bf16x2(uint64_t v) {
    uint32_t d;
    asm("{\n\t.reg .f32 lo, hi;\n\t"
        "mov.b64 {lo, hi}, %1;\n\t"
        "cvt.rn.relu.bf16x2.f32 %0, hi, lo;\n\t}"
        : "=r"(d)
        : "l"(v));
    return d;
}
__device__ __forceinline__ void tmem_ld_wait() {
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// ---- CTA pair (cta_group::2) and cluster primitives --------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cta address of this CTA -> shared::cluster address of the same offset in CTA `rank`
__device__ __forceinline__ uint32_t map_to_cta(uint32_t smem_addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(rank));
    return r;
}
// Remote arrives carry the default .release.cta semantics on purpose: a cluster-scope release or
// acquire compiles to MEMBAR.ALL.GPU / CCTL.IVALL (hundreds of cycles, measured) and everything these
// barriers order is either written by the async proxy (bulk copies, tcgen05.commit) or was fenced
// with fence.proxy.async before a local arrive that the relaying thread has already observed.
__device__ __forceinline__ void mbar_arrive_remote(uint32_t cluster_bar) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_bar) : "memory");
}
// remote arrive that also raises the destination barrier's expected transaction count (the bytes a
// following bulk_s2peer will complete on it)
__device__ __forceinline__ void mbar_arrive_expect_tx_remote(uint32_t cluster_bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cluster.b64 _, [%0], %1;" ::"r"(cluster_bar),
                 "r"(bytes)
                 : "memory");
}
// shared::cta -> peer's shared memory through the bulk-copy engine; completes (bytes) on an mbarrier
// that lives in the DESTINATION CTA.  Both destination and barrier are shared::cluster addresses.
__device__ __forceinline__ void bulk_s2peer(uint32_t dst_cluster, uint32_t src_smem, uint32_t bytes,
                                            uint32_t bar_cluster) {
    asm volatile(
        "cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
        ::"r"(dst_cluster), "r"(src_smem), "r"(bytes), "r"(bar_cluster)
        : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem of both CTAs] (+)= A * B^T with M = 256 split over the pair (each CTA's A rows come from its
// own shared memory at the descriptor's offset) and N split likewise; issued by the leader CTA only.
__device__ __forceinline__ void umma_bf16_pair(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                               uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit_pair(uint32_t bar, uint16_t cta_mask) {
    asm volatile(
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
        ::"r"(bar), "h"(cta_mask)
        : "memory");
}
__device__ __forceinline__ void tmem_st_wait() {
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ uint16_t f32_to_bf16_bits(float f) {
    return __bfloat16_as_ushort(__float2bfloat16_rn(f));
}

}  // namespace nsb
