// trunk_tmem.cu — the 128-channel trunk kernels that feed the weights through tensor memory (sm_100a).  Same contract
// as trunk_fused.cu (reference src/infer/trt.cc:256-261).
//
// The one-CTA-per-SM kernels leave the tensor pipe idle whenever their CTA is not issuing MMAs: accumulator hand-off,
// epilogue, feature expansion, heads, value MLP, decode - about 30 % of a 128-channel launch.  Overlapping the epilogue
// with the next layer inside one CTA did not pay (DESIGN.md §6.1).  Two independent CTAs on the same SM overlap
// everything for free: while one is in an epilogue (or its prologue / tail) the other one's MMAs own the tensor pipe.
// What made that impossible was the footprint of a CTA: 229 KB of shared memory (activations + a 96 KB weight ring),
// all 512 TMEM columns, 64 K registers.  Feeding the weights through tensor memory (trunk_ts.cu: L2 -> registers ->
// tcgen05.st -> A operand of tcgen05.mma) removes the ring, and the rest is diet.  A group of 2 positions (N = 192:
// the weight bytes per FLOP that L2 can sustain) owns two activation buffers and one accumulator; a CTA holds NGRP
// groups and ONE weight stream.
//
// trunk_duo_kernel, NGRP = 1, built for TWO CTAs PER SM:
//   shared memory 108 KB : two activation buffers; feature staging and the logits scratch alias
//                          buffer A while it is dead and are re-zeroed afterwards
//   tensor memory 256 col: one accumulator (192) + a 4-stage ring of 2 K steps (64)
//   registers     30 K   : 384 threads; setmaxnreg: 4 producer warps 72, 4 epilogue warps 128, MMA warp 40
//
// trunk_quad_kernel, NGRP = 2, one CTA per SM.  Two co-resident duo CTAs each stream the whole weight stream (6.1 MB
// per pass) through L2 -> L1 -> registers -> tcgen05.st for their own 2 positions, so every weight byte crosses that
// path twice per 4 positions of an SM, and the shared L1TEX holds the pair at ~69 % tensor duty (DESIGN.md §9).  Here
// every K = 16 weight step is stored into tensor memory once and issued as two N = 192 MMAs, one per group, so the
// weight path carries half the bytes per evaluation and each round of the MMA issue protocol (wait, fence, elect,
// commit) covers twice as many MMAs.
//   shared memory 222 KB : 2 groups x 2 activation buffers; feature staging and the logits scratch of a group alias
//                          its buffer A while it is dead and are re-zeroed afterwards
//   tensor memory 512 col: two accumulators (2 x 192) + an 8-stage ring of 2 K steps (128)
//   registers     64 K   : 512 threads; setmaxnreg: 4 producer warps 72, 8 epilogue warps 168, MMA warpgroup 40
//
// Each accumulator receives the same MMA sequence (layer, K block, tap, step; same accumulate flags) at either NGRP,
// so the two kernels' results are bit-identical.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "trunk_common.cuh"

namespace nsb {

namespace {

template <int NGRP_>
struct TmemGeom {
    static constexpr int C = 128;
    static constexpr int KCH = C / 8;
    static constexpr int NGRP = NGRP_;           // position groups per CTA
    static constexpr int NPOS = 2;               // positions per group
    static constexpr int QPOS = NGRP * NPOS;     // positions per CTA
    static constexpr int NCOLS = NPOS * 96;      // accumulator columns of a group
    static constexpr int GUARD = 12;
    static constexpr int SPITCH = (GUARD + NCOLS + 11) | 1;
    static constexpr int BUF_BYTES = ((KCH * SPITCH * 16 + 127) / 128) * 128;
    static constexpr int KC64 = C / 64;
    static constexpr int TMEM_COLS = 256 * NGRP;
    static constexpr int A_COL0 = NGRP * NCOLS;  // the ring follows the accumulators
    static constexpr int A_STAGES = 4 * NGRP;    // ring stages of 2 K steps = 16 columns each
    static constexpr int A_STAGE_COLS = 16;
    // warps 0-3 producers, 4 .. 4 + 4 NGRP - 1 epilogue, then the MMA warpgroup (its first warp issues); setmaxnreg
    // acts on whole warpgroups
    static constexpr int THREADS = 128 * (2 + NGRP);
    static constexpr int GRP_THREADS = 128;      // epilogue threads of a group: warps 4-7 = group 0, 8-11 = group 1
    static constexpr int EPI_WARPS = GRP_THREADS / 32;
    static constexpr int MMA_WARP = 4 + 4 * NGRP;
    static constexpr int MIN_BLOCKS = NGRP == 1 ? 2 : 1;  // CTAs per SM the footprint is built for
    static constexpr int PRODUCER_REGS = 72, EPI_REGS = NGRP == 1 ? 128 : 168, MMA_REGS = 40;  // setmaxnreg
    static constexpr int NBARS = 2 * A_STAGES + 2;  // a_full[], a_empty[], act, acc
    static constexpr int SCRATCH_BYTES = ((NPOS * kPolicySize * 4 + 15) / 16) * 16;
    static constexpr int FEAT_BYTES = NPOS * kMaxInChannels * 16;
    static constexpr int VBUF_BYTES = ((NPOS * 81 * 4 + 15) / 16) * 16;
    static constexpr int RED_BYTES = ((EPI_WARPS * NPOS * 2 * 4 + NPOS * 2 * 4 + 15) / 16) * 16;
    // dynamic shared memory map: group g owns buffers A (2g) and B (2g + 1), a vbuf and a red array.  The feature
    // staging (prologue) and the logits scratch (tail) of a group alias the front of its buffer A, dead in both phases.
    static constexpr int GRP_BYTES = 2 * BUF_BYTES;
    static constexpr int OFF_BUF_A = 0;
    static constexpr int OFF_BUF_B = BUF_BYTES;
    static constexpr int OFF_VBUF = NGRP * GRP_BYTES;
    static constexpr int OFF_RED = OFF_VBUF + NGRP * VBUF_BYTES;
    static constexpr int OFF_BARS = OFF_RED + NGRP * RED_BYTES;
    static constexpr int SMEM_BYTES = OFF_BARS + NBARS * 8 + 16 + 128;
    static_assert(BUF_BYTES == 55040, "each group has the duo kernel's activation layout");
    static_assert(NGRP > 1 || (OFF_VBUF == 110080 && OFF_RED == 110736 && OFF_BARS == 110816 && SMEM_BYTES == 111040),
                  "one group keeps the duo kernel's shared memory map");
    static_assert(SCRATCH_BYTES <= BUF_BYTES && FEAT_BYTES <= BUF_BYTES, "aliases fit into buffer A");
    static_assert(A_COL0 + A_STAGES * A_STAGE_COLS == TMEM_COLS, "accumulators + the ring fill the allocation");
    static_assert(MIN_BLOCKS * (SMEM_BYTES + 1024) <= 233472, "MIN_BLOCKS CTAs per SM");
    static_assert(128 * (PRODUCER_REGS + NGRP * EPI_REGS + MMA_REGS) <= 65536 / MIN_BLOCKS,
                  "re-balanced registers of MIN_BLOCKS CTAs fit the SM");
};

template <int NGRP>
__device__ __forceinline__ void trunk_tmem_body(const DeviceNet& net, const EvalArgs& a) {
    using G = TmemGeom<NGRP>;
    constexpr int C = G::C;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 127) & ~(uintptr_t)127);
    const uint32_t sbase = smem_u32(smem);
    const uint32_t bars = sbase + G::OFF_BARS;
    auto bar_afull = [&](int s) { return bars + 8u * s; };
    auto bar_aempty = [&](int s) { return bars + 8u * (G::A_STAGES + s); };
    const uint32_t bar_act = bars + 8u * (2 * G::A_STAGES);
    const uint32_t bar_acc = bars + 8u * (2 * G::A_STAGES + 1);
    volatile uint32_t* tmem_holder = reinterpret_cast<volatile uint32_t*>(smem + G::OFF_BARS + 8 * G::NBARS);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_eff = eval_count(a);
    const int units = (n_eff + G::QPOS - 1) / G::QPOS;
    const int my_passes =
        (int)blockIdx.x < units ? (units - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
    const int NL = net.num_layers;
    const bool stamp = eval_timeline(a) && blockIdx.x == 0;  // diagnostics: tools/timeline.py
    // diagnostics: where and when every CTA ran (co-residency of the two duo CTAs of an SM: tools/residency.py)
    unsigned long long* cta_rec = (eval_timeline(a) && blockIdx.x < 1024) ? eval_timeline(a) + 4 * NL + 16 + 3 * blockIdx.x : nullptr;
    if (cta_rec && threadIdx.x == 0) {
        unsigned smid;
        unsigned long long t;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        cta_rec[0] = smid;
        cta_rec[1] = t;
    }

    // ---- one-time setup ---------------------------------------------------------------------
    for (int i = threadIdx.x; i < G::NGRP * G::GRP_BYTES / 16; i += G::THREADS)
        reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
    if (threadIdx.x == 0) {
        for (int s = 0; s < G::A_STAGES; ++s) {
            mbar_init(bar_afull(s), 4);   // one arrival per producer warp
            mbar_init(bar_aempty(s), 1);  // tcgen05.commit of the MMAs (all groups) that read the stage
        }
        mbar_init(bar_act, G::NGRP * G::EPI_WARPS);
        mbar_init(bar_acc, 1);
        fence_mbar_init();
    }
    fence_proxy_async_smem();
    if (warp == G::MMA_WARP) tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_holder)), G::TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_holder;

    if (warp < 4) {
        // ===== weight producers: L2 -> registers -> tensor memory ================================
        // Thread = accumulator row = TMEM lane; the stream holds 128 rows x 32 B per K = 16 step
        // (weights.cc, pack_weights_ts).  A ring stage is two steps; three register stages rotate.
        setmaxnreg_dec<G::PRODUCER_REGS>();
        const int row = threadIdx.x;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(warp * 32) << 16) + G::A_COL0;
        const int steps_per_pass = net.stages_per_pass;  // K = 16 steps (always even per (K block, tap))
        uint32_t slot = 0, phase = 0;
        auto load_stage = [&](uint4 (&dst)[4], const uint4* s) {
            dst[0] = __ldg(s);
            dst[1] = __ldg(s + 1);
            dst[2] = __ldg(s + 256);
            dst[3] = __ldg(s + 257);
        };
        auto store_stage = [&](const uint4 (&buf)[4]) {
            mbar_wait(bar_aempty(slot), phase ^ 1u);
            tc_fence_after();
            asm volatile(
                "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
                "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
                ::"r"(lane_addr + slot * G::A_STAGE_COLS), "r"(buf[0].x), "r"(buf[0].y), "r"(buf[0].z), "r"(buf[0].w),
                  "r"(buf[1].x), "r"(buf[1].y), "r"(buf[1].z), "r"(buf[1].w), "r"(buf[2].x), "r"(buf[2].y), "r"(buf[2].z),
                  "r"(buf[2].w), "r"(buf[3].x), "r"(buf[3].y), "r"(buf[3].z), "r"(buf[3].w)
                : "memory");
            tmem_st_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_afull(slot));
            if (++slot == G::A_STAGES) { slot = 0; phase ^= 1u; }
        };
        const int stages_per_pass = steps_per_pass / 2;
        for (int p = 0; p < my_passes; ++p) {
            const uint4* src = reinterpret_cast<const uint4*>(net.tiles) + (size_t)row * 2;
            uint4 b0[4], b1[4], b2[4];
            int ld = 0, st = 0;  // stage cursors: stage s starts at src + s * 512 uint4
            if (ld < stages_per_pass) { load_stage(b0, src + (size_t)ld * 512); ++ld; }
            if (ld < stages_per_pass) { load_stage(b1, src + (size_t)ld * 512); ++ld; }
            if (ld < stages_per_pass) { load_stage(b2, src + (size_t)ld * 512); ++ld; }
            for (;;) {
                store_stage(b0); ++st;
                if (ld < stages_per_pass) { load_stage(b0, src + (size_t)ld * 512); ++ld; }
                if (st >= stages_per_pass) break;
                store_stage(b1); ++st;
                if (ld < stages_per_pass) { load_stage(b1, src + (size_t)ld * 512); ++ld; }
                if (st >= stages_per_pass) break;
                store_stage(b2); ++st;
                if (ld < stages_per_pass) { load_stage(b2, src + (size_t)ld * 512); ++ld; }
                if (st >= stages_per_pass) break;
            }
        }
    } else if (warp >= G::MMA_WARP) {
        setmaxnreg_dec<G::MMA_REGS>();
        if (warp == G::MMA_WARP) {
            // ===== MMA issuer: warp-uniform loop, one elected lane issues; per ring stage, the stage's K steps for
            //       group 0, then for group 1, ..., then one commit that frees the stage =========================
            constexpr uint32_t idesc = make_idesc_bf16_f32(128, G::NCOLS);
            constexpr uint32_t b_lbo = G::SPITCH * 16;
            uint32_t slot = 0, phase = 0, act_phase = 0;
            for (int p = 0; p < my_passes; ++p) {
                for (int L = 0; L < NL; ++L) {
                    mbar_wait(bar_act, act_phase);
                    act_phase ^= 1u;
                    tc_fence_after();
                    if (stamp && p == 0 && lane == 0) eval_timeline(a)[4 * L + 0] = clock64();
                    const bool head = (L == NL - 1);
                    const uint32_t in_buf = sbase + ((L & 1) ? G::OFF_BUF_A : G::OFF_BUF_B);  // group g at + g GRP_BYTES
                    const int ntaps = head ? 1 : 9;
                    for (int kc = 0; kc < G::KC64; ++kc) {
                        const int halves = block_steps(net, L, kc) / 2;  // ring stages per (K block, tap)
                        for (int tap = 0; tap < ntaps; ++tap) {
                            const int shift = head ? 0 : (tap / 3 - 1) * 10 + (tap % 3 - 1);
                            const uint32_t b_base = in_buf + (uint32_t)((kc * 8 * G::SPITCH + G::GUARD + shift) * 16);
                            if (halves == 2) {
                                // both ring stages of the tap in one round of the issue protocol (wait, fence,
                                // elect, commit, warp sync cost ~190 cycles a round): 4 NGRP MMAs per round
                                const uint32_t s0 = slot, s1 = (slot + 1) % G::A_STAGES;
                                const uint32_t ph1 = s1 == 0 ? phase ^ 1u : phase;
                                mbar_wait(bar_afull(s0), phase);
                                mbar_wait(bar_afull(s1), ph1);
                                tc_fence_after();
                                if (elect_one()) {
#pragma unroll
                                    for (int h = 0; h < 2; ++h) {
                                        const uint32_t a_base = tmem_base + G::A_COL0 + (h ? s1 : s0) * G::A_STAGE_COLS;
#pragma unroll
                                        for (int g = 0; g < G::NGRP; ++g) {
                                            const uint32_t b_lo = smem_desc_lo(b_base + g * G::GRP_BYTES, b_lbo);
#pragma unroll
                                            for (int k2 = 0; k2 < 2; ++k2) {
                                                const int k = 2 * h + k2;
                                                umma_bf16_ts(tmem_base + g * G::NCOLS, a_base + k2 * 8,
                                                             smem_desc_from(b_lo + (uint32_t)(2 * k * G::SPITCH), 128),
                                                             idesc, (uint32_t)((kc | tap | k) != 0));
                                            }
                                        }
                                        umma_commit(bar_aempty(h ? s1 : s0));
                                    }
                                }
                                __syncwarp();
                                slot = (slot + 2) % G::A_STAGES;
                                if (slot < 2) phase ^= 1u;
                                continue;
                            }
                            for (int h = 0; h < halves; ++h) {
                                mbar_wait(bar_afull(slot), phase);
                                tc_fence_after();
                                if (elect_one()) {
                                    const uint32_t a_base = tmem_base + G::A_COL0 + slot * G::A_STAGE_COLS;
#pragma unroll
                                    for (int g = 0; g < G::NGRP; ++g) {
                                        const uint32_t b_lo =
                                            smem_desc_lo(b_base + g * G::GRP_BYTES, b_lbo) + (uint32_t)(4 * h * G::SPITCH);
#pragma unroll
                                        for (int k2 = 0; k2 < 2; ++k2)
                                            umma_bf16_ts(tmem_base + g * G::NCOLS, a_base + k2 * 8,
                                                         smem_desc_from(b_lo + (uint32_t)(2 * k2 * G::SPITCH), 128),
                                                         idesc, (uint32_t)((kc | tap | h | k2) != 0));
                                    }
                                    umma_commit(bar_aempty(slot));
                                }
                                __syncwarp();
                                if (++slot == G::A_STAGES) { slot = 0; phase ^= 1u; }
                            }
                        }
                    }
                    if (elect_one()) umma_commit(bar_acc);
                    __syncwarp();
                    if (stamp && p == 0 && lane == 0) eval_timeline(a)[4 * L + 1] = clock64();
                }
            }
        }
    } else {
        // ===== expansion + epilogues + heads: per group 4 warps, one per TMEM lane quadrant, both positions =====
        setmaxnreg_inc<G::EPI_REGS>();
        // a compile-time 0 for one group: the named barrier id stays an immediate
        const int g = NGRP == 1 ? 0 : (warp - 4) >> 2;          // position group
        const int et = threadIdx.x - 128 - g * G::GRP_THREADS;  // 0..127 within the group
        const int q = warp & 3;                                 // TMEM lane quadrant
        const uint32_t bar = kEpiBar + g;                       // named barrier of the group's 4 warps
        uint8_t* gsmem = smem + g * G::GRP_BYTES;
        const uint32_t bufA = sbase + g * G::GRP_BYTES + G::OFF_BUF_A, bufB = sbase + g * G::GRP_BYTES + G::OFF_BUF_B;
        float* scratch = reinterpret_cast<float*>(gsmem + G::OFF_BUF_A);
        uint4* featS = reinterpret_cast<uint4*>(gsmem + G::OFF_BUF_A);
        float* vbuf = reinterpret_cast<float*>(smem + G::OFF_VBUF + g * G::VBUF_BYTES);
        float* red = reinterpret_cast<float*>(smem + G::OFF_RED + g * G::RED_BYTES);
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + g * G::NCOLS;
        const bool stamper = stamp && g == 0 && et == 0;
        EpilogueMask<3> mask0, mask1;
        mask0.init(0, lane);
        mask1.init(96, lane);
        uint32_t acc_phase = 0;
        for (int p = 0; p < my_passes; ++p) {
            const int b0 = ((int)blockIdx.x + p * (int)gridDim.x) * G::QPOS + g * G::NPOS;

            // -- stage 2 of feature extraction, straight into the stem's B operand (bufB); the bit
            //    strings are staged in the (dead) front of buffer A, which is zeroed again afterwards
            expand_features<G::NPOS, G::SPITCH, G::GUARD, G::GRP_THREADS>(net, a, n_eff, b0, featS, gsmem + G::OFF_BUF_B, et, nullptr, bar);
            named_bar_sync(bar, G::GRP_THREADS);
            for (int i = et; i < G::FEAT_BYTES / 16; i += G::GRP_THREADS) featS[i] = make_uint4(0, 0, 0, 0);
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_act);

            // -- conv layers: TMEM -> +bias (+skip) -> ReLU -> bf16 -> next layer's B operand ----
            for (int L = 0; L < NL - 1; ++L) {
                float bias[4];  // accumulator row 32q + 16lb + 8h + lane/4 = channel 64lb + 16q + 8h + lane/4
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    bias[k] = __ldg(net.bias + (size_t)L * C + 64 * (k >> 1) + 16 * q + 8 * (k & 1) + (lane >> 2));
                mbar_wait(bar_acc, acc_phase);
                acc_phase ^= 1u;
                tc_fence_after();
                if (stamper && p == 0) eval_timeline(a)[4 * L + 2] = clock64();
                const uint32_t out_buf = ((L & 1) ? bufB : bufA) + G::GUARD * 16;
                const bool residual = (L >= 2) && ((L & 1) == 0);
#pragma unroll
                for (int part = 0; part < 2; ++part)
#pragma unroll
                    for (int lb = 0; lb < 2; ++lb) {
                        if (residual)
                            epilogue_half<3, true, 8>(lb, taddr + 96 * part, out_buf, G::SPITCH * 16, 2 * q, 96 * part, bias,
                                                      part ? mask1 : mask0, lane);
                        else
                            epilogue_half<3, false, 8>(lb, taddr + 96 * part, out_buf, G::SPITCH * 16, 2 * q, 96 * part, bias,
                                                       part ? mask1 : mask0, lane);
                    }
                tc_fence_before();
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_act);
                if (stamper && p == 0) eval_timeline(a)[4 * L + 3] = clock64();
            }

            // -- heads: row 32*(h/7) + h%7 of the accumulator holds head channel h
            const int hp = 7 * q + lane;
            const float hbias = lane < 7 ? __ldg(net.bias + (size_t)(NL - 1) * C + hp) : 0.f;
            mbar_wait(bar_acc, acc_phase);
            acc_phase ^= 1u;
            tc_fence_after();
            // the head input (buffer A) is dead now: its front becomes the logits scratch
            head_read<0>(taddr, hbias, hp, scratch, vbuf, lane);
            head_read<96>(taddr + 96, hbias, hp, scratch, vbuf, lane);
            tc_fence_before();
            named_bar_sync(bar, G::GRP_THREADS);
            heads_tail_small<G::NPOS, G::GRP_THREADS>(net, a, n_eff, b0, scratch, vbuf, red, et, bar);
            if (p + 1 < my_passes) {  // the scratch overwrote guard / padding slots of buffer A: zero them again
                for (int i = et; i < G::SCRATCH_BYTES / 16; i += G::GRP_THREADS)
                    reinterpret_cast<uint4*>(scratch)[i] = make_uint4(0, 0, 0, 0);
                named_bar_sync(bar, G::GRP_THREADS);
            }
        }
    }

    // ---- teardown -------------------------------------------------------------------------------
    tc_fence_before();
    __syncthreads();
    if (cta_rec && threadIdx.x == 0) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        cta_rec[2] = t;
    }
    if (warp == G::MMA_WARP) {
        __syncwarp();
        tmem_dealloc(tmem_base, G::TMEM_COLS);
    }
}

// Not templates: tools and tests find the kernels by these names.
__global__ void __launch_bounds__(TmemGeom<1>::THREADS, TmemGeom<1>::MIN_BLOCKS)
    trunk_duo_kernel(const DeviceNet net, const EvalArgs a) { trunk_tmem_body<1>(net, a); }
__global__ void __launch_bounds__(TmemGeom<2>::THREADS, TmemGeom<2>::MIN_BLOCKS)
    trunk_quad_kernel(const DeviceNet net, const EvalArgs a) { trunk_tmem_body<2>(net, a); }

template <int NGRP>
constexpr auto tmem_kernel = NGRP == 1 ? trunk_duo_kernel : trunk_quad_kernel;

template <int NGRP>
int tmem_prepare(int* ctas_per_sm) {
    using G = TmemGeom<NGRP>;
    cudaError_t e = cudaFuncSetAttribute(tmem_kernel<NGRP>, cudaFuncAttributeMaxDynamicSharedMemorySize, G::SMEM_BYTES);
    if (e == cudaSuccess)
        e = cudaFuncSetAttribute(tmem_kernel<NGRP>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    int nb = 0;
    if (e == cudaSuccess)
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, tmem_kernel<NGRP>, G::THREADS, G::SMEM_BYTES);
    if (e != cudaSuccess || nb < 1) {
        set_error("trunk %s: cannot configure the kernel: %s (is this an sm_100a device?)", NGRP == 1 ? "duo" : "quad",
                  cudaGetErrorString(e));
        return NSB_ERR_NO_DEVICE;
    }
    // The occupancy calculator answers 1 for the duo kernel, the hardware co-schedules 2 (tools/residency.py: 296 CTAs
    // on 148 SMs, lifetimes overlapping 99 %): the footprint is built for two - 2 x (111 KB + 1 KB) of shared memory,
    // 2 x 256 TMEM columns, 2 x 30 K registers (static_asserts in TmemGeom).  An oversized grid would only cost a
    // second wave, an undersized one halves the kernel's reason to exist.
    if (ctas_per_sm) *ctas_per_sm = nb < G::MIN_BLOCKS ? G::MIN_BLOCKS : nb;
    return 0;
}

template <int NGRP>
int tmem_launch(const DeviceNet& net, const EvalArgs& a, int num_sms, int ctas_per_sm, cudaStream_t s) {
    using G = TmemGeom<NGRP>;
    if (a.n <= 0) return 0;
    const int units = (a.n + G::QPOS - 1) / G::QPOS;
    const int cap = num_sms * (ctas_per_sm > 0 ? ctas_per_sm : 1);
    const int grid = units < cap ? units : cap;
    tmem_kernel<NGRP><<<grid, G::THREADS, G::SMEM_BYTES, s>>>(net, a);
    return 1;
}

}  // namespace

int trunk_duo_prepare(int* ctas_per_sm) { return tmem_prepare<1>(ctas_per_sm); }

int launch_trunk_duo(const DeviceNet& net, const EvalArgs& a, int num_sms, int ctas_per_sm, cudaStream_t s) {
    return tmem_launch<1>(net, a, num_sms, ctas_per_sm, s);
}

int trunk_quad_prepare() { return tmem_prepare<2>(nullptr); }

int launch_trunk_quad(const DeviceNet& net, const EvalArgs& a, int num_sms, cudaStream_t s) {
    return tmem_launch<2>(net, a, num_sms, 1, s);
}

}  // namespace nsb
