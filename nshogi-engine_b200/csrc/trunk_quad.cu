// trunk_quad.cu — 128-channel trunk with FOUR positions per CTA and one CTA per SM (sm_100a).  Same contract as
// trunk_duo.cu (reference src/infer/trt.cc:256-261).
//
// Two co-resident trunk_duo_kernel CTAs each stream the whole weight stream (6.1 MB per pass) through
// L2 -> L1 -> registers -> tcgen05.st for their own 2 positions, so every weight byte crosses that path twice per
// 4 positions of an SM, and the shared L1TEX holds the pair at ~69 % tensor duty (DESIGN.md §9).  This kernel is the
// pair folded into one CTA: two groups of 2 positions, each with exactly the duo kernel's activation layout, and ONE
// weight stream.  Every K = 16 weight step is stored into tensor memory once and issued as two N = 192 MMAs, one per
// group, so the weight path carries half the bytes per evaluation and each round of the MMA issue protocol (wait,
// fence, elect, commit) covers twice as many MMAs.
//   shared memory 222 KB : 2 groups x 2 activation buffers of the duo kernel; feature staging and the logits scratch
//                          of a group alias its buffer A while it is dead and are re-zeroed afterwards
//   tensor memory 512 col: two accumulators (2 x 192) + an 8-stage ring of 2 K steps (128)
//   registers     64 K   : 512 threads; setmaxnreg: 4 producer warps 72, 8 epilogue warps 168, MMA warpgroup 40
// Each accumulator sees exactly the duo kernel's MMA sequence (layer, K block, tap, step; same accumulate flags), so
// the results are bit-identical to trunk_duo_kernel's.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "trunk_common.cuh"

namespace nsb {

namespace {

struct QuadGeom {
    static constexpr int C = 128;
    static constexpr int KCH = C / 8;
    static constexpr int NGRP = 2;               // position groups per CTA
    static constexpr int NPOS = 2;               // positions per group
    static constexpr int QPOS = NGRP * NPOS;     // positions per CTA
    static constexpr int NCOLS = NPOS * 96;      // accumulator columns of a group
    static constexpr int GUARD = 12;
    static constexpr int SPITCH = (GUARD + NCOLS + 11) | 1;
    static constexpr int BUF_BYTES = ((KCH * SPITCH * 16 + 127) / 128) * 128;
    static constexpr int KC64 = C / 64;
    static constexpr int TMEM_COLS = 512;
    static constexpr int A_COL0 = NGRP * NCOLS;  // 384
    static constexpr int A_STAGES = 8;           // ring stages of 2 K steps = 16 columns each
    static constexpr int A_STAGE_COLS = 16;
    static constexpr int THREADS = 512;          // warps 0-3 producers, 4-11 epilogue, 12 MMA (13-15 idle)
    static constexpr int GRP_THREADS = 128;      // epilogue threads of a group: warps 4-7 = group 0, 8-11 = group 1
    static constexpr int EPI_WARPS = GRP_THREADS / 32;
    static constexpr int MMA_WARP = 12;
    static constexpr int NBARS = 2 * A_STAGES + 2;  // a_full[], a_empty[], act, acc
    static constexpr int SCRATCH_BYTES = ((NPOS * kPolicySize * 4 + 15) / 16) * 16;
    static constexpr int FEAT_BYTES = NPOS * kMaxInChannels * 16;
    static constexpr int VBUF_BYTES = ((NPOS * 81 * 4 + 15) / 16) * 16;
    static constexpr int RED_BYTES = ((EPI_WARPS * NPOS * 2 * 4 + NPOS * 2 * 4 + 15) / 16) * 16;
    // dynamic shared memory map: group g owns buffers A (2g) and B (2g + 1), a vbuf and a red array
    static constexpr int GRP_BYTES = 2 * BUF_BYTES;
    static constexpr int OFF_BUF_A = 0;
    static constexpr int OFF_BUF_B = BUF_BYTES;
    static constexpr int OFF_VBUF = NGRP * GRP_BYTES;
    static constexpr int OFF_RED = OFF_VBUF + NGRP * VBUF_BYTES;
    static constexpr int OFF_BARS = OFF_RED + NGRP * RED_BYTES;
    static constexpr int SMEM_BYTES = OFF_BARS + NBARS * 8 + 16 + 128;
    static_assert(BUF_BYTES == 55040, "each group has the duo kernel's activation layout");
    static_assert(SCRATCH_BYTES <= BUF_BYTES && FEAT_BYTES <= BUF_BYTES, "aliases fit into buffer A");
    static_assert(A_COL0 + A_STAGES * A_STAGE_COLS == TMEM_COLS, "two accumulators + the ring fill tensor memory");
    static_assert(SMEM_BYTES <= 232448, "one CTA per SM");
    static_assert(THREADS == 4 * 128, "setmaxnreg acts on whole warpgroups");
    static_assert(128 * 72 + 2 * 128 * 168 + 128 * 40 <= 65536, "re-balanced registers fit the SM");
};

__global__ void __launch_bounds__(QuadGeom::THREADS, 1) trunk_quad_kernel(const DeviceNet net, const EvalArgs a) {
    using G = QuadGeom;
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
    const int quads = (n_eff + G::QPOS - 1) / G::QPOS;
    const int my_passes =
        (int)blockIdx.x < quads ? (quads - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
    const int NL = net.num_layers;
    const bool stamp = eval_timeline(a) && blockIdx.x == 0;  // diagnostics: tools/timeline.py
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
            mbar_init(bar_aempty(s), 1);  // tcgen05.commit of the MMAs (both groups) that read the stage
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
        // ===== weight producers: L2 -> registers -> tensor memory (trunk_duo.cu's, with an 8-stage ring) ==========
        setmaxnreg_dec<72>();
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
        setmaxnreg_dec<40>();
        if (warp == G::MMA_WARP) {
            // ===== MMA issuer: per ring stage, the stage's K steps for group 0, then for group 1, one commit ===========
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
                    const uint32_t in_buf = sbase + ((L & 1) ? G::OFF_BUF_A : G::OFF_BUF_B);  // group 0; group 1 at + GRP_BYTES
                    const int ntaps = head ? 1 : 9;
                    for (int kc = 0; kc < G::KC64; ++kc) {
                        const int halves = block_steps(net, L, kc) / 2;  // ring stages per (K block, tap)
                        for (int tap = 0; tap < ntaps; ++tap) {
                            const int shift = head ? 0 : (tap / 3 - 1) * 10 + (tap % 3 - 1);
                            const uint32_t b_base = in_buf + (uint32_t)((kc * 8 * G::SPITCH + G::GUARD + shift) * 16);
                            if (halves == 2) {
                                // both ring stages of the tap in one round of the issue protocol: 8 MMAs per round
                                const uint32_t s0 = slot, s1 = (slot + 1) % G::A_STAGES;
                                const uint32_t ph1 = s1 == 0 ? phase ^ 1u : phase;
                                mbar_wait(bar_afull(s0), phase);
                                mbar_wait(bar_afull(s1), ph1);
                                tc_fence_after();
                                if (elect_one()) {
                                    const uint32_t b_lo0 = smem_desc_lo(b_base, b_lbo);
                                    const uint32_t b_lo1 = smem_desc_lo(b_base + G::GRP_BYTES, b_lbo);
#pragma unroll
                                    for (int h = 0; h < 2; ++h) {
                                        const uint32_t a_base = tmem_base + G::A_COL0 + (h ? s1 : s0) * G::A_STAGE_COLS;
#pragma unroll
                                        for (int g = 0; g < G::NGRP; ++g)
#pragma unroll
                                            for (int k2 = 0; k2 < 2; ++k2) {
                                                const int k = 2 * h + k2;
                                                umma_bf16_ts(tmem_base + g * G::NCOLS, a_base + k2 * 8,
                                                             smem_desc_from((g ? b_lo1 : b_lo0) + (uint32_t)(2 * k * G::SPITCH), 128),
                                                             idesc, (uint32_t)((kc | tap | k) != 0));
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
                                    const uint32_t b_lo0 = smem_desc_lo(b_base, b_lbo) + (uint32_t)(4 * h * G::SPITCH);
                                    const uint32_t b_lo1 = smem_desc_lo(b_base + G::GRP_BYTES, b_lbo) + (uint32_t)(4 * h * G::SPITCH);
#pragma unroll
                                    for (int g = 0; g < G::NGRP; ++g)
#pragma unroll
                                        for (int k2 = 0; k2 < 2; ++k2)
                                            umma_bf16_ts(tmem_base + g * G::NCOLS, a_base + k2 * 8,
                                                         smem_desc_from((g ? b_lo1 : b_lo0) + (uint32_t)(2 * k2 * G::SPITCH), 128),
                                                         idesc, (uint32_t)((kc | tap | h | k2) != 0));
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
        // ===== expansion + epilogues + heads: per group 4 warps, one per TMEM lane quadrant, as in trunk_duo.cu ======
        setmaxnreg_inc<168>();
        const int g = (warp - 4) >> 2;                           // position group
        const int et = threadIdx.x - 128 - g * G::GRP_THREADS;   // 0..127 within the group
        const int q = warp & 3;                                  // TMEM lane quadrant (== warp % 4)
        const uint32_t bar = kEpiBar + g;                        // named barrier of the group's 4 warps
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

}  // namespace

int trunk_quad_prepare() {
    cudaError_t e = cudaFuncSetAttribute(trunk_quad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, QuadGeom::SMEM_BYTES);
    int nb = 0;
    if (e == cudaSuccess)
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, trunk_quad_kernel, QuadGeom::THREADS, QuadGeom::SMEM_BYTES);
    if (e != cudaSuccess || nb < 1) {
        set_error("trunk quad: cannot configure the kernel: %s (is this an sm_100a device?)", cudaGetErrorString(e));
        return NSB_ERR_NO_DEVICE;
    }
    return 0;
}

int launch_trunk_quad(const DeviceNet& net, const EvalArgs& a, int num_sms, cudaStream_t s) {
    if (a.n <= 0) return 0;
    const int quads = (a.n + QuadGeom::QPOS - 1) / QuadGeom::QPOS;
    const int grid = quads < num_sms ? quads : num_sms;
    trunk_quad_kernel<<<grid, QuadGeom::THREADS, QuadGeom::SMEM_BYTES, s>>>(net, a);
    return 1;
}

}  // namespace nsb
