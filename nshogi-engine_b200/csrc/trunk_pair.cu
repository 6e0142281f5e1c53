// trunk_pair.cu — the position-stationary trunk for 192- and 256-channel nets on a CTA PAIR (sm_100a,
// tcgen05 cta_group::2).  Same contract as trunk_fused.cu (reference src/infer/trt.cc:256-261).
//
// Why a pair (DESIGN.md §6.2): with 256 channels one SM's shared memory holds the activations of
// only ONE position, i.e. an M128 x N96 MMA whose A operand (4 KB of weights per K = 16 step) is
// read from shared memory for 96 columns of work: measured 80-96 cycles against a 48-cycle tensor
// floor.  Two CTAs of a cluster instead issue ONE M256 x N192 MMA: CTA r supplies the weight rows of
// Cout half r (A, 4 KB) and the 96 slots of ITS position (half of B, 3 KB) and receives
// D[Cout half r][both positions] in its own TMEM - the same shared-memory bytes now feed twice the
// math (floor 96 cycles).  The price is an exchange after every layer: CTA r holds Cout half r of
// the OTHER position's output, which belongs in the peer's activation buffer.  The epilogue writes
// that part into an exchange buffer (24 KB at 256 channels) and the bulk-copy engine pushes it through DSMEM
// (cp.async.bulk.shared::cluster.shared::cta), completing on the peer's activation barrier.  The
// skip connection of the foreign half travels the other way, ahead of time, into the same buffer.
//
// Warp roles per CTA (384 threads): warp 0 = weight producer (its Cout half of every tile pair),
// warp 1 = MMA issuer in the leader CTA / ring-full relay in the peer, warp 2 = activation relay +
// skip push, warp 3 = exchange push, warps 4-11 = expansion, epilogues (each warp: 16 of my Cout rows, first for the peer's
// position - pushed at once - then for my own), heads, tail.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "trunk_common.cuh"

namespace nsb {

namespace {

constexpr uint32_t kPushBar = 2;  // named barrier: 8 epilogue warps arrive, the push warp (warp 3) waits

// 192 channels (PairGeom<192>): the weight tiles keep 128 rows, of which rows 96..127 are zero, so the
// MMA is unchanged (M = 256 with a third of each half's rows wasted) while the K side shrinks to 3 blocks
// of 64.  The epilogue warps of TMEM quadrant 3 then write nothing, but keep arriving on bar_act and
// kPushBar, so that every barrier count is the same at both widths.
template <int CW>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1)
trunk_pair_kernel(const DeviceNet net, const EvalArgs a) {
    using G = PairGeom<CW>;
    constexpr int C = G::C;
    extern __shared__ uint8_t smem_raw[];
    // the dynamic window starts at the same shared::cta offset in both CTAs, so this alignment
    // (and therefore every offset below) is identical in the pair - required by cta_group::2
    uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 127) & ~(uintptr_t)127);
    const uint32_t sbase = smem_u32(smem);
    const uint32_t bufA = sbase + G::OFF_BUF_A, bufB = sbase + G::OFF_BUF_B;
    const uint32_t xbuf = sbase + G::OFF_XBUF;
    const uint32_t ring = sbase + G::OFF_RING;
    float* scratch = reinterpret_cast<float*>(smem + G::OFF_XBUF);
    uint4* featS = reinterpret_cast<uint4*>(smem + G::OFF_FEAT);
    float* vbuf = reinterpret_cast<float*>(smem + G::OFF_VBUF);
    float* red = reinterpret_cast<float*>(smem + G::OFF_RED);
    const uint32_t bars = sbase + G::OFF_BARS;
    auto bar_full = [&](int s) { return bars + 8u * s; };
    auto bar_empty = [&](int s) { return bars + 8u * (G::NSTAGES + s); };
    const uint32_t bar_act = bars + 8u * (2 * G::NSTAGES);           // my activation buffer + TMEM are ready
    const uint32_t bar_acc = bars + 8u * (2 * G::NSTAGES + 1);       // accumulator complete (multicast commit)
    const uint32_t bar_peer_act = bars + 8u * (2 * G::NSTAGES + 2);  // leader only: the peer's bar_act fired
    const uint32_t bar_skip = bars + 8u * (2 * G::NSTAGES + 3);      // foreign skip rows landed in xbuf
    volatile uint32_t* tmem_holder = reinterpret_cast<volatile uint32_t*>(smem + G::OFF_BARS + 8 * G::NBARS);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank(), peer = rank ^ 1u;
    const int pair = (int)blockIdx.x >> 1, npairs = (int)gridDim.x >> 1;
    const int n_eff = eval_count(a);
    const int groups = (n_eff + 1) / 2;
    const int my_passes = pair < groups ? (groups - pair + npairs - 1) / npairs : 0;
    const int NL = net.num_layers;
    const bool stamp = eval_timeline(a) && blockIdx.x == 0;

    if (stamp && threadIdx.x == 128) eval_timeline(a)[4 * NL + 0] = clock64();
    // ---- one-time setup ---------------------------------------------------------------------
    for (int i = threadIdx.x; i < (2 * G::BUF_BYTES + G::XBUF_BYTES) / 16; i += kThreads)
        reinterpret_cast<uint4*>(smem + G::OFF_BUF_A)[i] = make_uint4(0, 0, 0, 0);
    if (threadIdx.x == 0) {
        for (int s = 0; s < G::NSTAGES; ++s) {
            mbar_init(bar_full(s), rank == 0 ? 2 : 1);  // leader: own producer + the peer's relay
            mbar_init(bar_empty(s), 1);
        }
        mbar_init(bar_act, kEpiWarps + 1);  // one arrival per local epilogue warp + the peer's push warp
        mbar_init(bar_acc, 1);
        mbar_init(bar_peer_act, 1);
        mbar_init(bar_skip, 1);
        fence_mbar_init();
    }
    fence_proxy_async_smem();
    if (warp == 1) tmem_alloc_pair(smem_u32(const_cast<uint32_t*>(tmem_holder)), G::TMEM_COLS);
    tc_fence_before();
    cluster_sync_all();  // barriers of both CTAs initialised before any remote arrive / bulk push
    tc_fence_after();
    const uint32_t tmem_base = *tmem_holder;
    if (stamp && threadIdx.x == 128) eval_timeline(a)[4 * NL + 1] = clock64();

    if (warp == 0) {
        // ===== weight producer: my Cout half of every conv tile pair, all head tiles ===========
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;
            const int conv_stages = (net.stages_per_pass - G::KC64) / 2;
            for (int p = 0; p < my_passes; ++p) {
                for (int s = 0; s < conv_stages + G::KC64; ++s) {
                    const int tile = s < conv_stages ? 2 * s + (int)rank : 2 * conv_stages + (s - conv_stages);
                    mbar_wait(bar_empty(stage), phase ^ 1u);
                    mbar_arrive_expect_tx(bar_full(stage), kStageBytes);
                    bulk_g2s(ring + stage * kStageBytes, net.tiles + (size_t)tile * kStageBytes, kStageBytes,
                             bar_full(stage));
                    if (++stage == G::NSTAGES) { stage = 0; phase ^= 1u; }
                }
            }
        }
    } else if (warp == 1 && rank != 0) {
        // ===== peer CTA: tell the leader when my half of a ring stage has landed ================
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;
            const int per_pass = (net.stages_per_pass - G::KC64) / 2 + G::KC64;
            for (int p = 0; p < my_passes; ++p)
                for (int s = 0; s < per_pass; ++s) {
                    mbar_wait(bar_full(stage), phase);
                    mbar_arrive_remote(map_to_cta(bar_full(stage), 0));
                    if (++stage == G::NSTAGES) { stage = 0; phase ^= 1u; }
                }
        }
    } else if (warp == 1) {
        // ===== leader CTA: MMA issuer for the pair (warp-uniform loop, one elected lane issues) ==
        constexpr uint32_t idesc = make_idesc_bf16_f32(256, G::NPAIR);
        constexpr uint32_t b_lbo = G::SPITCH * 16;
        uint32_t stage = 0, phase = 0, act_phase = 0;
        for (int p = 0; p < my_passes; ++p) {
            for (int L = 0; L < NL; ++L) {
                mbar_wait(bar_act, act_phase);
                mbar_wait(bar_peer_act, act_phase);
                act_phase ^= 1u;
                tc_fence_after();
                if (stamp && p == 0 && lane == 0) eval_timeline(a)[4 * L + 0] = clock64();
                const bool head = (L == NL - 1);
                const uint32_t in_buf = (L & 1) ? bufA : bufB;
                const int ntaps = head ? 1 : 9;
                const int kblocks = (L == 0) ? kStemCin / 64 : G::KC64;
                for (int tap = 0; tap < ntaps; ++tap) {
                    const int shift = head ? 0 : (tap / 3 - 1) * 10 + (tap % 3 - 1);
                    for (int kc = 0; kc < kblocks; ++kc) {
                        const uint32_t b_base = in_buf + (uint32_t)((kc * 8 * G::SPITCH + G::GUARD + shift) * 16);
                        mbar_wait(bar_full(stage), phase);
                        tc_fence_after();
                        const int ksteps = (L == 0 && kc == 1) ? net.stem_steps - 4 : 4;
                        if (elect_one()) {
                            const uint32_t a_lo = smem_desc_lo(ring + stage * kStageBytes, 2048);
                            const uint32_t b_lo = smem_desc_lo(b_base, b_lbo);
#pragma unroll
                            for (int k = 0; k < 4; ++k) {
                                if (k >= ksteps) break;
                                umma_bf16_pair(tmem_base, smem_desc_from(a_lo + k * (4096 >> 4), 128),
                                               smem_desc_from(b_lo + (uint32_t)(2 * k * G::SPITCH), 128), idesc,
                                               (uint32_t)((tap | kc | k) != 0));
                            }
                            umma_commit_pair(bar_empty(stage), 3);  // frees the stage in BOTH rings
                        }
                        __syncwarp();
                        if (++stage == G::NSTAGES) { stage = 0; phase ^= 1u; }
                    }
                }
                if (elect_one()) umma_commit_pair(bar_acc, 3);  // accumulators of layer L complete in both CTAs
                __syncwarp();
                if (stamp && p == 0 && lane == 0) eval_timeline(a)[4 * L + 1] = clock64();
            }
        }
    } else if (warp == 2) {
        // ===== activation relay + skip push ======================================================
        // Phase L of bar_act = "my input of layer L is complete and my accumulator is drained".
        // The peer forwards that to the leader's MMA warp.  Before a residual layer (conv2 of a
        // block) the block input x of the channels the PEER will produce is pushed into the peer's
        // exchange buffer; the peer's previous push out of that buffer has landed here, or the
        // phase could not have completed.
        uint32_t act_phase = 0;
        for (int p = 0; p < my_passes; ++p)
            for (int L = 0; L < NL; ++L) {
                mbar_wait(bar_act, act_phase);
                act_phase ^= 1u;
                if (rank != 0 && lane == 0) mbar_arrive_remote(map_to_cta(bar_peer_act, 0));
                const bool residual = (L >= 2) && ((L & 1) == 0) && (L < NL - 1);
                if (residual) {
                    const uint32_t x_buf = bufA;  // == this layer's output buffer (updated in place)
                    const uint32_t dst_bar = map_to_cta(bar_skip, peer);
                    if (lane == 0) mbar_arrive_expect_tx_remote(dst_bar, G::XCH * G::XROW);
                    __syncwarp();
                    if (lane < G::XCH)
                        bulk_s2peer(map_to_cta(xbuf + lane * G::XPITCH, peer),
                                    x_buf + (uint32_t)(((G::XCH * peer + lane) * G::SPITCH + G::GUARD) * 16),
                                    G::XROW, dst_bar);
                }
                __syncwarp();
            }
    } else if (warp == 3) {
        // ===== push warp: the exchange buffer -> the peer's activation buffer, once per conv layer =====
        // The epilogue warps write the peer position's rows first and arrive on kPushBar without
        // waiting; this warp then issues the XCH bulk copies (one lane each: a copy costs its issuing
        // thread ~290 cycles, tools/bulk_probe.py) while they go on with their own position.
        for (int p = 0; p < my_passes; ++p)
            for (int L = 0; L < NL - 1; ++L) {
                named_bar_sync(kPushBar, kEpiThreads + 32);
                const uint32_t out_base = (L & 1) ? bufB : bufA;
                const uint32_t dst_bar = map_to_cta(bar_act, peer);
                if (lane == 0) mbar_arrive_expect_tx_remote(dst_bar, G::XCH * G::XROW);
                __syncwarp();
                if (lane < G::XCH)
                    bulk_s2peer(map_to_cta(out_base + (uint32_t)(((G::XCH * rank + lane) * G::SPITCH + G::GUARD) * 16), peer),
                                xbuf + lane * G::XPITCH, G::XROW, dst_bar);
                __syncwarp();
            }
    } else if (warp >= 4) {
        // ===== expansion + epilogues + heads =====================================================
        const int et = threadIdx.x - 128;  // 0..255
        const int ew = warp - 4;           // 0..7
        const int q = ew & 3;              // TMEM lane quadrant (== warp % 4): 32 of my C/2 Cout
        const int lbw = ew >> 2;           // the 16-lane block of that quadrant this warp owns (both positions)
        const bool writer = q < G::QUADS;  // quadrant 3 holds no real Cout rows at 192 channels
        if (stamp && et == 0) eval_timeline(a)[4 * NL + 11] = clock64();
        EpilogueMask<3> realmask;
        realmask.init(0, lane);
        uint32_t acc_phase = 0, skip_phase = 0;
        for (int p = 0; p < my_passes; ++p) {
            const int b0 = (pair + p * npairs) * 2 + (int)rank;  // my position

            // -- stage 2 of feature extraction, straight into the stem's B operand (bufB) --------
            unsigned long long* tl = (stamp && p == 0 && et == 0) ? eval_timeline(a) + 4 * NL : nullptr;
            if (tl) tl[8] = clock64();
            expand_features<1, G::SPITCH, G::GUARD>(net, a, n_eff, b0, featS, smem + G::OFF_BUF_B, et, tl);
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_act);
            if (et == 0) mbar_arrive_remote(map_to_cta(bar_act, peer));  // nothing to exchange for the stem input
            if (tl) tl[2] = clock64();

            // -- conv layers: TMEM -> +bias (+skip) -> ReLU -> bf16 -> next layer's B operand ----
            for (int L = 0; L < NL - 1; ++L) {
                float bias[4];
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    bias[k] = writer ? __ldg(net.bias + (size_t)L * C + rank * (C / 2) + q * 32 + 8 * k + (lane >> 2)) : 0.f;
                mbar_wait(bar_acc, acc_phase);
                acc_phase ^= 1u;
                tc_fence_after();
                if (stamp && p == 0 && et == 0) eval_timeline(a)[4 * L + 2] = clock64();
                const uint32_t out_base = (L & 1) ? bufB : bufA;
                const bool residual = (L >= 2) && ((L & 1) == 0);
                const uint32_t tq = tmem_base + ((uint32_t)(q * 32) << 16);
                // First the PEER's position: its rows go through the exchange buffer and are pushed into
                // the peer's activation buffer the moment this warp's two chunks are written, so that the
                // DSMEM transfer and the barrier relay to the leader run under the second half below.
                if (residual) {  // the peer's x rows for my channels, pushed during the MMA phase
                    mbar_wait(bar_skip, skip_phase);
                    skip_phase ^= 1u;
                }
                if (writer) {
                    if (residual)
                        epilogue_half<3, true>(lbw, tq + peer * G::NCOLS, xbuf, G::XPITCH, q * 4, 0, bias, realmask, lane);
                    else
                        epilogue_half<3, false>(lbw, tq + peer * G::NCOLS, xbuf, G::XPITCH, q * 4, 0, bias, realmask, lane);
                }
                fence_proxy_async_smem();
                named_bar_arrive(kPushBar, kEpiThreads + 32);  // hand the exchange buffer to the push warp, do not wait
                // then my own position, in place in my activation buffer
                if (writer) {
                    const uint32_t out_buf = out_base + G::GUARD * 16;
                    const int chunk0 = (int)rank * G::XCH + q * 4;
                    if (residual)
                        epilogue_half<3, true>(lbw, tq + rank * G::NCOLS, out_buf, G::SPITCH * 16, chunk0, 0, bias, realmask, lane);
                    else
                        epilogue_half<3, false>(lbw, tq + rank * G::NCOLS, out_buf, G::SPITCH * 16, chunk0, 0, bias, realmask, lane);
                }
                tc_fence_before();
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_act);
                if (stamp && p == 0 && et == 0) eval_timeline(a)[4 * L + 3] = clock64();
            }

            // -- heads: both CTAs loaded the same head tiles, so each holds the head rows of both
            //    positions; I read the 96 columns of mine (row 32*(h/7) + h%7 = head channel h)
            const int hp = 7 * q + lane;
            const float hbias = lane < 7 ? __ldg(net.bias + (size_t)(NL - 1) * C + hp) : 0.f;
            float wpre[kFcPrefetch];
            fc1_prefetch(net, et, wpre);
            mbar_wait(bar_acc, acc_phase);
            acc_phase ^= 1u;
            tc_fence_after();
            if (lbw == 0) {
                head_read<0>(tmem_base + ((uint32_t)(q * 32) << 16) + rank * G::NCOLS, hbias, hp, scratch, vbuf, lane);
                tc_fence_before();
            }
            named_bar_sync(kEpiBar, kEpiThreads);
            if (tl) tl[4] = clock64();
            heads_tail<1>(net, a, n_eff, b0, scratch, vbuf, red, wpre, et, tl);
        }
    }

    // ---- teardown: nobody leaves (or frees TMEM) while the peer may still touch this CTA ---------
    tc_fence_before();
    cluster_sync_all();
    if (warp == 1) {
        __syncwarp();
        tmem_dealloc_pair(tmem_base, G::TMEM_COLS);
    }
}

template <int CW>
int pair_prepare(int* max_pairs) {
    cudaError_t e = cudaFuncSetAttribute(trunk_pair_kernel<CW>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         PairGeom<CW>::SMEM_BYTES);
    if (e != cudaSuccess) {
        set_error("trunk pair: cudaFuncSetAttribute failed: %s (is this an sm_100a device?)", cudaGetErrorString(e));
        return NSB_ERR_NO_DEVICE;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2, 1, 1);
    cfg.blockDim = dim3(kThreads, 1, 1);
    cfg.dynamicSmemBytes = PairGeom<CW>::SMEM_BYTES;
    int clusters = 0;
    e = cudaOccupancyMaxActiveClusters(&clusters, trunk_pair_kernel<CW>, &cfg);
    if (e != cudaSuccess || clusters < 1) {
        set_error("trunk pair: no co-resident CTA pairs (%s)", cudaGetErrorString(e));
        return NSB_ERR_NO_DEVICE;
    }
    if (max_pairs) *max_pairs = clusters;
    return 0;
}
}  // namespace

int trunk_pair_prepare(int channels, int* max_pairs) {
    if (channels == 256) return pair_prepare<256>(max_pairs);
    if (channels == 192) return pair_prepare<192>(max_pairs);
    set_error("trunk pair: unsupported width %d (192 or 256)", channels);
    return NSB_ERR_INVALID;
}

int launch_trunk_pair(const DeviceNet& net, const EvalArgs& a, int max_pairs, cudaStream_t s) {
    if (a.n <= 0) return 0;
    const int groups = (a.n + 1) / 2;  // upper bound when the launch works on a miss list
    const int pairs = groups < max_pairs ? groups : max_pairs;
    if (net.channels == 256)
        trunk_pair_kernel<256><<<2 * pairs, kThreads, PairGeom<256>::SMEM_BYTES, s>>>(net, a);
    else if (net.channels == 192)
        trunk_pair_kernel<192><<<2 * pairs, kThreads, PairGeom<192>::SMEM_BYTES, s>>>(net, a);
    else {
        set_error("trunk pair: unsupported width %d (192 or 256)", net.channels);
        return NSB_ERR_INVALID;
    }
    return 1;
}

}  // namespace nsb
