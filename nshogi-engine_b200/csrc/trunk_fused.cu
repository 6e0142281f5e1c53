// trunk_fused.cu — position-stationary ResNet policy/value forward on tcgen05 (sm_100a).
//
// Replaces the reference's TensorRT enqueue (reference src/infer/trt.cc:256-261: extractBits +
// IExecutionContext::enqueueV3) with ONE persistent kernel per batch:
//
//   feature bitboards --(expand in-kernel)--> bf16 activations resident in SHARED MEMORY for the
//   whole network --> policy logits / value / draw (+ optional fused legal-move decode).
//
// Why this shape (DESIGN.md §6): leaf positions are independent 9x9 boards, so a CTA can own a
// few positions and run every layer on them without ever touching HBM for activations.  Each
// conv is computed transposed, D^T[Cout x slots] = W[Cout x Cin*9] * X^T, so the UMMA M dimension
// is Cout (128) and N is the number of board slots (192 = 2 positions, any multiple of 16).  The
// activations are stored as the UMMA K-major SWIZZLE_NONE B operand [Cin/8][slot][8] with a uniform
// 16-byte row pitch and a 10x10 zero-padded slot grid per position; a 3x3 tap (dh, dw) is then the
// SAME buffer with the descriptor start address moved by 10*dh + dw rows: im2col costs nothing.
// Weights stream from L2 through a 6-deep ring of 16 KB tiles filled by the bulk-copy engine.
//
// Warp roles (384 threads): warp 0 = weight producer, warp 1 = MMA issuer + TMEM owner,
// warps 4-11 = feature expansion, epilogues (TMEM -> bias/residual/ReLU -> bf16 -> smem via
// stmatrix, epilogue.cuh), heads.  Two epilogue warps share each TMEM lane quadrant and split the
// columns (C = 128: one position each) or the Cout halves (C = 256).
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>

#include "trunk_common.cuh"

namespace nsb {

namespace {

// CL > 1: the CTAs of a cluster of CL share ONE weight stream.  Every CTA of a launch reads the same tiles in the same
// order, so CTA r of a cluster fetches slice r of each tile (16 KB / CL) and the bulk-copy engine multicasts it into the
// ring slot of all CL CTAs: L2 -> SM weight traffic drops to 1 / CL.  A ring slot is free when the MMAs of ALL CL CTAs
// that read it have retired (the commit arrives on the slot's barrier in every CTA of the cluster), so the CTAs of a
// cluster run the same number of passes - one that has no positions left runs on empty boards and stores nothing.
template <int C, int CL = 1>
__global__ void __launch_bounds__(kThreads, 1) trunk_fused_kernel(const DeviceNet net, const EvalArgs a) {
    using G = TrunkGeom<C>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 127) & ~(uintptr_t)127);
    const uint32_t sbase = smem_u32(smem);
    const uint32_t bufA = sbase + G::OFF_BUF_A, bufB = sbase + G::OFF_BUF_B;
    const uint32_t ring = sbase + G::OFF_RING;
    float* scratch = reinterpret_cast<float*>(smem + G::OFF_SCRATCH);
    uint4* featS = reinterpret_cast<uint4*>(smem + G::OFF_FEAT);
    float* vbuf = reinterpret_cast<float*>(smem + G::OFF_VBUF);
    float* red = reinterpret_cast<float*>(smem + G::OFF_RED);  // [8][NPOS][2] + wd[NPOS][2]
    const uint32_t bars = sbase + G::OFF_BARS;
    auto bar_full = [&](int s) { return bars + 8u * s; };
    auto bar_empty = [&](int s) { return bars + 8u * (G::NSTAGES + s); };
    const uint32_t bar_act = bars + 8u * (2 * G::NSTAGES);
    const uint32_t bar_acc = bars + 8u * (2 * G::NSTAGES + 1);
    volatile uint32_t* tmem_holder =
        reinterpret_cast<volatile uint32_t*>(smem + G::OFF_BARS + 8 * (2 * G::NSTAGES + 2));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_eff = eval_count(a);
    const int groups = (n_eff + G::NPOS - 1) / G::NPOS;
    const uint32_t crank = CL > 1 ? cluster_ctarank() : 0u;
    const int first = (int)blockIdx.x - (int)crank;  // the cluster's first CTA has the most passes
    const int my_passes = first < groups ? (groups - first + (int)gridDim.x - 1) / (int)gridDim.x : 0;
    const int NL = net.num_layers;

    if (eval_timeline(a) && blockIdx.x == 0 && threadIdx.x == 128) eval_timeline(a)[4 * NL + 0] = clock64();
    // ---- one-time setup ---------------------------------------------------------------------
    for (int i = threadIdx.x; i < 2 * G::BUF_BYTES / 16; i += kThreads)
        reinterpret_cast<uint4*>(smem + G::OFF_BUF_A)[i] = make_uint4(0, 0, 0, 0);
    if (threadIdx.x == 0) {
        for (int s = 0; s < G::NSTAGES; ++s) {
            mbar_init(bar_full(s), 1);
            mbar_init(bar_empty(s), CL);  // the commit of every CTA that reads the slot
        }
        mbar_init(bar_act, kEpiWarps);  // one arrival per epilogue warp (256 arrivals on one word serialise)
        mbar_init(bar_acc, 1);
        fence_mbar_init();
        if constexpr (CL > 1) {
            // In a cluster the READER arms a slot's barrier - here for the first use, afterwards when it frees the slot -
            // so that a peer's slice can never arrive at a barrier that does not expect it yet.
            const uint32_t total = (uint32_t)my_passes * (uint32_t)net.stages_per_pass;
            for (uint32_t s = 0; s < (uint32_t)G::NSTAGES && s < total; ++s) mbar_arrive_expect_tx(bar_full(s), kStageBytes);
        }
    }
    fence_proxy_async_smem();
    if (warp == 1) tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_holder)), G::TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    if constexpr (CL > 1) cluster_sync_all();  // every CTA's barriers exist before a peer multicasts into them
    tc_fence_after();
    const uint32_t tmem_base = *tmem_holder;
    if (eval_timeline(a) && blockIdx.x == 0 && threadIdx.x == 128) eval_timeline(a)[4 * NL + 1] = clock64();

    if (warp == 0 || warp == 2) {
        // ===== weight producers: linear stream of 16 KB tiles, re-walked once per pass ==========
        // TWO of them, on alternate tiles: one thread cannot issue more than one bulk copy per ~290
        // cycles (tools/bulk_probe.py), and with its waits that is one tile per ~410 cycles - slower
        // than the 392 cycles the four MMAs of a tile take.  The ring position of tile t (tiles since
        // kernel start) is t % NSTAGES, its use number t / NSTAGES.
        if (lane == 0) {
            const uint32_t me = warp >> 1;
            const uint32_t total = (uint32_t)my_passes * (uint32_t)net.stages_per_pass;
            uint32_t s_in_pass = me % (uint32_t)net.stages_per_pass;
            for (uint32_t t = me; t < total; t += 2) {
                const uint32_t stage = t % G::NSTAGES, phase = (t / G::NSTAGES) & 1u;
                mbar_wait(bar_empty(stage), phase ^ 1u);
                if constexpr (CL == 1) mbar_arrive_expect_tx(bar_full(stage), kStageBytes);
                if constexpr (CL > 1) {
                    constexpr uint32_t kSlice = kStageBytes / CL;
                    bulk_g2s_multicast(ring + stage * kStageBytes + crank * kSlice,
                                       net.tiles + (size_t)s_in_pass * kStageBytes + crank * kSlice, kSlice, bar_full(stage),
                                       (uint16_t)((1u << CL) - 1u));
                } else {
                    bulk_g2s(ring + stage * kStageBytes, net.tiles + (size_t)s_in_pass * kStageBytes, kStageBytes,
                             bar_full(stage));
                }
                s_in_pass += 2;
                if (s_in_pass >= (uint32_t)net.stages_per_pass) s_in_pass -= (uint32_t)net.stages_per_pass;
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: the whole warp walks the loop (warp-uniform control flow and operands),
        // one elected lane issues the tcgen05 instructions =======================================
        constexpr uint32_t idesc = make_idesc_bf16_f32(128, G::NCOLS);
        constexpr uint32_t b_lbo = G::SPITCH * 16;
        uint32_t stage = 0, phase = 0, act_phase = 0;
        uint32_t tiles_done = 0;
        const uint32_t tiles_total = (uint32_t)my_passes * (uint32_t)net.stages_per_pass;
        for (int p = 0; p < my_passes; ++p) {
            for (int L = 0; L < NL; ++L) {
                mbar_wait(bar_act, act_phase);
                act_phase ^= 1u;
                tc_fence_after();
                if (eval_timeline(a) && blockIdx.x == 0 && p == 0 && lane == 0) eval_timeline(a)[4 * L + 0] = clock64();
                const bool head = (L == NL - 1);
                const uint32_t in_buf = (L & 1) ? bufA : bufB;
                const int ntaps = head ? 1 : 9;
                const int kblocks = (L == 0) ? kStemCin / 64 : G::KC64;
                const int nh = head ? 1 : G::NHALF;
                for (int tap = 0; tap < ntaps; ++tap) {
                    const int shift = head ? 0 : (tap / 3 - 1) * 10 + (tap % 3 - 1);
                    for (int kc = 0; kc < kblocks; ++kc) {
                        const uint32_t b_base = in_buf + (uint32_t)((kc * 8 * G::SPITCH + G::GUARD + shift) * 16);
                        for (int half = 0; half < nh; ++half) {
                            mbar_wait(bar_full(stage), phase);
                            tc_fence_after();
                            const int ksteps = (L == 0 && kc == 1) ? net.stem_steps - 4 : 4;
                            if (elect_one()) {
                                const uint32_t a_lo = smem_desc_lo(ring + stage * kStageBytes, 2048);
                                const uint32_t b_lo = smem_desc_lo(b_base, b_lbo);
#pragma unroll
                                for (int k = 0; k < 4; ++k) {
                                    if (k >= ksteps) break;
                                    umma_bf16(tmem_base + half * G::NCOLS, smem_desc_from(a_lo + k * (4096 >> 4), 128),
                                              smem_desc_from(b_lo + (uint32_t)(2 * k * G::SPITCH), 128), idesc,
                                              (uint32_t)((tap | kc | k) != 0));
                                }
                                // frees the ring slot when the MMAs retire (CL > 1: in every CTA of the cluster, after
                                // arming this CTA's barrier for the slot's next tile)
                                if constexpr (CL > 1) {
                                    if (tiles_done + G::NSTAGES < tiles_total) mbar_arrive_expect_tx(bar_full(stage), kStageBytes);
                                    umma_commit_multicast(bar_empty(stage), (uint16_t)((1u << CL) - 1u));
                                } else {
                                    umma_commit(bar_empty(stage));
                                }
                            }
                            __syncwarp();
                            ++tiles_done;
                            if (++stage == G::NSTAGES) { stage = 0; phase ^= 1u; }
                        }
                    }
                }
                if (elect_one()) umma_commit(bar_acc);  // accumulator(s) of layer L complete
                __syncwarp();
                if (eval_timeline(a) && blockIdx.x == 0 && p == 0 && lane == 0) eval_timeline(a)[4 * L + 1] = clock64();
            }
        }
    } else if (warp >= 4) {
        // ===== expansion + epilogues + heads =====================================================
        const int et = threadIdx.x - 128;  // 0..255
        const int ew = warp - 4;           // 0..7
        const int q = ew & 3;              // TMEM lane quadrant (== warp % 4)
        const int part = ew >> 2;          // C=128: column half (= position); C=256: Cout half
        const int e_col0 = (C == 128) ? 96 * part : 0;
        const int e_half = (C == 128) ? 0 : part;
        if (eval_timeline(a) && blockIdx.x == 0 && et == 0) eval_timeline(a)[4 * NL + 11] = clock64();
        EpilogueMask<3> realmask;
        realmask.init(e_col0, lane);
        uint32_t acc_phase = 0;
        for (int p = 0; p < my_passes; ++p) {
            const int b0 = ((int)blockIdx.x + p * (int)gridDim.x) * G::NPOS;

            // -- stage 2 of feature extraction, straight into the stem's B operand (bufB) --------
            if (eval_timeline(a) && blockIdx.x == 0 && p == 0 && et == 0) eval_timeline(a)[4 * NL + 8] = clock64();
            unsigned long long* tl = (eval_timeline(a) && blockIdx.x == 0 && p == 0 && et == 0) ? eval_timeline(a) + 4 * NL : nullptr;
            expand_features<G::NPOS, G::SPITCH, G::GUARD>(net, a, n_eff, b0, featS, smem + G::OFF_BUF_B, et, tl);
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_act);
            if (eval_timeline(a) && blockIdx.x == 0 && p == 0 && et == 0) eval_timeline(a)[4 * NL + 2] = clock64();

            // -- conv layers: TMEM -> +bias (+skip) -> ReLU -> bf16 -> next layer's B operand ----
            for (int L = 0; L < NL - 1; ++L) {
                float bias[4];
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    bias[k] = __ldg(net.bias + (size_t)L * C + e_half * 128 + q * 32 + 8 * k + (lane >> 2));
                mbar_wait(bar_acc, acc_phase);
                acc_phase ^= 1u;
                tc_fence_after();
                if (eval_timeline(a) && blockIdx.x == 0 && p == 0 && et == 0) eval_timeline(a)[4 * L + 2] = clock64();
                const uint32_t out_buf = ((L & 1) ? bufB : bufA) + G::GUARD * 16;
                const bool residual = (L >= 2) && ((L & 1) == 0);
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + e_half * G::NCOLS + e_col0;
                const int chunk0 = e_half * 16 + q * 4;
                if (residual)
                    epilogue_warp<3, true>(taddr, out_buf, G::SPITCH * 16, chunk0, e_col0, bias, realmask, lane);
                else
                    epilogue_warp<3, false>(taddr, out_buf, G::SPITCH * 16, chunk0, e_col0, bias, realmask, lane);
                tc_fence_before();
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_act);
                if (eval_timeline(a) && blockIdx.x == 0 && p == 0 && et == 0) eval_timeline(a)[4 * L + 3] = clock64();
            }

            // -- heads: accumulator row 32*(h/7) + h%7 holds head channel h (0..26 policy planes,
            //    27 = value conv), i.e. 7 useful lanes in every TMEM quadrant, so all epilogue warps help
            const int hp = 7 * q + lane;
            const float hbias = lane < 7 ? __ldg(net.bias + (size_t)(NL - 1) * C + hp) : 0.f;
            float wpre[kFcPrefetch];  // first FC1 weights, requested before the accumulator wait
            fc1_prefetch(net, et, wpre);
            mbar_wait(bar_acc, acc_phase);
            acc_phase ^= 1u;
            tc_fence_after();
            if (C == 128 || part == 0) {
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16);
                if (part == 0)
                    head_read<0>(taddr, hbias, hp, scratch, vbuf, lane);
                else
                    head_read<96>(taddr + 96, hbias, hp, scratch, vbuf, lane);
                tc_fence_before();
            }
            named_bar_sync(kEpiBar, kEpiThreads);
            if (tl) tl[4] = clock64();
            heads_tail<G::NPOS>(net, a, n_eff, b0, scratch, vbuf, red, wpre, et, tl);
        }
    }

    // ---- teardown -------------------------------------------------------------------------------
    tc_fence_before();
    __syncthreads();
    if constexpr (CL > 1) cluster_sync_all();  // no peer may still multicast into, or arrive on, a CTA that has left
    if (warp == 1) {
        __syncwarp();
        tmem_dealloc(tmem_base, G::TMEM_COLS);
    }
}

template <int CL>
int launch_cluster128(const DeviceNet& net, const EvalArgs& a, int num_sms, cudaStream_t s) {
    using G = TrunkGeom<128>;
    const int groups = (a.n + G::NPOS - 1) / G::NPOS;
    cudaLaunchConfig_t cfg = {};
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = G::SMEM_BYTES;
    cfg.stream = s;
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeClusterDimension;
    attr.val.clusterDim.x = CL;
    attr.val.clusterDim.y = 1;
    attr.val.clusterDim.z = 1;
    cfg.attrs = &attr;
    cfg.numAttrs = 1;
    // clusters of CL one-CTA-per-SM blocks the device holds at once (GPC boundaries cost a few SMs); asked once - several
    // host threads may race to ask, they get the same answer
    static std::atomic<int> resident_cached{0};
    int resident = resident_cached.load(std::memory_order_relaxed);
    if (resident == 0) {
        cfg.gridDim = dim3((unsigned)(num_sms / CL * CL));
        int clusters = 0;
        if (cudaOccupancyMaxActiveClusters(&clusters, trunk_fused_kernel<128, CL>, &cfg) != cudaSuccess || clusters < 1) {
            set_error("trunk: clusters of %d CTAs do not fit this device", CL);
            return NSB_ERR_NO_DEVICE;
        }
        resident = clusters * CL < num_sms ? clusters * CL : num_sms / CL * CL;
        resident_cached.store(resident, std::memory_order_relaxed);
    }
    int grid = (groups + CL - 1) / CL * CL;
    if (grid > resident) grid = resident;
    cfg.gridDim = dim3((unsigned)grid);
    const cudaError_t e = cudaLaunchKernelEx(&cfg, trunk_fused_kernel<128, CL>, net, a);
    if (e != cudaSuccess) {
        set_error("trunk: cluster launch (%d CTAs per cluster) failed: %s", CL, cudaGetErrorString(e));
        return NSB_ERR_CUDA;
    }
    return 1;
}

}  // namespace

int trunk_fused_prepare(int channels) {
    cudaError_t e;
    if (channels == 128) {
        e = cudaFuncSetAttribute(trunk_fused_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 TrunkGeom<128>::SMEM_BYTES);
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(trunk_fused_kernel<128, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, TrunkGeom<128>::SMEM_BYTES);
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(trunk_fused_kernel<128, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, TrunkGeom<128>::SMEM_BYTES);
    } else if (channels == 256)
#ifdef NSB_DIAG  // the one-CTA 256-channel kernel: superseded by trunk_pair.cu, kept as its bit-for-bit reference
        e = cudaFuncSetAttribute(trunk_fused_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 TrunkGeom<256>::SMEM_BYTES);
#else
        e = cudaSuccess;
#endif
    else if (channels == 192)  // runs on trunk_pair.cu only; there is no one-CTA 192-channel kernel
        e = cudaSuccess;
    else {
        set_error("trunk: unsupported width %d (128, 192 or 256)", channels);
        return NSB_ERR_INVALID;
    }
    if (e != cudaSuccess) {
        set_error("trunk: cudaFuncSetAttribute failed: %s (is this an sm_100a device?)", cudaGetErrorString(e));
        return NSB_ERR_NO_DEVICE;
    }
    return 0;
}

int launch_trunk_fused(const DeviceNet& net, const EvalArgs& a, int num_sms, cudaStream_t s, int cluster) {
    if (a.n <= 0) return 0;
    if (net.channels == 128 && cluster == 2) return launch_cluster128<2>(net, a, num_sms, s);
    if (net.channels == 128 && cluster == 4) return launch_cluster128<4>(net, a, num_sms, s);
    if (net.channels == 128) {
        using G = TrunkGeom<128>;
        const int groups = (a.n + G::NPOS - 1) / G::NPOS;
        const int grid = groups < num_sms ? groups : num_sms;
        trunk_fused_kernel<128><<<grid, kThreads, G::SMEM_BYTES, s>>>(net, a);
    } else {
#ifdef NSB_DIAG
        using G = TrunkGeom<256>;
        const int groups = (a.n + G::NPOS - 1) / G::NPOS;
        const int grid = groups < num_sms ? groups : num_sms;
        trunk_fused_kernel<256><<<grid, kThreads, G::SMEM_BYTES, s>>>(net, a);
#else
        set_error("trunk: 256-channel nets run on trunk_pair.cu (the one-CTA kernel is in the diagnostic build)");
        return NSB_ERR_INVALID;
#endif
    }
    return 1;
}

}  // namespace nsb
