// trunk_common.cuh — device code shared by the two position-stationary trunk kernels
// (trunk_fused.cu: one CTA, 128 channels; trunk_pair.cu: CTA pair, 256 channels):
// stage 2 of feature extraction straight into the stem operand, the head read-out and the
// tail (dense logits, value MLP, sigmoids, fused legal-move decode).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "cache_device.cuh"
#include "decode_device.cuh"
#include "epilogue.cuh"
#include "nsb_internal.h"
#include "pack_device.cuh"
#include "umma.cuh"

namespace nsb {

constexpr int kThreads = 384;
constexpr int kEpiThreads = 256;
constexpr int kEpiWarps = kEpiThreads / 32;
constexpr uint32_t kEpiBar = 1;  // named barrier id for the 8 epilogue warps

constexpr int kFcPrefetch = 27;

// One FeatureBitboard (reference src/cuda/extractbit.cu:20-37) -> {w0, w1, w2, value}: bit t of
// the 81-bit string w2:w1:w0 is the plane's value at output position t (rotation applied), and
// `value` holds the fp32 fill value as two bf16: low half = the value rounded to bf16, high half = the bf16 rounding
// of the remainder (what the twin channel of a scalar plane carries, nsb_internal.h kFirstScalarChannel).  Squares 0..62 live in lo bits 0..62,
// squares 63..80 in hi bits 0..17; every other bit of the input is ignored.
__device__ __forceinline__ uint4 plane_bits(uint4 f) {
    uint32_t s0 = f.x;
    uint32_t s1 = (f.y & 0x7FFFFFFFu) | (f.z << 31);
    uint32_t s2 = (f.z >> 1) & 0x1FFFFu;
    if ((f.z >> 24) & 1u) {  // rotate: out[t] = in[80 - t]  == (96-bit reversal) >> 15
        const uint32_t r0 = __brev(s2), r1 = __brev(s1), r2 = __brev(s0);
        s0 = __funnelshift_r(r0, r1, 15);
        s1 = __funnelshift_r(r1, r2, 15);
        s2 = r2 >> 15;
    }
    const float v = __uint_as_float(f.w);
    const uint32_t hi = (uint32_t)f32_to_bf16_bits(v);
    const float rest = v - __uint_as_float(hi << 16);  // exact in fp32; 0 for inf / nan inputs' sake below
    const uint32_t lo = (rest == rest && (hi & 0x7F80u) != 0x7F80u) ? (uint32_t)f32_to_bf16_bits(rest) : 0u;
    return make_uint4(s0, s1, s2, hi | (lo << 16));
}

// Diagnostics (tools/timeline.py, tools/residency.py): the clock64 stamps exist only in the diagnostic build of the
// library (libnsb_diag.so, -DNSB_DIAG); in the product build the pointer is a compile-time null and every stamp
// and its predicate fold away.
__device__ __forceinline__ unsigned long long* eval_timeline(const EvalArgs& a) {
#ifdef NSB_DIAG
    return a.timeline;
#else
    (void)a;
    return nullptr;
#endif
}

// A launch works on n positions, or - behind a cache probe - on the *count misses listed in index[].
__device__ __forceinline__ int eval_count(const EvalArgs& a) { return a.count ? __ldg(a.count) : a.n; }
// batch index of work-list entry li, -1 past the end
__device__ __forceinline__ int eval_index(const EvalArgs& a, int li, int n_eff) {
    return li < n_eff ? (a.index ? __ldg(a.index + li) : li) : -1;
}

// Stage 2 of feature extraction for the NPOS work-list entries starting at li0, executed by
// the 256 epilogue threads (et = 0..255): bitboards -> featS (bit strings) -> 16-byte records
// [chunk j][slot][8 channels] of the stem's B operand at `stem_buf` (generic pointer to slot 0 of
// chunk 0 minus the guard, i.e. the buffer base).  `tl` (optional) receives clock64 stamps.
// NT = number of threads doing the expansion (named barrier `bar` is used with NT threads).
template <int NPOS, int SPITCH, int GUARD, int NT = kEpiThreads>
__device__ __forceinline__ void expand_features(const DeviceNet& net, const EvalArgs& a, int n_eff, int li0, uint4* featS,
                                                uint8_t* stem_buf, int et, unsigned long long* tl,
                                                uint32_t bar = kEpiBar) {
    const int IN = net.in_channels, stem_chunks = 2 * net.stem_steps;
    // Per plane: the 81 occupancy bits as one contiguous little-endian bit string with the
    // rotation (extractbit.cu:20,26) already applied, plus the fill value as bf16 bits.
    if (a.positions != nullptr) {
        // stage 1 fused in: warp `pos` builds the position's 86 bitboards from its 108-byte record; they
        // go straight into featS and never exist in HBM.  The occupancy scratch is the position's own
        // first 28 featS slots (pack_device.cuh).
        const int pos = et >> 5, lane = et & 31;
        if (pos < NPOS) {
            uint4* mine = featS + pos * IN;  // (positions in: IN == 86, checked by the API)
            const int b = eval_index(a, li0 + pos, n_eff);
            if (b >= 0) {
                pack_position_warp(a.positions + b, lane, mine, [&](int c, uint4 f) { mine[c] = plane_bits(f); });
            } else {
                for (int c = lane; c < IN; c += 32) mine[c] = make_uint4(0, 0, 0, 0);
            }
        }
    } else {
        for (int i = et; i < NPOS * IN; i += NT) {
            const int pos = i / IN, c = i - pos * IN;
            const int b = eval_index(a, li0 + pos, n_eff);
            uint4 f = make_uint4(0, 0, 0, 0);
            if (b >= 0) f = __ldg(reinterpret_cast<const uint4*>(a.features) + (size_t)b * IN + c);
            featS[i] = plane_bits(f);
        }
    }
    if (tl) tl[9] = clock64();
    named_bar_sync(bar, NT);
    if (tl) tl[3] = clock64();
    // The stem reads stem_chunks chunks of 8 input channels: the real ones, the twins of the scalar planes, zero padding
    // (86 + 4 -> 96 channels = 12 chunks; 93 + 11 -> 128 = 16 chunks).  One work
    // item = (position, chunk, board row): the 8 planes' bit strings are loaded once, the
    // row's 9-bit field is cut out with a funnel shift, and 9 records of 16 B are written.
    for (int item = et; item < NPOS * stem_chunks * 9; item += NT) {
        const int pos = item / (stem_chunks * 9);
        const int r2 = item - pos * (stem_chunks * 9);
        const int j = r2 / 9, row = r2 - j * 9;
        const int bit0 = 9 * row, wi = bit0 >> 5, sh = bit0 & 31;
        uint32_t field[8], val[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int c = j * 8 + e;
            uint4 f = make_uint4(0, 0, 0, 0);
            const int src = stem_source_channel(c, IN);
            if (src >= 0) f = featS[pos * IN + src];
            const uint32_t lo = wi == 0 ? f.x : (wi == 1 ? f.y : f.z);
            const uint32_t hi = wi == 0 ? f.y : (wi == 1 ? f.z : 0u);
            field[e] = __funnelshift_r(lo, hi, sh);
            val[e] = c < IN ? (f.w & 0xFFFFu) : (f.w >> 16);  // a twin channel carries the remainder
        }
        uint8_t* dst = stem_buf + (size_t)((j * SPITCH + GUARD + pos * 100 + row * 10) * 16);
#pragma unroll
        for (int col = 0; col < 9; ++col) {
            uint32_t w[4];
#pragma unroll
            for (int e2 = 0; e2 < 4; ++e2) {
                const uint32_t a0 = val[2 * e2] & (0u - ((field[2 * e2] >> col) & 1u));
                const uint32_t a1 = val[2 * e2 + 1] & (0u - ((field[2 * e2 + 1] >> col) & 1u));
                w[e2] = a0 | (a1 << 16);
            }
            *reinterpret_cast<uint4*>(dst + col * 16) = make_uint4(w[0], w[1], w[2], w[3]);
        }
    }
    if (tl) tl[10] = clock64();
}

// Head accumulator: this warp's lanes 0..6 = head channels hp = 7q + lane (0..26 policy planes,
// 27 = value conv) for the 96 slots from COL0 (compile-time: slot -> square arithmetic folds);
// `taddr` already points at the TMEM column that holds slot COL0.
template <int COL0>
__device__ __forceinline__ void head_read(uint32_t taddr, float bias, int hp, float* scratch, float* vbuf, int lane) {
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        uint32_t v[32];
        tmem_ld32(taddr + j * 32, v);
        tmem_ld_wait();
        if (lane < 7) {
            float* dst = hp < kPolicyPlanes ? scratch + hp * 81 : vbuf;
            const bool relu = hp == kPolicyPlanes;
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                const int n = COL0 + j * 32 + i;
                if (is_real_slot(n)) {
                    const int pos = n / 100, m = n % 100, t = (m / 10) * 9 + (m % 10);
                    const float x = __uint_as_float(v[i]) + bias;
                    dst[(relu ? pos * 81 : pos * kPolicySize) + t] = relu ? fmaxf(x, 0.f) : x;  // plane-major logits
                }
            }
        }
    }
}

// First FC1 weights of this thread's hidden unit, requested before the accumulator wait.
__device__ __forceinline__ void fc1_prefetch(const DeviceNet& net, int et, float (&wpre)[kFcPrefetch]) {
    const int H = net.hidden;
#pragma unroll
    for (int t = 0; t < kFcPrefetch; ++t) wpre[t] = et < H ? __ldg(net.fc1t + (size_t)t * H + et) : 0.f;
}

// The decode part of a pass's tail, shared by all trunk kernels: NT epilogue threads, the logits of the NPOS
// positions in scratch[pos][2187], their win / draw rates in wd[pos * 2 + {0, 1}] (shared memory).  Warp `pos`
// decodes position pos (gather + softmax on logits that never left shared memory, decode_device.cuh) and, when
// the launch carries a cache, stores the row from its registers - probabilities for NSB_DECODE_PROBS
// (feedworker.cc:134-135), raw logits for LOGITS / BOTH (frame.cc:110-114), nothing for a row with NaNFound -;
// then all warps rank the rows (Node::sort) when the request asks for the order.  The caller has passed a
// barrier (named barrier `bar` of the NT threads) after writing scratch / wd and passes one before reusing them.
template <int NPOS, int NT>
__device__ __forceinline__ void decode_tail(const EvalArgs& a, int n_eff, int li0, float* scratch, const float* wd, int et,
                                            uint32_t bar = kEpiBar) {
    constexpr int NW = NT / 32;
    const int ew = et >> 5, lane = et & 31;
    if (ew < NPOS) {
        const int b = eval_index(a, li0 + ew, n_eff);
        if (b >= 0) {
            const uint32_t mb = __ldg(a.move_off + b), me = __ldg(a.move_off + b + 1);
            const int m = (int)(me - mb);
            const float w = wd[ew * 2 + 0], d = wd[ew * 2 + 1];
            const int rf = a.row_flags ? (int)__ldg(a.row_flags + b) : 0;
            float* row = scratch + ew * kPolicySize;
            float* lout = a.logits_out ? a.logits_out + mb : nullptr;
            bool nan_found;
            // (instantiations kept apart: the staging keeps the row's values live longer and the store drags the
            // cache code in, which costs the plain path microseconds if they are only predicated off)
            if (a.hashes != nullptr) {
                const uint64_t hash = __ldg(a.hashes + b);
                auto store = [&](const float (&v)[kDecodePerLane]) {
                    cache_store_warp_from(a.cache, hash, m, [&](int k) { return v[k]; }, w, d, lane);
                };
                nan_found = a.order_out ? warp_decode_row<true>(row, a.move_idx + mb, m, a.decode_mode, rf, w, d, a.legal_out + mb, lout, lane, row, store)
                                        : warp_decode_row<false>(row, a.move_idx + mb, m, a.decode_mode, rf, w, d, a.legal_out + mb, lout, lane, nullptr, store);
            } else {
                nan_found = a.order_out ? warp_decode_row<true>(row, a.move_idx + mb, m, a.decode_mode, rf, w, d, a.legal_out + mb, lout, lane, row)
                                        : warp_decode_row<false>(row, a.move_idx + mb, m, a.decode_mode, rf, w, d, a.legal_out + mb, lout, lane);
            }
            if (a.nan_flag && lane == 0) a.nan_flag[b] = nan_found ? 1 : 0;
        }
    }
    if (a.order_out != nullptr) {  // rank order of the rows (Node::sort): all epilogue warps share the work
        named_bar_sync(bar, NT);
        const int pos = ew % NPOS;
        const int b = eval_index(a, li0 + pos, n_eff);
        // the order is staged behind the row's values in the position's (dead) logits scratch
        uint16_t* ostage = reinterpret_cast<uint16_t*>(scratch + pos * kPolicySize + 608);
        if (b >= 0) {
            const uint32_t mb = __ldg(a.move_off + b), me = __ldg(a.move_off + b + 1);
            rank_row_coop(scratch + pos * kPolicySize, (int)(me - mb), ew / NPOS, NW / NPOS, lane, ostage);
        }
        named_bar_sync(bar, NT);
        if (b >= 0) {
            const uint32_t mb = __ldg(a.move_off + b), me = __ldg(a.move_off + b + 1);
            rank_row_copy_out(ostage, (int)(me - mb), ew / NPOS, NW / NPOS, lane, a.order_out + mb);
        }
    }
}

// K = 16 steps of the TS weight stream (trunk_tmem.cu) per (layer L, K block kc, any tap): the stem's second block holds channels 64..95 (or 64..127) only
__device__ __forceinline__ int block_steps(const DeviceNet& net, int L, int kc) { return (L == 0 && kc == 1) ? net.stem_steps - 4 : 4; }

// Tail of a pass with NT epilogue threads synchronised on named barrier `bar` (the 256-thread version with its FC1 prefetch is
// heads_tail below): dense logits, value MLP, sigmoids, fused decode (+ cache store).
template <int NPOS, int NT>
__device__ __forceinline__ void heads_tail_small(const DeviceNet& net, const EvalArgs& a, int n_eff, int li0,
                                                 float* scratch, const float* vbuf, float* red, int et,
                                                 uint32_t bar = kEpiBar) {
    constexpr int NW = NT / 32;
    const int ew = et >> 5, lane = et & 31;
    const int H = net.hidden;
    if (a.policy != nullptr) {
        for (int idx = et; idx < NPOS * kPolicySize; idx += NT) {
            const int pos = idx / kPolicySize, b = eval_index(a, li0 + pos, n_eff);
            if (b >= 0) a.policy[(size_t)b * kPolicySize + (idx - pos * kPolicySize)] = scratch[idx];
        }
    }
    float o[NPOS][2];
#pragma unroll
    for (int pos = 0; pos < NPOS; ++pos) o[pos][0] = o[pos][1] = 0.f;
    for (int h = et; h < H; h += NT) {  // FC(81 -> H) + ReLU, folded straight into FC(H -> 2)
        float acc[NPOS];
        const float b1 = __ldg(net.fc1b + h);
#pragma unroll
        for (int pos = 0; pos < NPOS; ++pos) acc[pos] = b1;
#pragma unroll 9
        for (int t = 0; t < 81; ++t) {
            const float w = __ldg(net.fc1t + (size_t)t * H + h);
#pragma unroll
            for (int pos = 0; pos < NPOS; ++pos) acc[pos] += w * vbuf[pos * 81 + t];
        }
        const float w0 = __ldg(net.fc2 + h), w1 = __ldg(net.fc2 + H + h);
#pragma unroll
        for (int pos = 0; pos < NPOS; ++pos) {
            const float hid = fmaxf(acc[pos], 0.f);
            o[pos][0] += w0 * hid;
            o[pos][1] += w1 * hid;
        }
    }
#pragma unroll
    for (int pos = 0; pos < NPOS; ++pos)
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const float s = warp_sum(o[pos][k]);
            if (lane == 0) red[(ew * NPOS + pos) * 2 + k] = s;
        }
    named_bar_sync(bar, NT);
    if (et < NPOS * 2) {
        const int pos = et >> 1, k = et & 1;
        float s = __ldg(net.fc2b + k);
#pragma unroll
        for (int qq = 0; qq < NW; ++qq) s += red[(qq * NPOS + pos) * 2 + k];
        const float val = 1.0f / (1.0f + expf(-s));
        red[NW * NPOS * 2 + pos * 2 + k] = val;
        const int b = eval_index(a, li0 + pos, n_eff);
        if (b >= 0) (k == 0 ? a.win : a.draw)[b] = val;
    }
    if (a.move_off != nullptr) {
        named_bar_sync(bar, NT);
        decode_tail<NPOS, NT>(a, n_eff, li0, scratch, red + NW * NPOS * 2, et, bar);
    }
    named_bar_sync(bar, NT);
}

// Tail of a pass for the NPOS work-list entries at li0, executed by the 256 epilogue threads after the
// logits (scratch[pos][2187], plane-major) and the value-conv plane (vbuf[pos][81], ReLU applied)
// are in shared memory and a kEpiBar barrier has been passed: dense logits (the Infer contract,
// trt.cc:265-267), value MLP FC(81 -> H) + ReLU, FC(H -> 2), sigmoid (one hidden unit per thread),
// fused legal-move decode on logits that never left shared memory and, when the launch carries a
// cache, the store of the decoded row (feedworker.cc:134-135: rows with NaNs are not stored).  Ends
// with a kEpiBar barrier (scratch / vbuf / red reusable).
template <int NPOS>
__device__ __forceinline__ void heads_tail(const DeviceNet& net, const EvalArgs& a, int n_eff, int li0, float* scratch,
                                           const float* vbuf, float* red, const float (&wpre)[kFcPrefetch], int et,
                                           unsigned long long* tl) {
    const int ew = et >> 5, lane = et & 31;
    const int H = net.hidden;
    if (a.policy != nullptr) {
        for (int idx = et; idx < NPOS * kPolicySize; idx += kEpiThreads) {
            const int pos = idx / kPolicySize, b = eval_index(a, li0 + pos, n_eff);
            if (b >= 0) a.policy[(size_t)b * kPolicySize + (idx - pos * kPolicySize)] = scratch[idx];
        }
    }
    if (tl) tl[5] = clock64();
    {
        float o[NPOS][2];
#pragma unroll
        for (int pos = 0; pos < NPOS; ++pos) o[pos][0] = o[pos][1] = 0.f;
        if (et < H) {
            const int h = et;
            float acc[NPOS];
            const float b1 = __ldg(net.fc1b + h);
            const float w0 = __ldg(net.fc2 + h), w1 = __ldg(net.fc2 + H + h);
#pragma unroll
            for (int pos = 0; pos < NPOS; ++pos) acc[pos] = b1;
#pragma unroll
            for (int t0 = 0; t0 < 81; t0 += kFcPrefetch) {
                float w[kFcPrefetch];
#pragma unroll
                for (int t = 0; t < kFcPrefetch; ++t)
                    w[t] = t0 == 0 ? wpre[t] : __ldg(net.fc1t + (size_t)(t0 + t) * H + h);
#pragma unroll
                for (int t = 0; t < kFcPrefetch; ++t)
#pragma unroll
                    for (int pos = 0; pos < NPOS; ++pos) acc[pos] += w[t] * vbuf[pos * 81 + t0 + t];
            }
#pragma unroll
            for (int pos = 0; pos < NPOS; ++pos) {
                const float hid = fmaxf(acc[pos], 0.f);
                o[pos][0] = w0 * hid;
                o[pos][1] = w1 * hid;
            }
        }
#pragma unroll
        for (int pos = 0; pos < NPOS; ++pos)
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                const float s = warp_sum(o[pos][k]);
                if (lane == 0) red[(ew * NPOS + pos) * 2 + k] = s;
            }
        named_bar_sync(kEpiBar, kEpiThreads);
        if (et < NPOS * 2) {
            const int pos = et >> 1, k = et & 1;
            float s = __ldg(net.fc2b + k);
#pragma unroll
            for (int qq = 0; qq < kEpiWarps; ++qq) s += red[(qq * NPOS + pos) * 2 + k];
            const float val = 1.0f / (1.0f + expf(-s));
            red[kEpiWarps * NPOS * 2 + pos * 2 + k] = val;
            const int b = eval_index(a, li0 + pos, n_eff);
            if (b >= 0) (k == 0 ? a.win : a.draw)[b] = val;
        }
    }
    if (tl) tl[6] = clock64();
    if (a.move_off != nullptr) {
        named_bar_sync(kEpiBar, kEpiThreads);
        decode_tail<NPOS, kEpiThreads>(a, n_eff, li0, scratch, red + kEpiWarps * NPOS * 2, et);
    }
    named_bar_sync(kEpiBar, kEpiThreads);
    if (tl) tl[7] = clock64();
}

}  // namespace nsb
