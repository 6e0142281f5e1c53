// weights.cc — host-side weight handling: canonical fp32 blob layout, deterministic random
// init, and repacking into the bf16 tile stream the trunk kernel consumes.
//
// The reference loads an external ONNX through TensorRT (reference src/infer/trt.cc:109-232) and
// ships no model; only the I/O contract is pinned (trt.cc:144-150,193-227).  The canonical
// random-init net and its blob layout are defined in DESIGN.md §5:
//   stem.w[C][IN][3][3] stem.b[C]
//   blocks x { conv1.w[C][C][3][3] conv1.b[C] conv2.w[C][C][3][3] conv2.b[C] }
//   policy.w[27][C] policy.b[27]   value.w[C] value.b[1]
//   fc1.w[H][81] fc1.b[H]   fc2.w[2][H] fc2.b[2]
#include <cmath>
#include <cstring>

#include "nsb_internal.h"

namespace nsb {

size_t blob_floats(const nsb_net_desc& d) {
    const size_t C = d.channels, IN = d.in_channels, H = d.value_hidden, NB = d.blocks;
    return C * IN * 9 + C + NB * 2 * (C * C * 9 + C) + kPolicyPlanes * C + kPolicyPlanes + C + 1 +
           H * 81 + H + 2 * H + 2;
}

// Output channels per 128-row tile: 128 channels are one tile; 192 and 256 are split into two Cout halves, one per
// CTA of trunk_pair.cu, and a 96-channel half fills rows 0..95 of its tile (rows 96..127 are zero).
static inline int cout_halves(int channels) { return channels == 128 ? 1 : 2; }

int stages_per_pass(const nsb_net_desc& d) {
    const int nhalf = cout_halves(d.channels), kc64 = d.channels / 64;
    return 9 * (kStemCin / 64) * nhalf + 2 * d.blocks * 9 * kc64 * nhalf + kc64;
}

static inline uint16_t bf16_bits_rne(float x) {
    uint32_t u;
    std::memcpy(&u, &x, 4);
    if ((u & 0x7F800000u) == 0x7F800000u) return (uint16_t)(u >> 16);
    u += 0x7FFFu + ((u >> 16) & 1u);
    return (uint16_t)(u >> 16);
}
static inline float bf16_round(float x) {
    const uint32_t u = (uint32_t)bf16_bits_rne(x) << 16;
    float r;
    std::memcpy(&r, &u, 4);
    return r;
}

namespace {
struct Rng {
    uint64_t s;
    uint64_t next() {  // splitmix64
        uint64_t z = (s += 0x9E3779B97F4A7C15ull);
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        return z ^ (z >> 31);
    }
    double uniform() { return ((double)(next() >> 11) + 0.5) * (1.0 / 9007199254740992.0); }
    float normal(float std) {  // Box-Muller, one value per call (deterministic, portable)
        const double u1 = uniform(), u2 = uniform();
        return (float)(std * std::sqrt(-2.0 * std::log(u1)) * std::cos(6.283185307179586 * u2));
    }
};
}  // namespace

void blob_random(const nsb_net_desc& d, uint64_t seed, float* blob) {
    const int C = d.channels, IN = d.in_channels, H = d.value_hidden, NB = d.blocks;
    Rng r{seed * 0x2545F4914F6CDD1Dull + 0x1234567ull};
    float* w = blob;
    auto fill = [&](size_t n, float std) {
        for (size_t i = 0; i < n; ++i) *w++ = bf16_round(r.normal(std));
    };
    // The feature planes are mostly 0/1 with ~20-40 of 86 planes active per square.
    fill((size_t)C * IN * 9, std::sqrt(2.0f / (float)(IN * 9)));
    fill(C, 0.05f);
    for (int b = 0; b < NB; ++b) {
        fill((size_t)C * C * 9, std::sqrt(2.0f / (float)(C * 9)));          // conv1: He-normal
        fill(C, 0.05f);
        fill((size_t)C * C * 9, 0.25f * std::sqrt(2.0f / (float)(C * 9)));  // conv2: damped branch
        fill(C, 0.05f);
    }
    fill((size_t)kPolicyPlanes * C, std::sqrt(1.0f / (float)C));
    fill(kPolicyPlanes, 0.05f);
    fill(C, std::sqrt(1.0f / (float)C));
    fill(1, 0.05f);
    fill((size_t)H * 81, std::sqrt(2.0f / 81.0f));
    fill(H, 0.05f);
    fill((size_t)2 * H, std::sqrt(1.0f / (float)H));
    fill(2, 0.05f);
}

// Tile = the A operand of four K=16 MMAs: [j = 8 K-chunks][row = 128 Cout][e = 8 Cin] bf16, i.e.
// K-major SWIZZLE_NONE canonical layout with LBO = 2048 B (between K chunks) and SBO = 128 B.
static inline size_t tile_index(int j, int row, int e) { return ((size_t)j * 128 + row) * 8 + e; }

void pack_weights(const nsb_net_desc& d, const float* blob, uint16_t* tiles, float* bias,
                  float* fc1t, float* fc1b, float* fc2, float* fc2b) {
    const int C = d.channels, IN = d.in_channels, H = d.value_hidden, NB = d.blocks;
    const int nhalf = cout_halves(C), rows = C / nhalf, kc64 = C / 64;
    const size_t tile_elems = kStageBytes / 2;
    const float* w = blob;
    uint16_t* t = tiles;
    int layer = 0;
    auto pack_conv = [&](const float* cw, int cin_real, int cin_pad, bool stem = false) {
        for (int tap = 0; tap < 9; ++tap)
            for (int kc = 0; kc < cin_pad / 64; ++kc)
                for (int half = 0; half < nhalf; ++half) {
                    for (int j = 0; j < 8; ++j)
                        for (int row = 0; row < 128; ++row)
                            for (int e = 0; e < 8; ++e) {
                                const int co = half * rows + row, ci = kc * 64 + j * 8 + e;
                                // the stem: twin channels repeat the weights of the scalar planes (nsb_internal.h)
                                const int src = stem ? stem_source_channel(ci, cin_real) : (ci < cin_real ? ci : -1);
                                const float v = src >= 0 && row < rows ? cw[((size_t)co * cin_real + src) * 9 + tap] : 0.f;
                                t[tile_index(j, row, e)] = bf16_bits_rne(v);
                            }
                    t += tile_elems;
                }
    };
    pack_conv(w, IN, kStemCin, true);
    w += (size_t)C * IN * 9;
    std::memcpy(bias + (size_t)layer * C, w, sizeof(float) * C);
    w += C;
    ++layer;
    for (int b = 0; b < 2 * NB; ++b) {
        pack_conv(w, C, C);
        w += (size_t)C * C * 9;
        std::memcpy(bias + (size_t)layer * C, w, sizeof(float) * C);
        w += C;
        ++layer;
    }
    // heads: head channel h (0..26 = policy planes, 27 = value conv) sits in tile row 32*(h/7) + h%7
    // (7 per TMEM lane quadrant, so all epilogue warps share the read-out); remaining rows zero
    const float* pw = w;
    const float* pb = w + (size_t)kPolicyPlanes * C;
    const float* vw = pb + kPolicyPlanes;
    const float* vb = vw + C;
    for (int kc = 0; kc < kc64; ++kc) {
        for (int j = 0; j < 8; ++j)
            for (int row = 0; row < 128; ++row)
                for (int e = 0; e < 8; ++e) {
                    const int ci = kc * 64 + j * 8 + e;
                    float v = 0.f;
                    const int hc = (row % 32) < 7 ? 7 * (row / 32) + (row % 32) : -1;
                    if (hc >= 0 && hc < kPolicyPlanes) v = pw[(size_t)hc * C + ci];
                    else if (hc == kPolicyPlanes) v = vw[ci];
                    t[tile_index(j, row, e)] = bf16_bits_rne(v);
                }
        t += tile_elems;
    }
    float* hb = bias + (size_t)layer * C;
    std::memset(hb, 0, sizeof(float) * C);
    std::memcpy(hb, pb, sizeof(float) * kPolicyPlanes);
    hb[kPolicyPlanes] = vb[0];
    w = vb + 1;
    for (int h = 0; h < H; ++h)
        for (int s = 0; s < 81; ++s) fc1t[(size_t)s * H + h] = w[(size_t)h * 81 + s];
    w += (size_t)H * 81;
    std::memcpy(fc1b, w, sizeof(float) * H);
    w += H;
    std::memcpy(fc2, w, sizeof(float) * 2 * H);
    w += 2 * H;
    std::memcpy(fc2b, w, sizeof(float) * 2);
}


// ---- "TS" weight stream (trunk_ts.cu: the A operand goes global -> registers -> tensor memory) ------
// One 4 KB block per K = 16 MMA step, [128 accumulator rows][16 input channels] bf16 (a row's 32
// bytes are exactly what one producer thread stores into its TMEM lane), in issue order:
//   layer, K block kc (64 input channels; the previous epilogue finishes them in this order),
//   tap, step k (16 channels).
// Accumulator row 32q + 16lb + r holds output channel 64lb + 16q + r, so that lane block lb of every
// TMEM quadrant - one half of the epilogue - is exactly K block lb of the next layer.  The head
// layer keeps its own row assignment (head channel h in row 32*(h/7) + h%7).
int ts_steps_per_pass(const nsb_net_desc& d) {
    const int kc64 = d.channels / 64;
    return 9 * stem_steps(d.in_channels) + 2 * d.blocks * 9 * kc64 * 4 + kc64 * 4;  // stem: 6 or 8 steps per tap
}

void pack_weights_ts(const nsb_net_desc& d, const float* blob, uint16_t* stream) {
    const int C = d.channels, IN = d.in_channels, NB = d.blocks;
    const int kc64 = C / 64;
    const float* w = blob;
    uint16_t* t = stream;
    auto row_channel = [](int row) { return 64 * ((row >> 4) & 1) + 16 * (row >> 5) + (row & 15); };
    auto pack_conv = [&](const float* cw, int cin_real, int kblocks, int last_block_steps, bool stem = false) {
        for (int kc = 0; kc < kblocks; ++kc)
            for (int tap = 0; tap < 9; ++tap)
                for (int k = 0; k < (kc + 1 == kblocks ? last_block_steps : 4); ++k) {
                    for (int row = 0; row < 128; ++row)
                        for (int e = 0; e < 16; ++e) {
                            const int co = row_channel(row), ci = kc * 64 + k * 16 + e;
                            const int src = stem ? stem_source_channel(ci, cin_real) : (ci < cin_real ? ci : -1);
                            const float v = src >= 0 ? cw[((size_t)co * cin_real + src) * 9 + tap] : 0.f;
                            t[row * 16 + e] = bf16_bits_rne(v);
                        }
                    t += 128 * 16;
                }
    };
    pack_conv(w, IN, 2, stem_steps(IN) - 4, true);  // stem: channels 0..63, then 64..95 (86 + 4 twins) or 64..127 (93 + 11)
    w += (size_t)C * IN * 9 + C;
    for (int b = 0; b < 2 * NB; ++b) {
        pack_conv(w, C, kc64, 4);
        w += (size_t)C * C * 9 + C;
    }
    const float* pw = w;
    const float* vw = w + (size_t)kPolicyPlanes * C + kPolicyPlanes;
    for (int kc = 0; kc < kc64; ++kc)
        for (int k = 0; k < 4; ++k) {
            for (int row = 0; row < 128; ++row)
                for (int e = 0; e < 16; ++e) {
                    const int ci = kc * 64 + k * 16 + e;
                    const int hc = (row % 32) < 7 ? 7 * (row / 32) + (row % 32) : -1;
                    float v = 0.f;
                    if (hc >= 0 && hc < kPolicyPlanes) v = pw[(size_t)hc * C + ci];
                    else if (hc == kPolicyPlanes) v = vw[ci];
                    t[row * 16 + e] = bf16_bits_rne(v);
                }
            t += 128 * 16;
        }
}

}  // namespace nsb
