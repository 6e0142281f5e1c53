// nsb_internal.h — shared host/device definitions for the leaf-evaluation kernels.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "../../include/nsb.h"

namespace nsb {

constexpr int kSquares = NSB_NUM_SQUARES;       // 81
constexpr int kPolicyPlanes = NSB_POLICY_PLANES; // 27
constexpr int kPolicySize = NSB_POLICY_SIZE;    // 2187
constexpr int kStemCin = 128;                   // stem input channels of the weight tiles (two K blocks of 64)
constexpr int kMaxInChannels = 96;              // feature channels a net may take (86 SimpleFeatures, 93 CustomFeaturesV1)
// Feature planes from this channel on carry arbitrary fp32 fill values (Progress, ProgressUnit, draw values, scores:
// reference src/evaluate/preset.h:61-66,112-121); the planes before it are 0/1 by construction (pieces, hands, colour).
// The stem sees each such plane twice: its value rounded to bf16, and - in a TWIN channel appended behind the real ones,
// with the same weights - the bf16 rounding of what that rounding lost, so these inputs reach the fp32 accumulator with
// ~16 mantissa bits instead of 8 (the reference feeds fp32 planes, src/infer/trt.cc:144-150).
constexpr int kFirstScalarChannel = 82;
__host__ __device__ constexpr int stem_twins(int in_channels) { return in_channels > kFirstScalarChannel ? in_channels - kFirstScalarChannel : 0; }
// K = 16 steps of the stem per tap: 6 (96 channels: 86 + 4 twins) or 8 (128 channels: 93 + 11 twins)
__host__ __device__ constexpr int stem_steps(int in_channels) { return in_channels + stem_twins(in_channels) <= 96 ? 6 : 8; }
// blob channel that stem input channel ci multiplies (-1: padding)
__host__ __device__ constexpr int stem_source_channel(int ci, int in_channels) {
    return ci < in_channels ? ci : (ci < in_channels + stem_twins(in_channels) ? kFirstScalarChannel + (ci - in_channels) : -1);
}
constexpr int kStageBytes = 16384;              // one weight tile: 128 Cout x 64 Cin bf16
constexpr int kMaxHidden = 256;

// Device-side geometry of the position-stationary trunk kernel (DESIGN.md §6).
// A position occupies 100 "slots": slot = 10 * (t / 9) + (t % 9) for board index t, the 10th
// column and 10th row are permanent zeros, so tap (dh, dw) is the slot offset 10*dh + dw.
template <int C>
struct TrunkGeom {
    static_assert(C == 128 || C == 256, "trunk width must be 128 or 256");
    static constexpr int KCH = C / 8;                     // 16-byte channel chunks per slot
    static constexpr int NPOS = (C == 128) ? 2 : 1;       // positions resident per CTA pass
    static constexpr int NCOLS = NPOS * 96;               // UMMA N: slots [0, NCOLS); last real slot 88 / 188
    static constexpr int NHALF = C / 128;                 // Cout halves (UMMA M = 128 each)
    static constexpr int GUARD = 12;                      // zero slots before slot 0 (>= 11)
    static constexpr int SPITCH = (GUARD + NCOLS + 11) | 1; // slots per channel chunk (odd)
    static constexpr int BUF_BYTES = ((KCH * SPITCH * 16 + 127) / 128) * 128;
    static constexpr int NSTAGES = 6;                     // weight ring depth
    static constexpr int KC64 = C / 64;                   // 64-channel K blocks per tap
    static constexpr int TMEM_COLS = 256;                 // >= NHALF * NCOLS, power of two
    static constexpr int SCRATCH_FLOATS = NPOS * kPolicySize;
    // dynamic shared memory map (byte offsets from a 128-aligned base)
    static constexpr int OFF_BUF_A = 0;
    static constexpr int OFF_BUF_B = OFF_BUF_A + BUF_BYTES;
    static constexpr int OFF_RING = OFF_BUF_B + BUF_BYTES;
    static constexpr int OFF_SCRATCH = OFF_RING + NSTAGES * kStageBytes;
    static constexpr int OFF_FEAT = OFF_SCRATCH + ((SCRATCH_FLOATS * 4 + 15) / 16) * 16;
    static constexpr int OFF_VBUF = OFF_FEAT + NPOS * kMaxInChannels * 16;
    static constexpr int OFF_RED = OFF_VBUF + ((NPOS * 81 * 4 + 15) / 16) * 16;
    static constexpr int OFF_BARS = OFF_RED + ((8 * NPOS * 2 * 4 + NPOS * 2 * 4 + 15) / 16) * 16;
    static constexpr int SMEM_BYTES = OFF_BARS + (2 * NSTAGES + 2) * 8 + 16 + 128; // + align slack
    static_assert(NCOLS % 16 == 0 && NCOLS <= 256, "UMMA N");
    static_assert(NHALF * NCOLS <= TMEM_COLS, "TMEM columns");
    static_assert(SMEM_BYTES <= 232448, "exceeds 227 KB of shared memory");
};

// Geometry of the CTA-pair trunk kernel for 192- and 256-channel nets (trunk_pair.cu, DESIGN.md §6.2):
// a cluster of two CTAs owns two positions, CTA r holds position r's activations (all C channels)
// and the weight rows of Cout half r; one cta_group::2 MMA (M = 256, N = 192) per K = 16 step.
// At C = 192 a Cout half is 96 channels: TMEM lanes 0..95 (quadrants 0..2) of each CTA; lanes
// 96..127 multiply zero weight rows and are never read back.  The K side is exact (3 blocks of 64).
template <int C_>
struct PairGeom {
    static_assert(C_ == 192 || C_ == 256, "pair trunk width must be 192 or 256");
    static constexpr int C = C_;
    static constexpr int KCH = C / 8;                     // channel chunks per slot (24 / 32)
    static constexpr int NCOLS = 96;                      // slots of this CTA's position (last real slot 88)
    static constexpr int NPAIR = 2 * NCOLS;               // UMMA N across the pair
    static constexpr int GUARD = 12;
    static constexpr int SPITCH = (GUARD + NCOLS + 11) | 1;
    static constexpr int BUF_BYTES = ((KCH * SPITCH * 16 + 127) / 128) * 128;
    static constexpr int XCH = C / 16;                    // channel chunks of one Cout half (12 / 16)
    static constexpr int QUADS = XCH / 4;                 // TMEM lane quadrants holding real Cout rows (3 / 4)
    static constexpr int XROW = 89 * 16;                  // bytes one bulk push moves per chunk: slots 0..88 (the rest
                                                          // of the 96 are padding that is zero on both sides already)
    static constexpr int XPITCH = (NCOLS + 1) * 16;       // exchange buffer chunk pitch: odd slot count, so that
                                                          // the two chunks of one stmatrix hit different banks
    static constexpr int XBUF_BYTES = XCH * XPITCH;
    static constexpr int NSTAGES = C == 256 ? 5 : 7;      // weight ring: as deep as shared memory allows
    static constexpr int KC64 = C / 64;
    static constexpr int TMEM_COLS = 256;
    static constexpr int NBARS = 2 * NSTAGES + 4;         // full[], empty[], act, acc, peer_act, skip
    static constexpr int OFF_BUF_A = 0;
    static constexpr int OFF_BUF_B = OFF_BUF_A + BUF_BYTES;
    static constexpr int OFF_XBUF = OFF_BUF_B + BUF_BYTES;  // also the logits scratch of the tail
    static constexpr int OFF_RING = OFF_XBUF + XBUF_BYTES;
    static constexpr int OFF_FEAT = OFF_RING + NSTAGES * kStageBytes;
    static constexpr int OFF_VBUF = OFF_FEAT + kMaxInChannels * 16;
    static constexpr int OFF_RED = OFF_VBUF + ((81 * 4 + 15) / 16) * 16;
    static constexpr int OFF_BARS = OFF_RED + ((8 * 2 * 4 + 2 * 4 + 15) / 16) * 16;
    static constexpr int SMEM_BYTES = OFF_BARS + NBARS * 8 + 16 + 128;
    static_assert(kPolicySize * 4 <= XBUF_BYTES, "logits scratch aliases the exchange buffer");
    static_assert(SMEM_BYTES <= 232448, "exceeds 227 KB of shared memory");
};

// Device pointers + shape of a loaded net (filled by weights.cc / nsb_api.cu).
struct DeviceNet {
    int channels;      // C
    int blocks;        // residual blocks
    int in_channels;   // feature channels per position (86; 93 for CustomFeaturesV1), <= kMaxInChannels
    int stem_steps;    // K = 16 steps of the stem per tap (stem_steps(in_channels))
    int hidden;        // value MLP hidden units (<= 256)
    int num_layers;    // 1 (stem) + 2*blocks + 1 (heads)
    int stages_per_pass;   // classic stream: 16 KB tiles per pass; TS stream: 4 KB K = 16 steps per pass
    const uint8_t* tiles;  // [stages_per_pass][16384] bf16 weight tiles in stream order (or the TS stream)
    const float* bias;     // [num_layers][C]  (head row: 27 policy biases, value-conv bias at 27)
    const float* fc1t;     // [81][hidden]  (transposed for coalesced reads)
    const float* fc1b;     // [hidden]
    const float* fc2;      // [2][hidden]
    const float* fc2b;     // [2]
};

// Device-resident evaluation cache (cache_device.cuh; reference src/mcts/evalcache.h:28-38 rows).
struct CacheEntry {
    uint64_t hash;
    uint32_t n;  // number of legal moves of the row (<= 164)
    uint32_t pad0;
    float win, draw;
    float policy[NSB_CACHE_MAX_MOVES];
    uint32_t pad1[2];
};
static_assert(sizeof(CacheEntry) == 688, "cache entry is 688 bytes (16-byte multiple)");
struct DeviceCache {
    CacheEntry* entries;            // [num_bundles][3]
    uint32_t* meta;                 // [num_bundles]: lock bit 31 | used bits 8..10 | recency order bits 0..5
    unsigned long long num_bundles; // 0 = no cache
};

struct EvalArgs {
    const nsb_feature_bitboard* features;  // [n][86]
    const nsb_position* positions;         // [n] or nullptr; when set, stage 1 runs in the kernel's prologue
                                           // and `features` is not read (SURVEY.md §8 f2)
    int n;
    float* policy;                // [n][2187] or nullptr (fused decode only)
    float* win;                   // [n]
    float* draw;                  // [n]
    const uint32_t* move_off;     // [n+1] or nullptr
    const uint16_t* move_idx;
    float* legal_out;
    uint16_t* order_out;          // optional: per position the rank order of its decoded row (decode_device.cuh)
    uint8_t* nan_flag;
    int decode_mode;              // NSB_DECODE_* [| NSB_DECODE_NAN_FALLBACK]
    const uint8_t* row_flags;     // [n] or nullptr: NSB_ROW_* bits (NSB_DECODE_BOTH)
    float* logits_out;            // optional (NSB_DECODE_BOTH): the raw gathered logits beside legal_out
    unsigned long long* timeline;  // optional (diagnostics): CTA 0 writes 4 clock64 stamps per layer
    // cached evaluation (optional): the launch works on the positions index[0 .. *count) (the misses
    // of a preceding cache probe) instead of 0 .. n-1, and stores every decoded row under hashes[b]
    const int* index;
    const int* count;
    const uint64_t* hashes;
    DeviceCache cache;
};

// host-side weight handling (weights.cc)
size_t blob_floats(const nsb_net_desc& d);
void blob_random(const nsb_net_desc& d, uint64_t seed, float* blob);
int stages_per_pass(const nsb_net_desc& d);
int ts_steps_per_pass(const nsb_net_desc& d);
void pack_weights_ts(const nsb_net_desc& d, const float* blob, uint16_t* stream);  // weight stream of the trunk_tmem.cu kernels
// Packs canonical blob -> host images of DeviceNet arrays (tiles as uint16 bf16 bits).
void pack_weights(const nsb_net_desc& d, const float* blob, uint16_t* tiles, float* bias,
                  float* fc1t, float* fc1b, float* fc2, float* fc2b);

// kernel launchers (each returns the number of kernels launched or <0 after setting last error)
int launch_extract(const nsb_feature_bitboard* d_fb, size_t n, int channels, int channels_first,
                   float* d_planes, cudaStream_t s);
int launch_pack_positions(const nsb_position* d_pos, size_t n, nsb_feature_bitboard* d_fb,
                          cudaStream_t s);
int launch_decode(const float* d_policy, const float* d_win, const float* d_draw, size_t n,
                  const uint32_t* d_off, const uint16_t* d_idx, int mode, float* d_out,
                  uint8_t* d_flag, cudaStream_t s, const uint8_t* d_row_flags = nullptr, float* d_logits_out = nullptr);
int launch_trunk_fused(const DeviceNet& net, const EvalArgs& a, int num_sms, cudaStream_t s);
int launch_cache_probe(const DeviceCache& c, const uint64_t* d_hashes, size_t n, const uint32_t* d_off, float* d_legal,
                       float* d_win, float* d_draw, uint8_t* d_hit, uint8_t* d_nan_flag, int* d_miss_idx, int* d_miss_count,
                       cudaStream_t s, uint16_t* d_order = nullptr, int mode = 0, const uint8_t* d_row_flags = nullptr,
                       float* d_logits_out = nullptr);
int launch_cache_store(const DeviceCache& c, const uint64_t* d_hashes, size_t n, const uint32_t* d_off,
                       const float* d_legal, const float* d_win, const float* d_draw, const uint8_t* d_skip,
                       uint8_t* d_stored, cudaStream_t s);
int launch_cache_clear(const DeviceCache& c, cudaStream_t s);
int trunk_fused_prepare(int channels);  // sets max dynamic smem attribute
int trunk_duo_prepare(int* ctas_per_sm);  // 128-channel trunk sized for two CTAs per SM (trunk_duo_kernel in trunk_tmem.cu)
int launch_trunk_duo(const DeviceNet& net, const EvalArgs& a, int num_sms, int ctas_per_sm, cudaStream_t s);
int trunk_quad_prepare();  // 128-channel trunk with four positions per CTA, one CTA per SM (trunk_quad_kernel in trunk_tmem.cu)
int launch_trunk_quad(const DeviceNet& net, const EvalArgs& a, int num_sms, cudaStream_t s);
int trunk_pair_prepare(int channels, int* max_pairs);  // same for the CTA-pair kernel of that width; reports co-resident clusters
int launch_trunk_pair(const DeviceNet& net, const EvalArgs& a, int max_pairs, cudaStream_t s);
int umma_probe(int gpu, int n_cols, int k_elems, int shift_rows, int layout, int iters, float* max_err,
               double* cycles_per_mma);
int bulk_rate_probe(int gpu, int ctas, int tile_bytes, int stages, int split, double* bytes_per_cycle);
int umma_selftest(int gpu, int n_cols, int k_elems, int shift_rows, float* max_err, float* epi_err);

void set_error(const char* fmt, ...);

// numa.cc: placement of host batch buffers next to a GPU (reference src/evaluate/evaluator.cc:39-83,127-136)
int gpu_numa_node(int gpu);
int numa_bind_thread_to_gpu(int gpu);
void* alloc_near_gpu(size_t bytes, int gpu, int* node_out);
void free_near_gpu(void* p, size_t bytes);

// shared device code: warp-level gather + softmax over one position's legal moves
}  // namespace nsb
