// nsb_api.cu — the C ABI of include/nsb.h: context, per-slot streams and device buffers, weight
// upload, and the host-buffer / device-buffer entry points of the leaf-evaluation path.
//
// Mirrors the life cycle of the reference's TensorRT executor (reference src/infer/trt.cc):
//   ctor :52-80   -> nsb_create          (cudaSetDevice, device buffers, non-blocking stream)
//   load :109-232 -> nsb_load_weights    (canonical blob -> bf16 tile stream in HBM)
//   computeNonBlocking :234-272 -> nsb_eval_async (H2D, kernels, D2H; returns immediately)
//   await :281-283 / isComputing :285-287 / resetGPU :289-291 / dtor :82-107
// Unlike the reference, every CUDA return code is checked and surfaced as a status.
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <mutex>
#include <new>
#include <vector>

#include "nsb_internal.h"
#ifdef NSB_DIAG
#include "../../include/nsb_diag.h"
#endif

namespace nsb {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
}

// Page-locked allocations made through nsb_host_alloc.  With unified addressing they are mapped into
// every device's address space at their host address, so a kernel can read its inputs from them and
// write its results into them over PCIe without a copy node on the stream ("direct" I/O mode).
static std::mutex g_host_mu;
enum class HostKind { Alloc, NodeAlloc, Registered, Adopted };
struct HostRange {
    size_t bytes = 0;
    bool direct = true;  // mapped at its host address: kernels may dereference the host pointer
    // Alloc: nsb_host_alloc (cudaFreeHost in nsb_host_free); NodeAlloc: nsb_host_alloc_near (anonymous pages on the
    // GPU's NUMA node, page-locked with cudaHostRegister; unregistered and unmapped in nsb_host_free); Registered: page-locked by nsb_host_register
    // (cudaHostUnregister is ours to call); Adopted: page-locked by the caller before we saw it (the reference's
    // Evaluator, evaluator.cc:95-106) - the caller unlocks it, we only forget it (nsb_host_unregister)
    HostKind kind = HostKind::Alloc;
};
static std::map<uintptr_t, HostRange> g_host_allocs;  // base -> range

static bool host_mapped(const void* p, size_t bytes) {
    if (p == nullptr) return false;
    const uintptr_t a = (uintptr_t)p;
    std::lock_guard<std::mutex> lock(g_host_mu);
    auto it = g_host_allocs.upper_bound(a);
    if (it == g_host_allocs.begin()) return false;
    --it;
    return it->second.direct && a + bytes <= it->first + it->second.bytes;
}

struct Slot {
    cudaStream_t stream = nullptr;
    nsb_feature_bitboard* d_feat = nullptr;
    nsb_position* d_pos = nullptr;
    float *d_policy = nullptr, *d_win = nullptr, *d_draw = nullptr, *d_legal = nullptr;
    uint32_t* d_off = nullptr;
    uint16_t* d_idx = nullptr;
    uint16_t* d_order = nullptr;  // rank order of the decoded rows (optional output)
    uint8_t* d_flag = nullptr;
    uint8_t* d_rowflags = nullptr;  // NSB_ROW_* bits of a NSB_DECODE_BOTH request
    float* d_logits = nullptr;      // raw logits beside the probabilities (allocated on first use)
    // cached evaluation (allocated by nsb_cache_create)
    uint64_t* d_hash = nullptr;
    uint8_t* d_hit = nullptr;
    int* d_miss_idx = nullptr;
    int* d_miss_count = nullptr;
    std::vector<cudaEvent_t> ev;  // start/stop pairs, one pair per trunk launch since the last await
    size_t ev_used = 0;
};

}  // namespace nsb

struct nsb_ctx {
    int gpu = 0, batch_max = 0, num_sms = 0;
    int max_pairs = 0;  // co-resident CTA pairs of the 192- / 256-channel trunk (0: single-CTA kernel)
    bool use_ts = false;       // 128-channel trunk with the weights fed through tensor memory (trunk_ts.cu)
    bool direct_io = false;    // kernels read / write the caller's page-locked buffers themselves (no copy nodes)
    bool fuse_pack = true;     // packed positions are expanded in the trunk prologue (NSB_FUSE_PACK=0: separate pack kernel)
    int duo_ctas = 0;          // > 0: the two-CTAs-per-SM 128-channel trunk (trunk_duo_kernel) is available, co-resident CTAs per SM
    int cluster128 = 1;        // NSB_TRUNK128=mc2 / mc4: trunk_fused.cu in clusters of 2 / 4 CTAs that share the weight stream by multicast
    bool duo_always = false;   // every launch uses it (multi-slot pipeline, or forced); otherwise it is chosen per batch size
    bool quad = false;         // every launch uses the four-positions-per-CTA 128-channel trunk (trunk_quad_kernel)
    nsb::DeviceNet net_duo{};  // the same net with the weight stream in trunk_duo_kernel's order (when both kernels are loaded)
    void* d_duo_tiles = nullptr;
    // launch durations (ms) that use_duo() chooses by; calibrated on this device / net at nsb_load_weights
    double t_classic_wave = 0.129, t_duo_single = 0.157, t_duo_pair = 0.215;
    bool calibrated = false;
    nsb::DeviceCache cache{};  // device-resident evaluation cache (nsb_cache_create / nsb_cache_attach)
    bool cache_owned = false;  // false: the table belongs to another ctx of the same device (nsb_cache_attach)
    nsb_net_desc desc{};
    bool loaded = false, timing = false;
    nsb::DeviceNet net{};
    void* d_weights[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    std::vector<nsb::Slot> slots;
    uint64_t launches = 0;
    double trunk_ms = 0.0;
    uint64_t trunk_launches = 0;
};

using namespace nsb;

#define NSB_CUDA(call)                                                                        \
    do {                                                                                      \
        cudaError_t e__ = (call);                                                             \
        if (e__ != cudaSuccess) {                                                             \
            set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
            return NSB_ERR_CUDA;                                                              \
        }                                                                                     \
    } while (0)

static int check_ctx(nsb_ctx* c, int slot) {
    if (!c) {
        set_error("null ctx");
        return NSB_ERR_INVALID;
    }
    if (slot < 0 || slot >= (int)c->slots.size()) {
        set_error("slot %d out of range [0,%d)", slot, (int)c->slots.size());
        return NSB_ERR_INVALID;
    }
    return 0;
}

static int check_batch(nsb_ctx* c, size_t n, bool need_weights) {
    if (n > (size_t)c->batch_max) {  // reference: assert(BatchSize <= BatchSizeM), trt.cc:237
        set_error("batch %zu exceeds batch_max %d", n, c->batch_max);
        return NSB_ERR_INVALID;
    }
    if (need_weights && !c->loaded) {
        set_error("weights not loaded (call nsb_load_weights first)");
        return NSB_ERR_STATE;
    }
    return 0;
}

static bool mode_ok(int mode) {
    const int kind = mode & NSB_DECODE_MODE_MASK;
    return (mode & ~(NSB_DECODE_MODE_MASK | NSB_DECODE_NAN_FALLBACK)) == 0 &&
           (kind == NSB_DECODE_PROBS || kind == NSB_DECODE_LOGITS || kind == NSB_DECODE_BOTH);
}

// CSR offsets of a request: start at 0, never decrease, at most 593 moves per row (the reference asserts these;
// here they would index the decode's registers, the cache rows and the rank staging).  O(n) on the host.
static int check_offsets(const uint32_t* off, size_t n, const char* who) {
    if (off[0] != 0) {
        set_error("%s: move_off must start at 0", who);
        return NSB_ERR_INVALID;
    }
    for (size_t i = 0; i < n; ++i) {
        if (off[i + 1] < off[i] || off[i + 1] - off[i] > (uint32_t)NSB_MAX_LEGAL_MOVES) {
            set_error("%s: move_off[%zu..%zu] = %u..%u: rows must hold 0..%d moves", who, i, i + 1, off[i], off[i + 1],
                      NSB_MAX_LEGAL_MOVES);
            return NSB_ERR_INVALID;
        }
    }
    return 0;
}

// Stage 1 on the device builds the 86 planes of preset::SimpleFeatures (pack_device.cuh); a net that takes another
// feature set (93-channel CustomFeaturesV1: check / pawn-file / score planes need the rules library) is fed bitboards.
static int check_positions_net(const nsb_ctx* c, const char* who) {
    if (c->desc.in_channels != NSB_FEATURE_CHANNELS) {
        set_error("%s: packed positions expand to the %d planes of SimpleFeatures; this net takes %d channels (feed bitboards)",
                  who, NSB_FEATURE_CHANNELS, c->desc.in_channels);
        return NSB_ERR_INVALID;
    }
    return 0;
}

static bool dense_outputs_mapped(size_t n, const float* policy, const float* win, const float* draw) {
    return host_mapped(policy, n * kPolicySize * sizeof(float)) && host_mapped(win, n * sizeof(float)) &&
           host_mapped(draw, n * sizeof(float));
}

extern "C" {

const char* nsb_last_error(void) { return g_err; }
const char* nsb_version(void) { return "nsb 0.3 (sm_100a: tcgen05 position-stationary trunk, cta_group::2 pair trunk, device-resident eval cache)"
#ifdef NSB_DIAG
           " [diagnostic build]"
#endif
        ; }

int nsb_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int nsb_create(nsb_ctx** out, int gpu, int batch_max, int slots, const nsb_net_desc* net) {
    if (!out || !net || batch_max <= 0 || batch_max > 65535 || slots < 1 || slots > 16) {
        set_error("nsb_create: bad arguments (batch_max 1..65535, slots 1..16)");
        return NSB_ERR_INVALID;
    }
    if ((net->channels != 128 && net->channels != 192 && net->channels != 256) || net->blocks < 1 || net->blocks > 80 ||
        net->in_channels < 1 || net->in_channels > kMaxInChannels || net->value_hidden < 1 ||
        net->value_hidden > kMaxHidden) {
        set_error("nsb_create: unsupported net (channels 128|192|256, blocks 1..80, in_channels<=%d, hidden<=%d)",
                  kMaxInChannels, kMaxHidden);
        return NSB_ERR_INVALID;
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || gpu < 0 || gpu >= ndev) {
        cudaGetLastError();
        set_error("nsb_create: no CUDA device %d (found %d); this library has no CPU fallback", gpu, ndev);
        return NSB_ERR_NO_DEVICE;
    }
    cudaDeviceProp prop;
    NSB_CUDA(cudaGetDeviceProperties(&prop, gpu));
    if (prop.major != 10) {
        set_error("nsb_create: device %d is sm_%d%d; the kernels are built for sm_100a only", gpu, prop.major,
                  prop.minor);
        return NSB_ERR_NO_DEVICE;
    }
    NSB_CUDA(cudaSetDevice(gpu));
    int rc = trunk_fused_prepare(net->channels);
    if (rc) return rc;
    int max_pairs = 0;
    // NSB_TRUNK256=single keeps the one-CTA kernel for A/B measurements (diagnostic build only); 192-channel nets
    // always run on the pair kernel
    const char* t256 = getenv("NSB_TRUNK256");
    const char* t128 = getenv("NSB_TRUNK128");
#ifndef NSB_DIAG
    if ((t256 && strcmp(t256, "single") == 0) || (t128 && strcmp(t128, "ts") == 0)) {
        set_error("nsb_create: NSB_TRUNK256=single / NSB_TRUNK128=ts exist in the diagnostic build only (libnsb_diag.so)");
        return NSB_ERR_INVALID;
    }
#endif
    if (net->channels == 192 || (net->channels == 256 && !(t256 && strcmp(t256, "single") == 0))) {
        if ((rc = trunk_pair_prepare(net->channels, &max_pairs))) return rc;
        if (max_pairs > prop.multiProcessorCount / 2) max_pairs = prop.multiProcessorCount / 2;
    }
    // 128 channels: a context with several slots is a throughput pipeline (batches in flight on
    // several streams) and gets the two-CTAs-per-SM kernel (trunk_duo_kernel: +6 % throughput, measured), or with
    // >= 4 slots the four-positions-per-CTA kernel (trunk_quad_kernel: one CTA per SM, so a launch of 256 positions fills
    // only 64 SMs and it takes about three launches in flight to cover the GPU);
    // a one-slot context evaluates one batch at a time and gets the kernel with the shorter launch
    // (trunk_fused.cu).  NSB_TRUNK128 = classic | duo | quad | mc2 | mc4 | ts forces one (mc2 / mc4: trunk_fused.cu in clusters
    // that share the weight stream by multicast; ts: experimental trunk_ts.cu, diagnostic build).
    const bool is128 = net->channels == 128;
    const bool use_ts = is128 && t128 && strcmp(t128, "ts") == 0;
    // Unforced, a 128-channel context loads BOTH kernels: a pipeline of 2-3 slots always launches the duo kernel; a
    // one-slot context picks per batch - trunk_fused.cu while the batch fits one wave of one CTA per SM (shortest
    // launch), trunk_duo_kernel (two co-resident CTAs per SM share the tensor pipe) where that is faster (use_duo()).
    const int cluster128 = (is128 && t128 && strcmp(t128, "mc2") == 0) ? 2 : (is128 && t128 && strcmp(t128, "mc4") == 0) ? 4 : 1;
    const bool want_quad = is128 && (t128 ? strcmp(t128, "quad") == 0 : slots >= 4);
    const bool want_duo = is128 && !use_ts && !want_quad && (t128 ? strcmp(t128, "duo") == 0 : true);
    const bool duo_always = want_duo && (t128 ? true : slots >= 2);
#ifdef NSB_DIAG
    if (use_ts && (rc = trunk_ts_prepare())) return rc;
#endif
    int duo_ctas = 0;
    if (want_duo && (rc = trunk_duo_prepare(&duo_ctas))) return rc;
    if (want_quad && (rc = trunk_quad_prepare())) return rc;
    nsb_ctx* c = new (std::nothrow) nsb_ctx();
    if (!c) {
        set_error("out of host memory");
        return NSB_ERR_NOMEM;
    }
    c->gpu = gpu;
    c->batch_max = batch_max;
    c->num_sms = prop.multiProcessorCount;
    c->max_pairs = max_pairs;
    c->use_ts = use_ts;
    c->duo_ctas = duo_ctas;
    c->duo_always = duo_always;
    c->quad = want_quad;
    c->cluster128 = cluster128;
    if (const char* dc = getenv("NSB_DUO_CTAS")) c->duo_ctas = duo_ctas > 0 ? atoi(dc) : 0;  // diagnostics: force the grid cap
    if (const char* fp = getenv("NSB_FUSE_PACK")) c->fuse_pack = strcmp(fp, "0") != 0;
    // A one-slot context is the latency configuration (one batch at a time: every copy node is serial
    // time) and defaults to direct I/O; a multi-slot pipeline overlaps its copies with other batches'
    // kernels and keeps them.  NSB_IO = direct | staged or nsb_set_io_mode() override.
    c->direct_io = slots == 1;
    if (const char* io = getenv("NSB_IO")) c->direct_io = strcmp(io, "direct") == 0;
    c->desc = *net;
    c->slots.resize(slots);
    const size_t B = (size_t)batch_max;
    for (auto& s : c->slots) {
        cudaError_t e = cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking);  // trt.cc:79
        if (e == cudaSuccess) e = cudaMalloc(&s.d_feat, B * (size_t)net->in_channels * sizeof(nsb_feature_bitboard));
        if (e == cudaSuccess) e = cudaMalloc(&s.d_pos, B * sizeof(nsb_position));
        if (e == cudaSuccess) e = cudaMalloc(&s.d_policy, B * kPolicySize * sizeof(float));
        if (e == cudaSuccess) e = cudaMalloc(&s.d_win, B * sizeof(float));
        if (e == cudaSuccess) e = cudaMalloc(&s.d_draw, B * sizeof(float));
        if (e == cudaSuccess) e = cudaMalloc(&s.d_legal, B * NSB_MAX_LEGAL_MOVES * sizeof(float));
        if (e == cudaSuccess) e = cudaMalloc(&s.d_off, (B + 1) * sizeof(uint32_t));
        if (e == cudaSuccess) e = cudaMalloc(&s.d_idx, B * NSB_MAX_LEGAL_MOVES * sizeof(uint16_t));
        if (e == cudaSuccess) e = cudaMalloc(&s.d_order, B * NSB_MAX_LEGAL_MOVES * sizeof(uint16_t));
        if (e == cudaSuccess) e = cudaMalloc(&s.d_flag, B);
        if (e == cudaSuccess) e = cudaMalloc(&s.d_rowflags, B);
        if (e != cudaSuccess) {
            set_error("nsb_create: device allocation failed: %s", cudaGetErrorString(e));
            nsb_destroy(c);
            return e == cudaErrorMemoryAllocation ? NSB_ERR_NOMEM : NSB_ERR_CUDA;
        }
    }
    *out = c;
    return 0;
}

void nsb_destroy(nsb_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->gpu);
    for (auto& s : c->slots) {
        if (s.stream) cudaStreamSynchronize(s.stream);
        cudaFree(s.d_feat); cudaFree(s.d_pos); cudaFree(s.d_policy); cudaFree(s.d_win); cudaFree(s.d_draw);
        cudaFree(s.d_legal); cudaFree(s.d_off); cudaFree(s.d_idx); cudaFree(s.d_order); cudaFree(s.d_flag); cudaFree(s.d_rowflags); cudaFree(s.d_logits);
        cudaFree(s.d_hash); cudaFree(s.d_hit); cudaFree(s.d_miss_idx); cudaFree(s.d_miss_count);
        for (cudaEvent_t e : s.ev) cudaEventDestroy(e);
        if (s.stream) cudaStreamDestroy(s.stream);
    }
    for (void* p : c->d_weights) cudaFree(p);
    cudaFree(c->d_duo_tiles);
    if (c->cache_owned) {
        cudaFree(c->cache.entries);
        cudaFree(c->cache.meta);
    }
    delete c;
}

int nsb_bind_thread(nsb_ctx* c) {
    if (!c) {
        set_error("null ctx");
        return NSB_ERR_INVALID;
    }
    NSB_CUDA(cudaSetDevice(c->gpu));
    return 0;
}

size_t nsb_weight_blob_floats(const nsb_net_desc* net) { return net ? blob_floats(*net) : 0; }

int nsb_weight_blob_random(const nsb_net_desc* net, uint64_t seed, float* blob) {
    if (!net || !blob) {
        set_error("nsb_weight_blob_random: null argument");
        return NSB_ERR_INVALID;
    }
    blob_random(*net, seed, blob);
    return 0;
}

static int calibrate_kernel_choice(nsb_ctx* c);

int nsb_load_weights(nsb_ctx* c, const float* blob, size_t n_floats) {
    if (!c || !blob) {
        set_error("nsb_load_weights: null argument");
        return NSB_ERR_INVALID;
    }
    if (n_floats != blob_floats(c->desc)) {
        set_error("nsb_load_weights: blob has %zu floats, net needs %zu", n_floats, blob_floats(c->desc));
        return NSB_ERR_INVALID;
    }
    NSB_CUDA(cudaSetDevice(c->gpu));
    for (auto& s : c->slots) NSB_CUDA(cudaStreamSynchronize(s.stream));
    c->loaded = false;  // a reload that fails half-way must not leave launches on freed weight buffers possible
    const nsb_net_desc& d = c->desc;
    const int C = d.channels, H = d.value_hidden, NL = 2 * d.blocks + 2;
    int stages = stages_per_pass(d);
    std::vector<uint16_t> tiles((size_t)stages * kStageBytes / 2);
    std::vector<float> bias((size_t)NL * C), fc1t((size_t)81 * H), fc1b(H), fc2(2 * (size_t)H), fc2b(2);
    pack_weights(d, blob, tiles.data(), bias.data(), fc1t.data(), fc1b.data(), fc2.data(), fc2b.data());
    const bool ts_only = c->use_ts || c->quad || (c->duo_ctas > 0 && c->duo_always);
    std::vector<uint16_t> ts_tiles;
    int ts_stages = 0;
    if (ts_only || c->duo_ctas > 0) {  // same bias / FC arrays; the conv weights as a stream of 4 KB K = 16 steps
        ts_stages = ts_steps_per_pass(d);
        ts_tiles.assign((size_t)ts_stages * 2048, 0);
        pack_weights_ts(d, blob, ts_tiles.data());
        if (ts_only) {
            stages = ts_stages;
            tiles.swap(ts_tiles);
        }
    }
    const void* src[6] = {tiles.data(), bias.data(), fc1t.data(), fc1b.data(), fc2.data(), fc2b.data()};
    const size_t bytes[6] = {tiles.size() * 2, bias.size() * 4, fc1t.size() * 4, fc1b.size() * 4, fc2.size() * 4,
                             fc2b.size() * 4};
    for (int i = 0; i < 6; ++i) {
        if (c->d_weights[i]) {
            cudaFree(c->d_weights[i]);
            c->d_weights[i] = nullptr;
        }
        NSB_CUDA(cudaMalloc(&c->d_weights[i], bytes[i]));
        NSB_CUDA(cudaMemcpy(c->d_weights[i], src[i], bytes[i], cudaMemcpyHostToDevice));
    }
    DeviceNet& n = c->net;
    n.channels = C;
    n.blocks = d.blocks;
    n.in_channels = d.in_channels;
    n.stem_steps = stem_steps(d.in_channels);
    n.hidden = H;
    n.num_layers = NL;
    n.stages_per_pass = stages;
    n.tiles = static_cast<const uint8_t*>(c->d_weights[0]);
    n.bias = static_cast<const float*>(c->d_weights[1]);
    n.fc1t = static_cast<const float*>(c->d_weights[2]);
    n.fc1b = static_cast<const float*>(c->d_weights[3]);
    n.fc2 = static_cast<const float*>(c->d_weights[4]);
    n.fc2b = static_cast<const float*>(c->d_weights[5]);
    if (c->duo_ctas > 0 && !c->duo_always) {  // both kernels: a second weight stream beside the first
        cudaFree(c->d_duo_tiles);
        c->d_duo_tiles = nullptr;
        NSB_CUDA(cudaMalloc(&c->d_duo_tiles, ts_tiles.size() * 2));
        NSB_CUDA(cudaMemcpy(c->d_duo_tiles, ts_tiles.data(), ts_tiles.size() * 2, cudaMemcpyHostToDevice));
        c->net_duo = n;
        c->net_duo.stages_per_pass = ts_stages;
        c->net_duo.tiles = static_cast<const uint8_t*>(c->d_duo_tiles);
    } else {
        c->net_duo = n;
    }
    c->loaded = true;
    return calibrate_kernel_choice(c);
}

// One-slot 128-channel contexts hold both trunk kernels and choose per batch from three launch durations: trunk_fused.cu
// per wave of one CTA per SM (2 positions each), trunk_duo_kernel while at most one CTA per SM is resident, and
// trunk_duo_kernel per wave of two co-resident CTAs per SM.  The durations are measured at nsb_load_weights on this
// device with this net (calibrate_kernel_choice); the initial values (10 x 128 on a B200 at full clocks) only serve
// contexts whose batch_max is too small for the choice to exist.
static bool use_duo(const nsb_ctx* c, int n) {
    if (c->duo_ctas <= 0) return false;
    if (c->duo_always) return true;
    const int groups = (n + 1) / 2, sms = c->num_sms;
    const double classic = c->t_classic_wave * ((groups + sms - 1) / sms);
    const int full = groups / (2 * sms), rest = groups % (2 * sms);  // waves of co-resident pairs, then the remainder
    const double duo = c->t_duo_pair * full + (rest == 0 ? 0.0 : rest <= sms ? c->t_duo_single : c->t_duo_pair);
    return duo < classic;  // in effect: more than one CTA per SM worth of position pairs
}

// Times the two 128-channel kernels on empty boards (the kernels' duration does not depend on the data): best of three
// launches after a warm-up each, CUDA events on slot 0's stream.  ~12 launches, once per nsb_load_weights.
static int calibrate_kernel_choice(nsb_ctx* c) {
    const int sms = c->num_sms;
    if (c->duo_ctas <= 0 || c->duo_always || c->batch_max <= 2 * sms) return 0;  // one wave of trunk_fused.cu: no choice to make
    Slot& s = c->slots[0];
    const int n_wave = 2 * sms, n_pair = c->batch_max < 4 * sms ? c->batch_max : 4 * sms;
    NSB_CUDA(cudaMemsetAsync(s.d_feat, 0, (size_t)n_pair * c->desc.in_channels * sizeof(nsb_feature_bitboard), s.stream));
    cudaEvent_t e0, e1;
    NSB_CUDA(cudaEventCreate(&e0));
    NSB_CUDA(cudaEventCreate(&e1));
    auto best_of = [&](bool duo, int n, double* out) -> int {
        EvalArgs a{};
        a.features = s.d_feat;
        a.n = n;
        a.win = s.d_win;
        a.draw = s.d_draw;
        float best = 1e30f;
        for (int it = 0; it < 4; ++it) {
            NSB_CUDA(cudaEventRecord(e0, s.stream));
            const int k = duo ? launch_trunk_duo(c->net_duo, a, sms, c->duo_ctas, s.stream) : launch_trunk_fused(c->net, a, sms, s.stream);
            if (k < 0) return k;
            NSB_CUDA(cudaGetLastError());
            NSB_CUDA(cudaEventRecord(e1, s.stream));
            NSB_CUDA(cudaEventSynchronize(e1));
            float ms = 0.f;
            NSB_CUDA(cudaEventElapsedTime(&ms, e0, e1));
            if (it > 0 && ms < best) best = ms;
        }
        *out = best;
        return 0;
    };
    int rc = best_of(false, n_wave, &c->t_classic_wave);
    if (!rc) rc = best_of(true, n_wave, &c->t_duo_single);
    if (!rc) rc = best_of(true, n_pair, &c->t_duo_pair);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    c->calibrated = rc == 0;
    return rc;
}

/* ---- shared launch helper ------------------------------------------------------------------ */

static int run_trunk(nsb_ctx* c, Slot& s, const EvalArgs& a) {
    if (c->timing) {
        while (s.ev.size() < s.ev_used + 2) {
            cudaEvent_t e;
            NSB_CUDA(cudaEventCreate(&e));
            s.ev.push_back(e);
        }
        NSB_CUDA(cudaEventRecord(s.ev[s.ev_used], s.stream));
    }
    int k = c->max_pairs > 0 ? launch_trunk_pair(c->net, a, c->max_pairs, s.stream)
            : c->quad        ? launch_trunk_quad(c->net, a, c->num_sms, s.stream)
            : use_duo(c, a.n) ? launch_trunk_duo(c->net_duo, a, c->num_sms, c->duo_ctas, s.stream)
#ifdef NSB_DIAG
            : c->use_ts      ? launch_trunk_ts(c->net, a, c->num_sms, s.stream)
#endif
                             : launch_trunk_fused(c->net, a, c->num_sms, s.stream, c->cluster128);
    if (k < 0) return k;
    NSB_CUDA(cudaGetLastError());
    c->launches += (uint64_t)k;
    if (c->timing) {
        NSB_CUDA(cudaEventRecord(s.ev[s.ev_used + 1], s.stream));
        s.ev_used += 2;
    }
    return 0;
}

static int harvest_timing(nsb_ctx* c, Slot& s) {
    for (size_t i = 0; i + 1 < s.ev_used; i += 2) {
        float ms = 0.f;
        NSB_CUDA(cudaEventElapsedTime(&ms, s.ev[i], s.ev[i + 1]));
        c->trunk_ms += ms;
        c->trunk_launches += 1;
    }
    s.ev_used = 0;
    return 0;
}

/* ---- the Infer contract -------------------------------------------------------------------- */

int nsb_eval_async(nsb_ctx* c, int slot, const nsb_feature_bitboard* features, size_t n, float* policy,
                   float* win, float* draw) {
    int rc = check_ctx(c, slot);
    if (rc) return rc;
    if ((rc = check_batch(c, n, true))) return rc;
    if (!features || !policy || !win || !draw) {
        set_error("nsb_eval_async: null buffer");
        return NSB_ERR_INVALID;
    }
    if (n == 0) return 0;
    Slot& s = c->slots[slot];
    if (c->direct_io && host_mapped(features, n * (size_t)c->desc.in_channels * sizeof(nsb_feature_bitboard)) &&
        dense_outputs_mapped(n, policy, win, draw)) {
        EvalArgs a{};
        a.features = features;
        a.n = (int)n;
        a.policy = policy;
        a.win = win;
        a.draw = draw;
        return run_trunk(c, s, a);
    }
    NSB_CUDA(cudaMemcpyAsync(s.d_feat, features, n * (size_t)c->desc.in_channels * sizeof(nsb_feature_bitboard),
                             cudaMemcpyHostToDevice, s.stream));  // trt.cc:240-242
    EvalArgs a{};
    a.features = s.d_feat;
    a.n = (int)n;
    a.policy = s.d_policy;
    a.win = s.d_win;
    a.draw = s.d_draw;
    if ((rc = run_trunk(c, s, a))) return rc;
    NSB_CUDA(cudaMemcpyAsync(policy, s.d_policy, n * kPolicySize * sizeof(float), cudaMemcpyDeviceToHost,
                             s.stream));  // trt.cc:265-271
    NSB_CUDA(cudaMemcpyAsync(win, s.d_win, n * sizeof(float), cudaMemcpyDeviceToHost, s.stream));
    NSB_CUDA(cudaMemcpyAsync(draw, s.d_draw, n * sizeof(float), cudaMemcpyDeviceToHost, s.stream));
    return 0;
}

static bool decode_buffers_mapped(size_t n, size_t total, const uint32_t* move_off, const uint16_t* move_idx,
                                  const float* legal_out, const float* win, const float* draw, const uint8_t* nan_flag) {
    return host_mapped(move_off, (n + 1) * sizeof(uint32_t)) && host_mapped(move_idx, (total ? total : 1) * sizeof(uint16_t)) &&
           host_mapped(legal_out, (total ? total : 1) * sizeof(float)) && host_mapped(win, n * sizeof(float)) &&
           host_mapped(draw, n * sizeof(float)) && (nan_flag == nullptr || host_mapped(nan_flag, n));
}

// Stage 1 for a batch whose packed positions are already in s.d_pos: either it is left to the trunk
// kernel's prologue (*fused = s.d_pos; the bitboards never exist in HBM, SURVEY.md §8 f2), or the
// standalone pack kernel fills s.d_feat (*fused = nullptr).
static int stage1(nsb_ctx* c, Slot& s, size_t n, const nsb_position** fused) {
    if (c->fuse_pack) {
        *fused = s.d_pos;
        return 0;
    }
    *fused = nullptr;
    int k = launch_pack_positions(s.d_pos, n, s.d_feat, s.stream);
    if (k < 0) return k;
    NSB_CUDA(cudaGetLastError());
    c->launches += (uint64_t)k;
    return 0;
}

static int eval_request(nsb_ctx* c, int slot, const nsb_decode_request& r, const char* who);

int nsb_eval_request_async(nsb_ctx* c, int slot, const nsb_decode_request* request) {
    if (!request) {
        set_error("nsb_eval_request_async: null request");
        return NSB_ERR_INVALID;
    }
    return eval_request(c, slot, *request, "nsb_eval_request_async");
}

int nsb_eval_decode_async(nsb_ctx* c, int slot, const nsb_feature_bitboard* features, size_t n,
                          const uint32_t* move_off, const uint16_t* move_idx, int mode, float* legal_out,
                          float* win, float* draw, uint8_t* nan_flag) {
    nsb_decode_request r{};
    r.features = features;
    r.n = n;
    r.move_off = move_off;
    r.move_idx = move_idx;
    r.mode = mode;
    r.legal_out = legal_out;
    r.win = win;
    r.draw = draw;
    r.nan_flag = nan_flag;
    if (!features) {
        set_error("nsb_eval_decode_async: null buffer or bad mode");
        return NSB_ERR_INVALID;
    }
    return eval_request(c, slot, r, "nsb_eval_decode_async");
}

int nsb_eval_positions_async(nsb_ctx* c, int slot, const nsb_position* positions, size_t n, float* policy,
                             float* win, float* draw) {
    int rc = check_ctx(c, slot);
    if (rc) return rc;
    if ((rc = check_batch(c, n, true))) return rc;
    if (!positions || !policy || !win || !draw) {
        set_error("nsb_eval_positions_async: null buffer");
        return NSB_ERR_INVALID;
    }
    if ((rc = check_positions_net(c, "nsb_eval_positions_async"))) return rc;
    if (n == 0) return 0;
    Slot& s = c->slots[slot];
    if (c->direct_io && c->fuse_pack && host_mapped(positions, n * sizeof(nsb_position)) &&
        dense_outputs_mapped(n, policy, win, draw)) {
        EvalArgs a{};
        a.positions = positions;
        a.n = (int)n;
        a.policy = policy;
        a.win = win;
        a.draw = draw;
        return run_trunk(c, s, a);
    }
    NSB_CUDA(cudaMemcpyAsync(s.d_pos, positions, n * sizeof(nsb_position), cudaMemcpyHostToDevice, s.stream));
    const nsb_position* fused = nullptr;
    if ((rc = stage1(c, s, n, &fused))) return rc;
    EvalArgs a{};
    a.features = s.d_feat;
    a.positions = fused;
    a.n = (int)n;
    a.policy = s.d_policy;
    a.win = s.d_win;
    a.draw = s.d_draw;
    if ((rc = run_trunk(c, s, a))) return rc;
    NSB_CUDA(cudaMemcpyAsync(policy, s.d_policy, n * kPolicySize * sizeof(float), cudaMemcpyDeviceToHost, s.stream));
    NSB_CUDA(cudaMemcpyAsync(win, s.d_win, n * sizeof(float), cudaMemcpyDeviceToHost, s.stream));
    NSB_CUDA(cudaMemcpyAsync(draw, s.d_draw, n * sizeof(float), cudaMemcpyDeviceToHost, s.stream));
    return 0;
}

int nsb_eval_positions_decode_async(nsb_ctx* c, int slot, const nsb_position* positions, size_t n,
                                    const uint32_t* move_off, const uint16_t* move_idx, int mode,
                                    float* legal_out, float* win, float* draw, uint8_t* nan_flag) {
    nsb_decode_request r{};
    r.positions = positions;
    r.n = n;
    r.move_off = move_off;
    r.move_idx = move_idx;
    r.mode = mode;
    r.legal_out = legal_out;
    r.win = win;
    r.draw = draw;
    r.nan_flag = nan_flag;
    if (!positions) {
        set_error("nsb_eval_positions_decode_async: null buffer or bad mode");
        return NSB_ERR_INVALID;
    }
    return eval_request(c, slot, r, "nsb_eval_positions_decode_async");
}

int nsb_await(nsb_ctx* c, int slot) {
    int rc = check_ctx(c, slot);
    if (rc) return rc;
    Slot& s = c->slots[slot];
    NSB_CUDA(cudaStreamSynchronize(s.stream));  // trt.cc:281-283
    return harvest_timing(c, s);
}

int nsb_is_computing(nsb_ctx* c, int slot) {
    int rc = check_ctx(c, slot);
    if (rc) return rc;
    cudaError_t e = cudaStreamQuery(c->slots[slot].stream);  // trt.cc:285-287
    if (e == cudaSuccess) return 0;
    if (e == cudaErrorNotReady) return 1;
    set_error("cudaStreamQuery failed: %s", cudaGetErrorString(e));
    return NSB_ERR_CUDA;
}

/* ---- device-resident entry points ----------------------------------------------------------- */

int nsb_eval_device(nsb_ctx* c, int slot, const nsb_feature_bitboard* d_features, size_t n, float* d_policy,
                    float* d_win, float* d_draw) {
    int rc = check_ctx(c, slot);
    if (rc) return rc;
    if (n > 65535u * 64u) {
        set_error("nsb_eval_device: n too large");
        return NSB_ERR_INVALID;
    }
    if (!c->loaded) {
        set_error("weights not loaded");
        return NSB_ERR_STATE;
    }
    if (!d_features || !d_win || !d_draw) {
        set_error("nsb_eval_device: null buffer");
        return NSB_ERR_INVALID;
    }
    if (n == 0) return 0;
    EvalArgs a{};
    a.features = d_features;
    a.n = (int)n;
    a.policy = d_policy;
    a.win = d_win;
    a.draw = d_draw;
    return run_trunk(c, c->slots[slot], a);
}

int nsb_eval_decode_device(nsb_ctx* c, int slot, const nsb_feature_bitboard* d_features, size_t n,
                           const uint32_t* d_move_off, const uint16_t* d_move_idx, int mode, float* d_policy,
                           float* d_legal_out, float* d_win, float* d_draw, uint8_t* d_nan_flag) {
    int rc = check_ctx(c, slot);
    if (rc) return rc;
    if (!c->loaded) {
        set_error("weights not loaded");
        return NSB_ERR_STATE;
    }
    if (!d_features || !d_win || !d_draw || !d_move_off || !d_move_idx || !d_legal_out || !mode_ok(mode)) {
        set_error("nsb_eval_decode_device: null buffer or bad mode");
        return NSB_ERR_INVALID;
    }
    if (n == 0) return 0;
    EvalArgs a{};
    a.features = d_features;
    a.n = (int)n;
    a.policy = d_policy;
    a.win = d_win;
    a.draw = d_draw;
    a.move_off = d_move_off;
    a.move_idx = d_move_idx;
    a.legal_out = d_legal_out;
    a.nan_flag = d_nan_flag;
    a.decode_mode = mode;
    return run_trunk(c, c->slots[slot], a);
}

/* ---- device-resident evaluation cache (reference src/mcts/evalcache.{h,cc}) -------------------- */

int nsb_cache_create(nsb_ctx* c, size_t memory_mb) {
    int rc = check_ctx(c, 0);
    if (rc) return rc;
    if (memory_mb == 0 || memory_mb > 160 * 1024) {
        set_error("nsb_cache_create: memory_mb must be in 1..163840");
        return NSB_ERR_INVALID;
    }
    if (c->cache.num_bundles) {
        set_error("nsb_cache_create: this ctx already has a cache");
        return NSB_ERR_STATE;
    }
    NSB_CUDA(cudaSetDevice(c->gpu));
    // evalcache.cc:17-19: NumBundle = MemorySize MiB / (entry size * bundle size)
    const unsigned long long bundles = (unsigned long long)memory_mb * 1024ull * 1024ull / (3ull * sizeof(CacheEntry) + 4ull);
    DeviceCache dc{};
    dc.num_bundles = bundles;
    cudaError_t e = cudaMalloc(&dc.entries, bundles * 3ull * sizeof(CacheEntry));
    if (e == cudaSuccess) e = cudaMalloc(&dc.meta, bundles * sizeof(uint32_t));
    const size_t B = (size_t)c->batch_max;
    for (auto& s : c->slots) {
        if (e == cudaSuccess) e = cudaMalloc(&s.d_hash, B * sizeof(uint64_t));
        if (e == cudaSuccess) e = cudaMalloc(&s.d_hit, B);
        if (e == cudaSuccess) e = cudaMalloc(&s.d_miss_idx, B * sizeof(int));
        if (e == cudaSuccess) e = cudaMalloc(&s.d_miss_count, sizeof(int));
    }
    if (e != cudaSuccess) {
        cudaFree(dc.entries);
        cudaFree(dc.meta);
        set_error("nsb_cache_create: device allocation of %zu MiB failed: %s", memory_mb, cudaGetErrorString(e));
        return e == cudaErrorMemoryAllocation ? NSB_ERR_NOMEM : NSB_ERR_CUDA;
    }
    c->cache = dc;
    c->cache_owned = true;
    return nsb_cache_clear(c);
}

int nsb_cache_attach(nsb_ctx* c, nsb_ctx* owner) {
    int rc = check_ctx(c, 0);
    if (rc) return rc;
    if (!owner || owner == c || !owner->cache.num_bundles || owner->gpu != c->gpu) {
        set_error("nsb_cache_attach: the owner must be another ctx of the same device that has a cache");
        return NSB_ERR_INVALID;
    }
    if (c->cache.num_bundles) {
        set_error("nsb_cache_attach: this ctx already has a cache");
        return NSB_ERR_STATE;
    }
    NSB_CUDA(cudaSetDevice(c->gpu));
    const size_t B = (size_t)c->batch_max;
    cudaError_t e = cudaSuccess;
    for (auto& s : c->slots) {
        if (e == cudaSuccess) e = cudaMalloc(&s.d_hash, B * sizeof(uint64_t));
        if (e == cudaSuccess) e = cudaMalloc(&s.d_hit, B);
        if (e == cudaSuccess) e = cudaMalloc(&s.d_miss_idx, B * sizeof(int));
        if (e == cudaSuccess) e = cudaMalloc(&s.d_miss_count, sizeof(int));
    }
    if (e != cudaSuccess) {
        set_error("nsb_cache_attach: device allocation failed: %s", cudaGetErrorString(e));
        return e == cudaErrorMemoryAllocation ? NSB_ERR_NOMEM : NSB_ERR_CUDA;
    }
    c->cache = owner->cache;  // the bundles' lock words make concurrent kernels of several contexts safe
    c->cache_owned = false;
    return 0;
}

int nsb_cache_clear(nsb_ctx* c) {
    int rc = check_ctx(c, 0);
    if (rc) return rc;
    if (!c->cache.num_bundles) {
        set_error("nsb_cache_clear: no cache (call nsb_cache_create)");
        return NSB_ERR_STATE;
    }
    for (auto& s : c->slots) NSB_CUDA(cudaStreamSynchronize(s.stream));
    int k = launch_cache_clear(c->cache, c->slots[0].stream);
    NSB_CUDA(cudaGetLastError());
    c->launches += (uint64_t)k;
    NSB_CUDA(cudaStreamSynchronize(c->slots[0].stream));
    return 0;
}

const char* nsb_trunk_kernel_name(nsb_ctx* c) {
    if (!c) return "";
    if (c->max_pairs > 0)
        return c->desc.channels == 192 ? "trunk_pair_kernel (192 ch, cta_group::2 CTA pair, Cout halves padded to 128 rows)"
                                       : "trunk_pair_kernel (256 ch, cta_group::2 CTA pair)";
    if (c->quad) return "trunk_quad_kernel (128 ch, 4 positions per CTA, weights via TMEM, 1 CTA per SM)";
    if (c->duo_ctas > 0 && c->duo_always) {
        static thread_local char name[96];
        snprintf(name, sizeof name, "trunk_duo_kernel (128 ch, weights via TMEM, %d CTA%s per SM)", c->duo_ctas,
                 c->duo_ctas == 1 ? "" : "s");
        return name;
    }
    if (c->duo_ctas > 0) return "trunk_fused_kernel<128> (trunk_duo_kernel for batches where two CTAs per SM are faster)";
    if (c->use_ts) return "trunk_ts_kernel (128 ch, weights via TMEM, experimental)";
    return c->desc.channels == 128 ? "trunk_fused_kernel<128>" : "trunk_fused_kernel<256>";
}

uint64_t nsb_cache_num_bundles(nsb_ctx* c) { return c ? (uint64_t)c->cache.num_bundles : 0; }

static int check_cache(nsb_ctx* c, int slot, const char* who) {
    int rc = check_ctx(c, slot);
    if (rc) return rc;
    if (!c->cache.num_bundles) {
        set_error("%s: no cache (call nsb_cache_create)", who);
        return NSB_ERR_STATE;
    }
    return 0;
}

int nsb_cache_store_device(nsb_ctx* c, int slot, const uint64_t* d_hashes, size_t n, const uint32_t* d_move_off,
                           const float* d_legal, const float* d_win, const float* d_draw, const uint8_t* d_skip,
                           uint8_t* d_stored) {
    int rc = check_cache(c, slot, "nsb_cache_store_device");
    if (rc) return rc;
    if (!d_hashes || !d_move_off || !d_legal || !d_win || !d_draw) {
        set_error("nsb_cache_store_device: null buffer");
        return NSB_ERR_INVALID;
    }
    int k = launch_cache_store(c->cache, d_hashes, n, d_move_off, d_legal, d_win, d_draw, d_skip, d_stored,
                               c->slots[slot].stream);
    NSB_CUDA(cudaGetLastError());
    c->launches += (uint64_t)k;
    return 0;
}

int nsb_cache_probe_device(nsb_ctx* c, int slot, const uint64_t* d_hashes, size_t n, const uint32_t* d_move_off,
                           float* d_legal_out, float* d_win, float* d_draw, uint8_t* d_hit, int* d_miss_idx,
                           int* d_miss_count) {
    int rc = check_cache(c, slot, "nsb_cache_probe_device");
    if (rc) return rc;
    if (!d_hashes || !d_move_off || !d_legal_out || !d_win || !d_draw || !d_hit || !d_miss_idx || !d_miss_count) {
        set_error("nsb_cache_probe_device: null buffer");
        return NSB_ERR_INVALID;
    }
    Slot& s = c->slots[slot];
    NSB_CUDA(cudaMemsetAsync(d_miss_count, 0, sizeof(int), s.stream));
    int k = launch_cache_probe(c->cache, d_hashes, n, d_move_off, d_legal_out, d_win, d_draw, d_hit, nullptr, d_miss_idx,
                               d_miss_count, s.stream);
    NSB_CUDA(cudaGetLastError());
    c->launches += (uint64_t)k;
    return 0;
}

// probe -> trunk on the misses (fused decode + fused store); everything on the slot's stream
static int eval_cached_enqueue(nsb_ctx* c, Slot& s, const nsb_feature_bitboard* d_features,
                               const nsb_position* d_positions, size_t n,
                               const uint64_t* d_hashes, const uint32_t* d_off, const uint16_t* d_idx, int mode,
                               float* d_legal, float* d_win, float* d_draw, uint8_t* d_nan_flag, uint8_t* d_hit) {
    NSB_CUDA(cudaMemsetAsync(s.d_miss_count, 0, sizeof(int), s.stream));
    int k = launch_cache_probe(c->cache, d_hashes, n, d_off, d_legal, d_win, d_draw, d_hit, d_nan_flag, s.d_miss_idx,
                               s.d_miss_count, s.stream, nullptr, mode);
    NSB_CUDA(cudaGetLastError());
    c->launches += (uint64_t)k;
    EvalArgs a{};
    a.features = d_features;
    a.positions = d_positions;  // set: stage 1 runs in the trunk prologue, for the misses only
    a.n = (int)n;
    a.win = d_win;
    a.draw = d_draw;
    a.move_off = d_off;
    a.move_idx = d_idx;
    a.legal_out = d_legal;
    a.nan_flag = d_nan_flag;
    a.decode_mode = mode;
    a.index = s.d_miss_idx;
    a.count = s.d_miss_count;
    a.hashes = d_hashes;
    a.cache = c->cache;
    return run_trunk(c, s, a);
}

int nsb_eval_cached_decode_device(nsb_ctx* c, int slot, const nsb_feature_bitboard* d_features, size_t n,
                                  const uint64_t* d_hashes, const uint32_t* d_move_off, const uint16_t* d_move_idx,
                                  int mode, float* d_legal_out, float* d_win, float* d_draw, uint8_t* d_nan_flag,
                                  uint8_t* d_hit) {
    int rc = check_cache(c, slot, "nsb_eval_cached_decode_device");
    if (rc) return rc;
    if ((rc = check_batch(c, n, true))) return rc;
    if (!d_features || !d_hashes || !d_move_off || !d_move_idx || !d_legal_out || !d_win || !d_draw || !d_hit ||
        !mode_ok(mode)) {
        set_error("nsb_eval_cached_decode_device: null buffer or bad mode");
        return NSB_ERR_INVALID;
    }
    if (n == 0) return 0;
    return eval_cached_enqueue(c, c->slots[slot], d_features, nullptr, n, d_hashes, d_move_off, d_move_idx, mode, d_legal_out, d_win,
                               d_draw, d_nan_flag, d_hit);
}

int nsb_eval_cached_decode_async(nsb_ctx* c, int slot, const nsb_feature_bitboard* features, size_t n,
                                 const uint64_t* hashes, const uint32_t* move_off, const uint16_t* move_idx, int mode,
                                 float* legal_out, float* win, float* draw, uint8_t* nan_flag, uint8_t* hit_flag) {
    nsb_decode_request r{};
    r.features = features;
    r.n = n;
    r.hashes = hashes;
    r.move_off = move_off;
    r.move_idx = move_idx;
    r.mode = mode;
    r.legal_out = legal_out;
    r.win = win;
    r.draw = draw;
    r.nan_flag = nan_flag;
    r.hit_flag = hit_flag;
    int rc = check_cache(c, slot, "nsb_eval_cached_decode_async");
    if (rc) return rc;
    if (!features || !hashes) {
        set_error("nsb_eval_cached_decode_async: null buffer or bad mode");
        return NSB_ERR_INVALID;
    }
    return eval_request(c, slot, r, "nsb_eval_cached_decode_async");
}

int nsb_eval_positions_cached_decode_async(nsb_ctx* c, int slot, const nsb_position* positions, size_t n,
                                           const uint64_t* hashes, const uint32_t* move_off, const uint16_t* move_idx,
                                           int mode, float* legal_out, float* win, float* draw, uint8_t* nan_flag,
                                           uint8_t* hit_flag) {
    nsb_decode_request r{};
    r.positions = positions;
    r.n = n;
    r.hashes = hashes;
    r.move_off = move_off;
    r.move_idx = move_idx;
    r.mode = mode;
    r.legal_out = legal_out;
    r.win = win;
    r.draw = draw;
    r.nan_flag = nan_flag;
    r.hit_flag = hit_flag;
    int rc = check_cache(c, slot, "nsb_eval_positions_cached_decode_async");
    if (rc) return rc;
    if (!positions || !hashes) {
        set_error("nsb_eval_positions_cached_decode_async: null buffer or bad mode");
        return NSB_ERR_INVALID;
    }
    return eval_request(c, slot, r, "nsb_eval_positions_cached_decode_async");
}

// The one implementation behind every host-buffer entry point of the fused path (include/nsb.h,
// nsb_decode_request): bitboards or packed positions in; through the device cache when hashes are given;
// rank order out when asked for.  Direct I/O: when every buffer of the request is mapped page-locked memory
// the kernels work on the caller's buffers themselves; otherwise copy nodes around them (trt.cc:240-242,265-271).
static int eval_request(nsb_ctx* c, int slot, const nsb_decode_request& r, const char* who) {
    int rc = r.hashes ? check_cache(c, slot, who) : check_ctx(c, slot);
    if (rc) return rc;
    const size_t n = r.n;
    if ((rc = check_batch(c, n, true))) return rc;
    if ((r.features != nullptr) == (r.positions != nullptr) || !r.move_off || !r.move_idx || !r.legal_out || !r.win || !r.draw ||
        !mode_ok(r.mode)) {
        set_error("%s: null buffer or bad mode", who);
        return NSB_ERR_INVALID;
    }
    if (r.positions && (rc = check_positions_net(c, who))) return rc;
    if (n == 0) return 0;
    if ((rc = check_offsets(r.move_off, n, who))) return rc;
    const size_t total = r.move_off[n];
    const bool both = (r.mode & NSB_DECODE_MODE_MASK) == NSB_DECODE_BOTH;
    const uint8_t* row_flags = both ? r.row_flags : nullptr;  // the other modes have no per-row variants
    float* logits_out = both ? r.logits_out : nullptr;
    Slot& s = c->slots[slot];
    const size_t in_bytes = r.features ? n * (size_t)c->desc.in_channels * sizeof(nsb_feature_bitboard) : n * sizeof(nsb_position);
    const void* in = r.features ? (const void*)r.features : (const void*)r.positions;

    EvalArgs a{};
    a.n = (int)n;
    a.decode_mode = r.mode;
    const bool direct = c->direct_io && (r.features || c->fuse_pack) && host_mapped(in, in_bytes) &&
                        decode_buffers_mapped(n, total, r.move_off, r.move_idx, r.legal_out, r.win, r.draw, r.nan_flag) &&
                        (!r.hashes || host_mapped(r.hashes, n * sizeof(uint64_t))) && (!r.hit_flag || host_mapped(r.hit_flag, n)) &&
                        (!r.order_out || host_mapped(r.order_out, (total ? total : 1) * sizeof(uint16_t))) &&
                        (!row_flags || host_mapped(row_flags, n)) &&
                        (!logits_out || host_mapped(logits_out, (total ? total : 1) * sizeof(float)));
    const uint64_t* hashes = r.hashes;
    uint8_t* hit = r.hit_flag ? r.hit_flag : s.d_hit;
    if (direct) {
        a.features = r.features;
        a.positions = r.positions;
        a.win = r.win;
        a.draw = r.draw;
        a.move_off = r.move_off;
        a.move_idx = r.move_idx;
        a.legal_out = r.legal_out;
        a.order_out = r.order_out;
        a.nan_flag = r.nan_flag ? r.nan_flag : (r.hashes ? s.d_flag : nullptr);
        a.row_flags = row_flags;
        a.logits_out = logits_out;
    } else {
        NSB_CUDA(cudaMemcpyAsync(r.features ? (void*)s.d_feat : (void*)s.d_pos, in, in_bytes, cudaMemcpyHostToDevice, s.stream));
        a.features = s.d_feat;
        if (r.positions && (rc = stage1(c, s, n, &a.positions))) return rc;
        if (r.hashes) {
            NSB_CUDA(cudaMemcpyAsync(s.d_hash, r.hashes, n * sizeof(uint64_t), cudaMemcpyHostToDevice, s.stream));
            hashes = s.d_hash;
            hit = s.d_hit;
        }
        NSB_CUDA(cudaMemcpyAsync(s.d_off, r.move_off, (n + 1) * sizeof(uint32_t), cudaMemcpyHostToDevice, s.stream));
        if (total)
            NSB_CUDA(cudaMemcpyAsync(s.d_idx, r.move_idx, total * sizeof(uint16_t), cudaMemcpyHostToDevice, s.stream));
        a.win = s.d_win;
        a.draw = s.d_draw;
        a.move_off = s.d_off;
        a.move_idx = s.d_idx;
        a.legal_out = s.d_legal;
        a.order_out = r.order_out ? s.d_order : nullptr;
        a.nan_flag = s.d_flag;
        if (row_flags) {
            NSB_CUDA(cudaMemcpyAsync(s.d_rowflags, row_flags, n, cudaMemcpyHostToDevice, s.stream));
            a.row_flags = s.d_rowflags;
        }
        if (logits_out) {
            if (!s.d_logits) NSB_CUDA(cudaMalloc(&s.d_logits, (size_t)c->batch_max * NSB_MAX_LEGAL_MOVES * sizeof(float)));
            a.logits_out = s.d_logits;
        }
    }
    if (r.hashes) {
        NSB_CUDA(cudaMemsetAsync(s.d_miss_count, 0, sizeof(int), s.stream));
        int k = launch_cache_probe(c->cache, hashes, n, a.move_off, a.legal_out, a.win, a.draw, hit, a.nan_flag, s.d_miss_idx,
                                   s.d_miss_count, s.stream, a.order_out, r.mode, a.row_flags, a.logits_out);
        NSB_CUDA(cudaGetLastError());
        c->launches += (uint64_t)k;
        a.index = s.d_miss_idx;   // the trunk launch works on the probe's miss list and stores what it decodes
        a.count = s.d_miss_count;
        a.hashes = hashes;
        a.cache = c->cache;
    }
    if ((rc = run_trunk(c, s, a))) return rc;
    if (direct) return 0;
    if (total) {
        NSB_CUDA(cudaMemcpyAsync(r.legal_out, s.d_legal, total * sizeof(float), cudaMemcpyDeviceToHost, s.stream));
        if (r.order_out)
            NSB_CUDA(cudaMemcpyAsync(r.order_out, s.d_order, total * sizeof(uint16_t), cudaMemcpyDeviceToHost, s.stream));
        if (logits_out)
            NSB_CUDA(cudaMemcpyAsync(logits_out, s.d_logits, total * sizeof(float), cudaMemcpyDeviceToHost, s.stream));
    }
    NSB_CUDA(cudaMemcpyAsync(r.win, s.d_win, n * sizeof(float), cudaMemcpyDeviceToHost, s.stream));
    NSB_CUDA(cudaMemcpyAsync(r.draw, s.d_draw, n * sizeof(float), cudaMemcpyDeviceToHost, s.stream));
    if (r.nan_flag) NSB_CUDA(cudaMemcpyAsync(r.nan_flag, s.d_flag, n, cudaMemcpyDeviceToHost, s.stream));
    if (r.hashes && r.hit_flag) NSB_CUDA(cudaMemcpyAsync(r.hit_flag, s.d_hit, n, cudaMemcpyDeviceToHost, s.stream));
    return 0;
}

#ifdef NSB_DIAG
static int debug_timeline(nsb_ctx* c, int slot, const nsb_feature_bitboard* d_features, const nsb_position* d_positions,
                          size_t n, uint64_t* host_stamps, size_t max_stamps) {
    int rc = check_ctx(c, slot);
    if (rc) return rc;
    if (!c->loaded || (!d_features && !d_positions) || !host_stamps || n == 0) {
        set_error("nsb_debug_trunk_timeline: bad arguments or weights not loaded");
        return NSB_ERR_INVALID;
    }
    // 4 per layer + 16 phase stamps + per CTA {SM id, globaltimer at start, at end} for up to 1,024 CTAs (trunk_tmem.cu)
    const size_t need = (size_t)c->net.num_layers * 4 + 16 + 3 * 1024;
    if (max_stamps < need) {
        set_error("nsb_debug_trunk_timeline: need room for %zu stamps", need);
        return NSB_ERR_INVALID;
    }
    Slot& s = c->slots[slot];
    unsigned long long* d_t = nullptr;
    NSB_CUDA(cudaMalloc(&d_t, need * 8));
    NSB_CUDA(cudaMemsetAsync(d_t, 0, need * 8, s.stream));
    EvalArgs a{};
    a.features = d_features;
    a.positions = d_positions;
    a.n = (int)n;
    a.policy = s.d_policy;
    a.win = s.d_win;
    a.draw = s.d_draw;
    a.timeline = d_t;
    if (n > (size_t)c->batch_max) {
        cudaFree(d_t);
        set_error("nsb_debug_trunk_timeline: n exceeds batch_max");
        return NSB_ERR_INVALID;
    }
    rc = run_trunk(c, s, a);
    if (rc == 0) {
        cudaError_t e = cudaStreamSynchronize(s.stream);
        if (e == cudaSuccess) e = cudaMemcpy(host_stamps, d_t, need * 8, cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) {
            set_error("nsb_debug_trunk_timeline: %s", cudaGetErrorString(e));
            rc = NSB_ERR_CUDA;
        }
    }
    cudaFree(d_t);
    return rc;
}

int nsb_debug_trunk_timeline(nsb_ctx* c, int slot, const nsb_feature_bitboard* d_features, size_t n,
                             uint64_t* host_stamps, size_t max_stamps) {
    return debug_timeline(c, slot, d_features, nullptr, n, host_stamps, max_stamps);
}

int nsb_debug_trunk_timeline_positions(nsb_ctx* c, int slot, const nsb_position* d_positions, size_t n,
                                       uint64_t* host_stamps, size_t max_stamps) {
    return debug_timeline(c, slot, nullptr, d_positions, n, host_stamps, max_stamps);
}

#endif  // NSB_DIAG

int nsb_extract_device(nsb_ctx* c, int slot, const nsb_feature_bitboard* d_features, size_t n, int channels,
                       int channels_first, float* d_planes) {
    int rc = check_ctx(c, slot);
    if (rc) return rc;
    if (!d_features || !d_planes || channels < 1 || channels > 1024) {
        set_error("nsb_extract_device: bad arguments");
        return NSB_ERR_INVALID;
    }
    int k = launch_extract(d_features, n, channels, channels_first, d_planes, c->slots[slot].stream);
    if (k < 0) return k;
    NSB_CUDA(cudaGetLastError());
    c->launches += (uint64_t)k;
    return 0;
}

int nsb_pack_positions_device(nsb_ctx* c, int slot, const nsb_position* d_positions, size_t n,
                              nsb_feature_bitboard* d_features) {
    int rc = check_ctx(c, slot);
    if (rc) return rc;
    if (!d_positions || !d_features) {
        set_error("nsb_pack_positions_device: null buffer");
        return NSB_ERR_INVALID;
    }
    int k = launch_pack_positions(d_positions, n, d_features, c->slots[slot].stream);
    if (k < 0) return k;
    NSB_CUDA(cudaGetLastError());
    c->launches += (uint64_t)k;
    return 0;
}

int nsb_decode_device(nsb_ctx* c, int slot, const float* d_policy, const float* d_win, const float* d_draw,
                      size_t n, const uint32_t* d_move_off, const uint16_t* d_move_idx, int mode,
                      float* d_legal_out, uint8_t* d_nan_flag) {
    int rc = check_ctx(c, slot);
    if (rc) return rc;
    return nsb_decode_device_ex(c, slot, d_policy, d_win, d_draw, n, d_move_off, d_move_idx, mode, nullptr, d_legal_out,
                                nullptr, d_nan_flag);
}

int nsb_decode_device_ex(nsb_ctx* c, int slot, const float* d_policy, const float* d_win, const float* d_draw,
                         size_t n, const uint32_t* d_move_off, const uint16_t* d_move_idx, int mode,
                         const uint8_t* d_row_flags, float* d_legal_out, float* d_logits_out, uint8_t* d_nan_flag) {
    int rc = check_ctx(c, slot);
    if (rc) return rc;
    if (!d_policy || !d_win || !d_draw || !d_move_off || !d_move_idx || !d_legal_out || !mode_ok(mode)) {
        set_error("nsb_decode_device: null buffer or bad mode");
        return NSB_ERR_INVALID;
    }
    int k = launch_decode(d_policy, d_win, d_draw, n, d_move_off, d_move_idx, mode, d_legal_out, d_nan_flag,
                          c->slots[slot].stream, d_row_flags, d_logits_out);
    if (k < 0) return k;
    NSB_CUDA(cudaGetLastError());
    c->launches += (uint64_t)k;
    return 0;
}

void* nsb_stream(nsb_ctx* c, int slot) {
    if (check_ctx(c, slot)) return nullptr;
    return c->slots[slot].stream;
}

int nsb_set_timing(nsb_ctx* c, int enabled) {
    if (!c) {
        set_error("null ctx");
        return NSB_ERR_INVALID;
    }
    c->timing = enabled != 0;
    return 0;
}

int nsb_trunk_time(nsb_ctx* c, double* sum_ms, uint64_t* launches) {
    if (!c) {
        set_error("null ctx");
        return NSB_ERR_INVALID;
    }
    if (sum_ms) *sum_ms = c->trunk_ms;
    if (launches) *launches = c->trunk_launches;
    return 0;
}

int nsb_trunk_time_reset(nsb_ctx* c) {
    if (!c) {
        set_error("null ctx");
        return NSB_ERR_INVALID;
    }
    c->trunk_ms = 0.0;
    c->trunk_launches = 0;
    return 0;
}

uint64_t nsb_launch_count(nsb_ctx* c) { return c ? c->launches : 0; }

/* ---- misc ------------------------------------------------------------------------------------ */

int nsb_host_alloc(void** out, size_t bytes) {
    if (!out) return NSB_ERR_INVALID;
    NSB_CUDA(cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocPortable | cudaHostAllocMapped));
    std::lock_guard<std::mutex> lock(g_host_mu);
    g_host_allocs[(uintptr_t)*out] = HostRange{bytes ? bytes : 1, true, HostKind::Alloc};
    return 0;
}
int nsb_host_alloc_near(void** out, size_t bytes, int gpu) {
    if (!out) return NSB_ERR_INVALID;
    int node = -1;
    void* p = alloc_near_gpu(bytes ? bytes : 1, gpu, &node);
    if (!p) {
        set_error("nsb_host_alloc_near: mmap of %zu bytes failed", bytes);
        return NSB_ERR_NOMEM;
    }
    const cudaError_t e = cudaHostRegister(p, bytes ? bytes : 1, cudaHostRegisterPortable | cudaHostRegisterMapped);
    if (e != cudaSuccess) {
        cudaGetLastError();
        free_near_gpu(p, bytes ? bytes : 1);
        set_error("nsb_host_alloc_near: cudaHostRegister failed: %s", cudaGetErrorString(e));
        return NSB_ERR_CUDA;
    }
    void* dp = nullptr;
    const bool direct = cudaHostGetDevicePointer(&dp, p, 0) == cudaSuccess && dp == p;
    if (!direct) cudaGetLastError();
    std::lock_guard<std::mutex> lock(g_host_mu);
    g_host_allocs[(uintptr_t)p] = HostRange{bytes ? bytes : 1, direct, HostKind::NodeAlloc};
    *out = p;
    return 0;
}
int nsb_gpu_numa_node(int gpu) { return gpu_numa_node(gpu); }
int nsb_numa_bind_thread(int gpu) { return numa_bind_thread_to_gpu(gpu); }
int nsb_host_free(void* p) {
    HostRange r{};
    bool known = false;
    {
        std::lock_guard<std::mutex> lock(g_host_mu);
        auto it = g_host_allocs.find((uintptr_t)p);
        if (it != g_host_allocs.end()) {
            r = it->second;
            known = true;
            g_host_allocs.erase(it);
        }
    }
    if (known && r.kind == HostKind::NodeAlloc) {
        NSB_CUDA(cudaHostUnregister(p));
        free_near_gpu(p, r.bytes);
        return 0;
    }
    NSB_CUDA(cudaFreeHost(p));
    return 0;
}
// The registry entry that covers [p, p + bytes), if any (caller holds g_host_mu).
static std::map<uintptr_t, HostRange>::iterator host_find_locked(const void* p, size_t bytes) {
    const uintptr_t a = (uintptr_t)p;
    auto it = g_host_allocs.upper_bound(a);
    if (it == g_host_allocs.begin()) return g_host_allocs.end();
    --it;
    return a + bytes <= it->first + it->second.bytes ? it : g_host_allocs.end();
}

int nsb_host_register(void* p, size_t bytes) {
    if (!p || bytes == 0) {
        set_error("nsb_host_register: bad arguments");
        return NSB_ERR_INVALID;
    }
    {
        std::lock_guard<std::mutex> lock(g_host_mu);
        auto it = host_find_locked(p, bytes);
        if (it != g_host_allocs.end()) {
            if (it->second.kind != HostKind::Adopted) return NSB_HOST_ALREADY_LOCKED;  // nsb_host_alloc memory, or registered before
            // An adopted range belongs to the caller, who may have unlocked and freed it since (the reference's
            // ~Evaluator runs before ~Infer): trust the entry only if the driver still knows the range.
            void* dp = nullptr;
            if (cudaHostGetDevicePointer(&dp, p, 0) == cudaSuccess && dp == p) return NSB_HOST_ALREADY_LOCKED;
            cudaGetLastError();
            g_host_allocs.erase(it);  // stale: the address has been reused; register it afresh below
        }
    }
    const cudaError_t e = cudaHostRegister(p, bytes, cudaHostRegisterPortable | cudaHostRegisterMapped);  // evaluator.cc:95-106
    const bool adopted = e == cudaErrorHostMemoryAlreadyRegistered;  // the caller pinned it (the reference's Evaluator does)
    if (adopted) {
        cudaGetLastError();
    } else if (e != cudaSuccess) {
        cudaGetLastError();
        set_error("cudaHostRegister failed: %s", cudaGetErrorString(e));
        return NSB_ERR_CUDA;
    }
    // direct I/O needs the device to reach the range at its host address (true on unified-addressing
    // x86 hosts); otherwise the range stays page-locked but calls using it take the staged path
    void* dp = nullptr;
    const bool direct = cudaHostGetDevicePointer(&dp, p, 0) == cudaSuccess && dp == p;
    if (!direct) cudaGetLastError();
    if (direct || !adopted) {
        std::lock_guard<std::mutex> lock(g_host_mu);
        g_host_allocs[(uintptr_t)p] = HostRange{bytes, direct, adopted ? HostKind::Adopted : HostKind::Registered};
    }
    return adopted ? NSB_HOST_ALREADY_LOCKED : NSB_OK;
}
int nsb_host_unregister(void* p) {
    bool ours = false;
    {
        std::lock_guard<std::mutex> lock(g_host_mu);
        auto it = g_host_allocs.find((uintptr_t)p);
        if (it != g_host_allocs.end() && it->second.kind != HostKind::Alloc && it->second.kind != HostKind::NodeAlloc) {  // nsb_host_alloc* memory goes with nsb_host_free
            ours = it->second.kind == HostKind::Registered;
            g_host_allocs.erase(it);
        }
    }
    if (ours) NSB_CUDA(cudaHostUnregister(p));  // an adopted range stays locked: its owner unlocks it
    return 0;
}
int nsb_set_io_mode(nsb_ctx* c, int mode) {
    if (!c || (mode != NSB_IO_STAGED && mode != NSB_IO_DIRECT)) {
        set_error("nsb_set_io_mode: bad arguments");
        return NSB_ERR_INVALID;
    }
    c->direct_io = mode == NSB_IO_DIRECT;
    return 0;
}
int nsb_io_mode(nsb_ctx* c) { return c && c->direct_io ? NSB_IO_DIRECT : NSB_IO_STAGED; }
int nsb_device_alloc(void** out, size_t bytes) {
    if (!out) return NSB_ERR_INVALID;
    NSB_CUDA(cudaMalloc(out, bytes ? bytes : 1));
    return 0;
}
int nsb_device_free(void* p) {
    NSB_CUDA(cudaFree(p));
    return 0;
}
int nsb_memcpy_h2d(void* dst, const void* src, size_t bytes) {
    NSB_CUDA(cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice));
    return 0;
}
int nsb_memcpy_d2h(void* dst, const void* src, size_t bytes) {
    NSB_CUDA(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost));
    return 0;
}
int nsb_memset_device(void* dst, int value, size_t bytes) {
    NSB_CUDA(cudaMemset(dst, value, bytes));
    return 0;
}
int nsb_device_sync(void) {
    NSB_CUDA(cudaDeviceSynchronize());
    return 0;
}

int nsb_umma_selftest(int gpu, int n_cols, int k_elems, int shift_rows, float* max_err, float* epi_err) {
    return umma_selftest(gpu, n_cols, k_elems, shift_rows, max_err, epi_err);
}

#ifdef NSB_DIAG
int nsb_debug_umma_probe(int gpu, int n_cols, int k_elems, int shift_rows, int layout, int iters, float* max_err,
                         double* cycles_per_mma) {
    return umma_probe(gpu, n_cols, k_elems, shift_rows, layout, iters, max_err, cycles_per_mma);
}

int nsb_debug_bulk_rate_probe(int gpu, int ctas, int tile_bytes, int stages, int split, double* bytes_per_cycle) {
    return bulk_rate_probe(gpu, ctas, tile_bytes, stages, split, bytes_per_cycle);
}

#endif  // NSB_DIAG

int nsb_event_create(void** out) {
    if (!out) return NSB_ERR_INVALID;
    cudaEvent_t e;
    NSB_CUDA(cudaEventCreate(&e));
    *out = e;
    return 0;
}
int nsb_event_destroy(void* ev) {
    NSB_CUDA(cudaEventDestroy(static_cast<cudaEvent_t>(ev)));
    return 0;
}
int nsb_event_record(void* ev, nsb_ctx* c, int slot) {
    int rc = check_ctx(c, slot);
    if (rc) return rc;
    NSB_CUDA(cudaEventRecord(static_cast<cudaEvent_t>(ev), c->slots[slot].stream));
    return 0;
}
int nsb_event_sync(void* ev) {
    NSB_CUDA(cudaEventSynchronize(static_cast<cudaEvent_t>(ev)));
    return 0;
}
int nsb_event_elapsed_ms(void* start, void* stop, float* ms) {
    if (!ms) return NSB_ERR_INVALID;
    NSB_CUDA(cudaEventElapsedTime(ms, static_cast<cudaEvent_t>(start), static_cast<cudaEvent_t>(stop)));
    return 0;
}

}  // extern "C"
