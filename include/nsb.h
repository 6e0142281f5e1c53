/*
 * nsb.h — C ABI of the B200-native leaf-evaluation executor ("nsb" = nshogi-b200).
 *
 * This is the drop-in boundary for nyashiki/nshogi-engine's NN leaf-evaluation path.
 * The reference selects its executor at compile time behind the C++ virtual class
 * `nshogi::engine::infer::Infer` (reference src/infer/infer.h:19-32).  The reference has no
 * C ABI of its own; every entry point below names the reference interface it replaces so
 * a thin `infer::B200 : Infer` (nshogi-engine_b200/host/infer_b200.h) can forward to it.
 *
 * Conventions
 *   - plain pointers and sizes only; no C++/torch types cross this boundary
 *   - every function returns 0 on success or a negative nsb_status; nsb_last_error()
 *     returns a thread-local human-readable message for the last failure
 *   - there is NO CPU fallback: if no CUDA device / kernel image is usable the call fails
 *   - one nsb_ctx per host evaluator thread (reference: one Infer per EvaluationWorker,
 *     src/mcts/evaluationworker.cc:75-103); a ctx is not thread-safe
 *   - "host" pointers may be pageable or pinned; pinned (cudaHostRegister'd, as the
 *     reference's Evaluator does at src/evaluate/evaluator.cc:95-106) makes copies async
 */
#ifndef NSB_H
#define NSB_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default) /* the library is built -fvisibility=hidden */
#endif

#define NSB_NUM_SQUARES 81      /* nshogi core::NumSquares                               */
#define NSB_POLICY_PLANES 27    /* 27 move-type planes (src/mcts/evaluationworker.cc:166) */
#define NSB_POLICY_SIZE 2187    /* ml::MoveIndexMax = 27 * 81 (src/infer/trt.cc:205)      */
#define NSB_FEATURE_CHANNELS 86 /* preset::SimpleFeatures (src/evaluate/preset.h:20-66)   */
#define NSB_MAX_LEGAL_MOVES 593 /* upper bound on legal shogi moves                      */
#define NSB_CACHE_MAX_MOVES 164 /* EvalCache row width (src/mcts/evalcache.h:26-38)      */

typedef enum nsb_status {
    NSB_OK = 0,
    NSB_ERR_INVALID = -1,   /* bad argument / precondition (reference: assert, trt.cc:237-238) */
    NSB_ERR_CUDA = -2,      /* CUDA runtime error (reference never checks these)               */
    NSB_ERR_NO_DEVICE = -3, /* no usable sm_100a device: the product path has no CPU fallback  */
    NSB_ERR_STATE = -4,     /* weights not loaded / ctx busy                                   */
    NSB_ERR_NOMEM = -5
} nsb_status;

/* 16-byte packed feature plane == nshogi ml::FeatureBitboard.
 * Layout pinned by reference src/cuda/extractbit.cu:20-37 (see DESIGN.md §3):
 *   lo bits 0..62 = squares 0..62; hi bits 0..17 = squares 63..80; hi bit 24 = rotate;
 *   hi bits 32..63 = IEEE-754 fp32 fill value. */
typedef struct nsb_feature_bitboard {
    uint64_t lo;
    uint64_t hi;
} nsb_feature_bitboard;

/* ResNet shape.  The reference ships no model (external ONNX, src/context.h:93); only the
 * tensor contract is pinned (src/infer/trt.cc:144-150,193-227).  DESIGN.md §5 defines the
 * canonical random-init net: stem conv3x3(in->C) ; blocks x [conv3x3, conv3x3 + skip] ;
 * policy conv1x1(C->27) ; value conv1x1(C->1) -> FC(81->hidden) -> FC(hidden->2) -> sigmoid. */
typedef struct nsb_net_desc {
    int32_t in_channels;  /* feature planes per position: 86 (SimpleFeatures), 93 (CustomFeaturesV1), <= 96 */
    int32_t channels;     /* trunk width C (128, 192 or 256)     */
    int32_t blocks;       /* residual blocks (10, 20, 40)        */
    int32_t value_hidden; /* hidden units of the value MLP (256) */
} nsb_net_desc;

/* Compact position record (builder-defined; stage-1 input, SURVEY.md App. A.2).
 * board[sq]: 0 = empty, else 1 + piece_type + 14 * colour, piece_type in
 *   0..13 = {P,L,N,S,G,K,B,R,+P,+L,+N,+S,+B,+R} (channel order of preset.h:20-33),
 *   colour 0 = black, 1 = white.  hands[colour][k], k in {P,L,N,S,G,B,R}. */
typedef struct nsb_position {
    uint8_t board[81];
    uint8_t side; /* 0 = black to move, 1 = white to move */
    uint8_t hands[2][7];
    uint16_t ply;
    uint16_t max_ply;
    float black_draw_value;
    float white_draw_value;
} nsb_position; /* 108 bytes */

typedef struct nsb_ctx nsb_ctx;

/* ---- lifecycle ------------------------------------------------------------------------- */

/* Replaces TensorRT::TensorRT(int GPUId, uint16_t BatchSizeMax, uint16_t NumChannels)
 * (reference src/infer/trt.cc:52-80): selects the device, allocates device buffers for
 * `batch_max` samples and `slots` independent in-flight batches (>=1), creates one
 * non-blocking stream per slot. */
int nsb_create(nsb_ctx** out, int gpu, int batch_max, int slots, const nsb_net_desc* net);

/* Replaces TensorRT::~TensorRT (trt.cc:82-107). */
void nsb_destroy(nsb_ctx* ctx);

/* Replaces TensorRT::resetGPU (trt.cc:289-291): cudaSetDevice on the calling thread. */
int nsb_bind_thread(nsb_ctx* ctx);

/* Number of floats in the canonical fp32 weight blob for `net` (layout: DESIGN.md §5). */
size_t nsb_weight_blob_floats(const nsb_net_desc* net);

/* Deterministic random init of a canonical blob (He-normal convs, small biases); every
 * stored value is exactly representable in bf16 so that the CPU oracle and the device see
 * identical weights.  Host-only helper (no device work). */
int nsb_weight_blob_random(const nsb_net_desc* net, uint64_t seed, float* blob);

/* Replaces TensorRT::load(path, useCache) (trt.cc:109-232): takes the canonical fp32 blob,
 * repacks it into the bf16 UMMA tile order the trunk kernel streams, uploads it. */
int nsb_load_weights(nsb_ctx* ctx, const float* blob, size_t n_floats);

/* ---- the Infer contract (host buffers) ------------------------------------------------- */

/* Replaces Infer::computeNonBlocking (src/infer/infer.h:24-26; TRT impl trt.cc:234-272):
 * enqueue H2D of n*C feature bitboards, feature expansion + ResNet forward, D2H of
 * policy[n*2187] raw logits (plane-major), win[n], draw[n] (probabilities).  Returns
 * immediately; results are valid after nsb_await(ctx, slot).  Precondition: n <= batch_max
 * and the slot is idle. */
int nsb_eval_async(nsb_ctx* ctx, int slot, const nsb_feature_bitboard* features, size_t n,
                   float* policy, float* win, float* draw);

/* Fused-decode variant (replaces trt.cc:234-272 + FeedWorker::feedResult gather/softmax,
 * src/mcts/feedworker.cc:100-127, or Frame::setEvaluation, src/selfplay/frame.cc:96-118):
 * the caller supplies CSR legal-move policy indices (move_off[n+1], move_idx[move_off[n]],
 * values from ml::getMoveIndex) and receives per-move outputs instead of dense logits.
 *   mode NSB_DECODE_PROBS : MCTS flavour (FeedWorker::feedResult, feedworker.cc:100-136): softmax over the
 *                           legal moves (T=1); a 1-move row is 1.0 without a gather (:101-103); with a
 *                           cache the PROBABILITIES are stored (:134-135)
 *   mode NSB_DECODE_LOGITS: raw gathered logits only (the first half of Frame::setEvaluation, frame.cc:96-114)
 *   mode NSB_DECODE_BOTH  : self-play flavour, the whole of Frame::setEvaluation<false> (frame.cc:93-118) in one
 *                           launch: gather -> the RAW LOGITS go to the cache (:110-114) -> softmax (no 1-move
 *                           shortcut; skipped for rows flagged NSB_ROW_SKIP_SOFTMAX = the Gumbel root, :116-118)
 *                           -> legal_out; nsb_decode_request::logits_out (optional) also returns the raw logits.
 *                           Rows served from the cache take the same route from the stored logits.  The
 *                           Dirichlet mix at the AlphaZero root (:121-133) is host/selfplay_feed.h.
 *   | NSB_DECODE_NAN_FALLBACK : feedResult<NaNFallbackEnabled = true>.  The reference ships it OFF
 *                           (src/context.h:103), and so does mode & 0x100 == 0: NaNs flow through the softmax,
 *                           nan_flag[i] = 0, rows are stored in the cache whatever they hold.  With the bit set:
 *                             - a NaN among the gathered logits of a row with >= 2 moves replaces every legal
 *                               logit by 1 before the softmax, i.e. a uniform row (feedworker.cc:106-118);
 *                             - a NaN win / draw rate leaves the row's softmax alone (:58-85: the caller replaces
 *                               the value from the parent node, host/mcts_feed.h) and is returned as is;
 *                             - nan_flag[i] = 1 for either (NaNFound), and such rows are not stored (:134).
 *                           NaN test: bit pattern, src/math/math.h:23-39. */
#define NSB_DECODE_PROBS 0
#define NSB_DECODE_LOGITS 1
#define NSB_DECODE_BOTH 2
#define NSB_DECODE_MODE_MASK 0xFF
#define NSB_DECODE_NAN_FALLBACK 0x100
#define NSB_ROW_SKIP_SOFTMAX 1 /* nsb_decode_request::row_flags bit: Gumbel root (frame.cc:116-118) */
int nsb_eval_decode_async(nsb_ctx* ctx, int slot, const nsb_feature_bitboard* features, size_t n,
                          const uint32_t* move_off, const uint16_t* move_idx, int mode,
                          float* legal_out, float* win, float* draw, uint8_t* nan_flag);

/* Same two calls fed from compact position records: stage 1 (position -> 86 feature
 * bitboards; replaces FeatureStackComptime::constructAt at
 * src/selfplay/evaluationworker.cc:87-92) also runs on the device. */
int nsb_eval_positions_async(nsb_ctx* ctx, int slot, const nsb_position* positions, size_t n,
                             float* policy, float* win, float* draw);

/* Fully fused variant: stage 1 on the device, forward, fused legal-move decode.  This is the
 * self-play evaluation step (src/selfplay/evaluationworker.cc:87-108) in one call: 108 B up and
 * ~4 B per legal move down per position instead of 1,376 B up and 8,756 B down. */
int nsb_eval_positions_decode_async(nsb_ctx* ctx, int slot, const nsb_position* positions, size_t n,
                                    const uint32_t* move_off, const uint16_t* move_idx, int mode,
                                    float* legal_out, float* win, float* draw, uint8_t* nan_flag);

/* The general form of the fused path; every nsb_eval_*decode_async call is this request with some
 * fields left NULL.
 *   features / positions : exactly one is set (bitboards in, or packed positions with stage 1 in the
 *                          trunk kernel's prologue)
 *   hashes               : non-NULL -> through the device-resident cache (nsb_cache_create): hits are
 *                          served from HBM, misses evaluated and stored; hit_flag[i] = 1 for a hit
 *   order_out (optional) : per position the RANK ORDER of its decoded row: order_out[move_off[i] + r] =
 *                          index within the row (0 .. n_i-1) of the move with the r-th largest value,
 *                          ties by lower index first; identity for a row flagged NaN.  This is the
 *                          permutation the reference applies with Node::sort() - std::sort of the edges by
 *                          decreasing probability, src/mcts/node.h:163-168, on a feed thread for every leaf
 *                          (feedworker.cc:129) - so the caller writes its edges in search order in one
 *                          pass instead of sorting them (std::sort leaves the order of ties unspecified;
 *                          here it is defined).  Rows served from the cache are ranked too.  A row whose
 *                          values contain a NaN (possible without NSB_DECODE_NAN_FALLBACK) gets the identity. */
typedef struct nsb_decode_request {
    const nsb_feature_bitboard* features; /* [n][86] or NULL                      */
    const nsb_position* positions;        /* [n]     or NULL                      */
    size_t n;
    const uint64_t* hashes;               /* [n] or NULL (no cache)               */
    const uint32_t* move_off;             /* [n+1] CSR offsets                    */
    const uint16_t* move_idx;             /* [move_off[n]] policy slots           */
    int mode;                             /* NSB_DECODE_* [| NSB_DECODE_NAN_FALLBACK] */
    float* legal_out;                     /* [move_off[n]]                        */
    uint16_t* order_out;                  /* [move_off[n]] or NULL                */
    float* win;                           /* [n]                                  */
    float* draw;                          /* [n]                                  */
    uint8_t* nan_flag;                    /* [n] or NULL                          */
    uint8_t* hit_flag;                    /* [n] or NULL (cached requests only)   */
    const uint8_t* row_flags;             /* [n] or NULL: NSB_ROW_* bits (NSB_DECODE_BOTH)            */
    float* logits_out;                    /* [move_off[n]] or NULL: raw logits too (NSB_DECODE_BOTH) */
} nsb_decode_request;
int nsb_eval_request_async(nsb_ctx* ctx, int slot, const nsb_decode_request* request);

/* Replaces Infer::await (trt.cc:281-283). */
int nsb_await(nsb_ctx* ctx, int slot);
/* Replaces Infer::isComputing (trt.cc:285-287): 1 busy, 0 idle, <0 error. */
int nsb_is_computing(nsb_ctx* ctx, int slot);

/* ---- device-resident entry points (inputs/outputs already in HBM) ----------------------- */

/* Whole path on device pointers, enqueued on the slot's stream (bench `value` leg). */
int nsb_eval_device(nsb_ctx* ctx, int slot, const nsb_feature_bitboard* d_features, size_t n,
                    float* d_policy, float* d_win, float* d_draw);

/* Whole path + fused decode on device pointers; d_policy may be NULL (logits stay on chip). */
int nsb_eval_decode_device(nsb_ctx* ctx, int slot, const nsb_feature_bitboard* d_features, size_t n,
                           const uint32_t* d_move_off, const uint16_t* d_move_idx, int mode,
                           float* d_policy, float* d_legal_out, float* d_win, float* d_draw,
                           uint8_t* d_nan_flag);

/* Stage 2 alone == cuda::extractBits<ChannelsFirst> (src/cuda/extractbit.h:21-23):
 * feature bitboards -> fp32 planes, NCHW (channels_first=1) or NHWC (0).  Bit-exact. */
int nsb_extract_device(nsb_ctx* ctx, int slot, const nsb_feature_bitboard* d_features, size_t n,
                       int channels, int channels_first, float* d_planes);

/* Stage 1 alone: position records -> feature bitboards (86 per position). */
int nsb_pack_positions_device(nsb_ctx* ctx, int slot, const nsb_position* d_positions, size_t n,
                              nsb_feature_bitboard* d_features);

/* Decode alone from dense logits (feedworker.cc:100-127 / frame.cc:96-118). */
int nsb_decode_device(nsb_ctx* ctx, int slot, const float* d_policy, const float* d_win,
                      const float* d_draw, size_t n, const uint32_t* d_move_off,
                      const uint16_t* d_move_idx, int mode, float* d_legal_out,
                      uint8_t* d_nan_flag);

/* The same with the per-row flags and the second output of NSB_DECODE_BOTH (d_row_flags, d_logits_out optional). */
int nsb_decode_device_ex(nsb_ctx* ctx, int slot, const float* d_policy, const float* d_win, const float* d_draw,
                         size_t n, const uint32_t* d_move_off, const uint16_t* d_move_idx, int mode,
                         const uint8_t* d_row_flags, float* d_legal_out, float* d_logits_out, uint8_t* d_nan_flag);

/* ---- device-resident evaluation cache (SURVEY.md §8 f3) --------------------------------- */

/* Replaces EvalCache::EvalCache(MemorySize MiB) (reference src/mcts/evalcache.cc:17-47) with a
 * table in HBM: rows of <= 164 legal-move values + win + draw keyed by the 64-bit state hash,
 * bundles of 3 entries in recency order, bundle = hash % NumBundle, try-lock per bundle (a busy
 * bundle drops the operation, evalcache.cc:58-62,127-131).  One cache per ctx, shared by its slots.
 * A cache holds what the decode mode of the launches that fill it stores: probabilities for NSB_DECODE_PROBS
 * (MCTS, feedworker.cc:135), raw logits for NSB_DECODE_LOGITS / NSB_DECODE_BOTH (self-play, frame.cc:110-114);
 * a hit is post-processed by the mode of the request that probes (BOTH: softmax of the stored logits), so a
 * cache is filled and probed with one mode - as in the reference, where the MCTS manager and the self-play
 * frames each own theirs. */
int nsb_cache_create(nsb_ctx* ctx, size_t memory_mb);
int nsb_cache_clear(nsb_ctx* ctx);
/* The reference has ONE EvalCache per Manager, shared by all evaluation workers (src/mcts/manager.cc:202-206)
 * - by default two executors per GPU (context.h:75).  nsb_cache_attach lets `ctx` use the table `owner`
 * created (same device): launches of both contexts probe and fill it concurrently, the bundles' lock words
 * arbitrate.  The owner must outlive every ctx attached to it. */
int nsb_cache_attach(nsb_ctx* ctx, nsb_ctx* owner);
uint64_t nsb_cache_num_bundles(nsb_ctx* ctx);

/* == EvalCache::store (evalcache.cc:49-121) for a batch of CSR rows on device pointers; rows with
 * d_skip[i] != 0 (NaN rows, feedworker.cc:134) are not stored; d_stored[i] (optional) = 1 when the
 * entry is present afterwards. */
int nsb_cache_store_device(nsb_ctx* ctx, int slot, const uint64_t* d_hashes, size_t n,
                           const uint32_t* d_move_off, const float* d_legal, const float* d_win,
                           const float* d_draw, const uint8_t* d_skip, uint8_t* d_stored);

/* == EvalCache::load (evalcache.cc:123-169) + the caller's move-count check
 * (src/mcts/searchworker.cc:545-556) for a batch: hits get their row / win / draw written and
 * d_hit[i] = 1; misses are appended (in no particular order) to d_miss_idx[0 .. *d_miss_count). */
int nsb_cache_probe_device(nsb_ctx* ctx, int slot, const uint64_t* d_hashes, size_t n,
                           const uint32_t* d_move_off, float* d_legal_out, float* d_win, float* d_draw,
                           uint8_t* d_hit, int* d_miss_idx, int* d_miss_count);

/* nsb_eval_decode_async behind the cache: probe, evaluate only the misses (the trunk launch works
 * on the probe's miss list), and store every evaluated row whose nan flag is clear - the sequence
 * searchworker.cc:540-559 -> evaluation -> feedworker.cc:134-135, in two kernel launches.
 * hit_flag[i] (optional) = 1 when position i was served from the cache. */
int nsb_eval_cached_decode_async(nsb_ctx* ctx, int slot, const nsb_feature_bitboard* features, size_t n,
                                 const uint64_t* hashes, const uint32_t* move_off, const uint16_t* move_idx,
                                 int mode, float* legal_out, float* win, float* draw, uint8_t* nan_flag,
                                 uint8_t* hit_flag);
/* The same from compact position records (stage 1 on the device first): the self-play evaluation
 * step of src/selfplay/evaluationworker.cc:87-108 behind Frame's evaluation cache
 * (src/selfplay/frame.cc:89-114). */
int nsb_eval_positions_cached_decode_async(nsb_ctx* ctx, int slot, const nsb_position* positions, size_t n,
                                           const uint64_t* hashes, const uint32_t* move_off,
                                           const uint16_t* move_idx, int mode, float* legal_out, float* win,
                                           float* draw, uint8_t* nan_flag, uint8_t* hit_flag);
int nsb_eval_cached_decode_device(nsb_ctx* ctx, int slot, const nsb_feature_bitboard* d_features, size_t n,
                                  const uint64_t* d_hashes, const uint32_t* d_move_off,
                                  const uint16_t* d_move_idx, int mode, float* d_legal_out, float* d_win,
                                  float* d_draw, uint8_t* d_nan_flag, uint8_t* d_hit);

/* Stream of a slot as an opaque cudaStream_t (for event timing from the host side). */
void* nsb_stream(nsb_ctx* ctx, int slot);

/* Device time of the trunk kernel, measured with CUDA events recorded on the slot's stream
 * around every trunk launch and harvested in nsb_await(): running sum (ms) and launch count
 * since creation or the last nsb_trunk_time_reset().  Enabled by nsb_set_timing(ctx, 1). */
int nsb_set_timing(nsb_ctx* ctx, int enabled);
int nsb_trunk_time(nsb_ctx* ctx, double* sum_ms, uint64_t* launches);
int nsb_trunk_time_reset(nsb_ctx* ctx);

/* CUDA events on a slot's stream, for timing a region from the host side of the ABI
 * (torch.cuda.Event only sees torch's own streams). */
int nsb_event_create(void** out);
int nsb_event_destroy(void* ev);
int nsb_event_record(void* ev, nsb_ctx* ctx, int slot);
int nsb_event_sync(void* ev);
int nsb_event_elapsed_ms(void* start, void* stop, float* ms);

/* Which trunk kernel this ctx launches (chosen at nsb_create from the net width and the number of
 * slots: a one-slot ctx gets the kernel with the shortest launch, a multi-slot ctx the one with the
 * highest throughput when several batches are in flight). */
const char* nsb_trunk_kernel_name(nsb_ctx* ctx);

/* Kernel launches issued by this ctx since creation (bench "gpu_launches"). */
uint64_t nsb_launch_count(nsb_ctx* ctx);

/* ---- misc ------------------------------------------------------------------------------ */

/* Pinned host allocation helpers (reference pins with cudaHostRegister, evaluator.cc:95-106).
 * Memory from nsb_host_alloc is page-locked AND mapped into the device's address space. */
int nsb_host_alloc(void** out, size_t bytes);
int nsb_host_free(void* p);
/* The same, placed on the NUMA node of `gpu` (its PCI function's numa_node): what the reference's Evaluator does with
 * numa_alloc_onnode in NUMA_ENABLED builds (src/evaluate/evaluator.cc:127-136) - except that the node is the GPU's own.
 * On an 8-GPU box this keeps each GPU's D2H stream (8,756 B per sample through the Infer contract) on its own socket.
 * Falls back to ordinary placement where the node is unknown.  Free with nsb_host_free. */
int nsb_host_alloc_near(void** out, size_t bytes, int gpu);
/* NUMA node of a GPU (-1: unknown / single node). */
int nsb_gpu_numa_node(int gpu);
/* Pin the calling thread to the CPUs of the GPU's NUMA node (== the affinity half of evaluator.cc:39-83).  0 = done,
 * 1 = nothing to do on this machine (not an error). */
int nsb_numa_bind_thread(int gpu);
/* Page-lock (or adopt, if the caller already did: cudaHostRegister in evaluator.cc:95-106) a buffer the
 * caller owns, so that calls using it qualify for NSB_IO_DIRECT below.  Returns NSB_OK when this call locked the
 * range (undo with nsb_host_unregister), NSB_HOST_ALREADY_LOCKED (> 0, not an error) when it already was - by the
 * caller or by an earlier call - and < 0 on failure (the buffer still works, through the staged path).
 * nsb_host_unregister forgets the range and unlocks it only if nsb_host_register locked it (nsb_host_alloc
 * memory is left alone).  A registered or adopted range must outlive every call that uses it; whoever made the
 * library know a range calls nsb_host_unregister before the memory is unlocked / freed by its owner, or at the
 * latest when the executor goes (infer::B200 does both for the Infer contract's arrays).  An adopted range is
 * re-validated with the driver whenever it is registered again, so an address the caller has freed and the
 * allocator has reused is never taken for page-locked memory. */
#define NSB_HOST_ALREADY_LOCKED 1
int nsb_host_register(void* p, size_t bytes);
int nsb_host_unregister(void* p);

/* How the host-buffer entry points (nsb_eval_async, nsb_eval_decode_async and their nsb_eval_positions_*
 * twins) move data.
 *   NSB_IO_STAGED: copy nodes on the slot's stream around the kernel (H2D inputs, D2H results), the
 *                  reference's scheme (trt.cc:240-242,265-271).  Default for contexts with >= 2 slots:
 *                  the copies of one batch overlap the kernels of the others.
 *   NSB_IO_DIRECT: when every buffer of the call lies in nsb_host_alloc memory, the one trunk launch
 *                  reads its inputs from and writes its results into those buffers itself over PCIe:
 *                  no copy nodes, one stream operation per batch.  Default for one-slot contexts,
 *                  where every copy node is serial latency.  Calls with other buffers fall back to
 *                  the staged path.  Results are complete after nsb_await() either way; the inputs
 *                  must stay untouched until then (the Infer contract, evaluationworker.cc:158-180).
 * Environment override at nsb_create: NSB_IO=direct|staged. */
#define NSB_IO_STAGED 0
#define NSB_IO_DIRECT 1
int nsb_set_io_mode(nsb_ctx* ctx, int mode);
int nsb_io_mode(nsb_ctx* ctx);
int nsb_device_alloc(void** out, size_t bytes);
int nsb_device_free(void* p);
int nsb_memcpy_h2d(void* dst, const void* src, size_t bytes);
int nsb_memcpy_d2h(void* dst, const void* src, size_t bytes);
int nsb_memset_device(void* dst, int value, size_t bytes);
int nsb_device_sync(void);

const char* nsb_last_error(void);
const char* nsb_version(void);
int nsb_device_count(void);

/* tcgen05 self-test: one CTA runs D[128 x n_cols] = A * B^T with the K-major SWIZZLE_NONE
 * descriptors the trunk uses, B's start address moved by shift_rows 16-byte rows, and the host
 * compares against an fp32 loop (max_err), then runs the trunk's epilogue path (16x256b TMEM
 * fragments + stmatrix.trans, plain and with the skip connection) and compares the bf16 records
 * (epi_err).  n_cols in {96, 192}.  Inputs are exact in bf16: expect 0 for both. */
int nsb_umma_selftest(int gpu, int n_cols, int k_elems, int shift_rows, float* max_err, float* epi_err);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* NSB_H */
