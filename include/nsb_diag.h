/*
 * nsb_diag.h - diagnostic entry points, exported ONLY by the diagnostic build of the library
 * (nshogi-engine_b200/libnsb_diag.so = the same sources compiled with -DNSB_DIAG).  That build also carries what the
 * product library (libnsb.so, include/nsb.h) leaves out: clock64 stamps inside the trunk kernels (tools/timeline.py,
 * tools/residency.py), the tcgen05 / bulk-copy probes (tools/umma_probe.py, tools/bulk_probe.py) and the superseded
 * one-CTA 256-channel kernel (NSB_TRUNK256=single, the bit-for-bit reference of the CTA-pair kernel).  Nothing here
 * replaces a reference interface.
 */
#ifndef NSB_DIAG_H
#define NSB_DIAG_H

#include "nsb.h"

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default)
#endif

/* run one trunk launch and return CTA 0's clock64 stamps, 4 per layer
 * {MMA issue start, MMA issue end, accumulator ready (epilogue start), epilogue end}, then 8 phase
 * stamps {entry, setup done, features expanded, features loaded, heads read, policy written, value
 * MLP done, decode done}: 4 * layers + 8 values. */
int nsb_debug_trunk_timeline(nsb_ctx* ctx, int slot, const nsb_feature_bitboard* d_features, size_t n,
                             uint64_t* host_stamps, size_t max_stamps);
/* Same launch fed with packed positions (stage 1 in the kernel's prologue). */
int nsb_debug_trunk_timeline_positions(nsb_ctx* ctx, int slot, const nsb_position* d_positions, size_t n,
                                       uint64_t* host_stamps, size_t max_stamps);

/* issue-to-retire rate (cycles per M128 x n_cols x K16 MMA) and numerical check of one
 * operand layout with a row-shifted B start: layout 0 = SWIZZLE_NONE 16-byte rows, 1 = SWIZZLE_128B. */
int nsb_debug_umma_probe(int gpu, int n_cols, int k_elems, int shift_rows, int layout, int iters,
                         float* max_err, double* cycles_per_mma);

/* sustained cp.async.bulk (L2 -> shared ring) rate per CTA in bytes per SM cycle. */
int nsb_debug_bulk_rate_probe(int gpu, int ctas, int tile_bytes, int stages, int split, double* bytes_per_cycle);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* NSB_DIAG_H */
