/*
 * echo_b200_debug.h — diagnostic entry points of libecho_b200.so. Not part of the drop-in surface: they exist so the
 * parity tests can drive individual device routines (BxDFs, FastMath shims, per-sample radiance) against the oracle,
 * and so bench.py can read the traversal visit counters that give the algorithmic bytes of a batch
 * (the device counterpart of Accelerator.TraceCost, Aggregation/Acceleration/QuadBoundingVolumeHierarchy.cs:317-361).
 */
#ifndef ECHO_B200_DEBUG_H
#define ECHO_B200_DEBUG_H

#include "echo_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* like echo_b200_trace_batch_device / occlude, additionally accumulating {node, triangle, sphere} visit totals into
 * d_counts3 (3 x uint64 on the device, added to, not reset). */
int32_t echo_b200_trace_batch_device_counted(EchoScene*, const EchoRay* d_rays, uint64_t n, EchoHit* d_hits, uint64_t* d_counts3, void* stream);
int32_t echo_b200_occlude_batch_device_counted(EchoScene*, const EchoRay* d_rays, uint64_t n, uint8_t* d_occluded, uint64_t* d_counts3, void* stream);

/* BxDF known-answer hook, same kinds / parameter packing / outputs as oracle_bxdf_batch (oracle/oracle.h). Host buffers. */
int32_t echo_b200_debug_bxdf_batch(int32_t device, int32_t kind, const float* params11, const float* outgoing3, const float* samples2,
                                   uint64_t n, float* sampled8, float* evaluated4, float* inverse4);

/* FastMath / sincos shims, same op codes as oracle_fastmath (op 100: sin, 101: cos of the deterministic sincos). Host buffers. */
int32_t echo_b200_debug_math(int32_t device, int32_t op, const float* a, const float* b, const float* c, uint64_t n, float* out);

/* One Evaluator.Evaluate per listed (pixel, sample index): out_rgb receives n x 3 floats. Host buffers. */
int32_t echo_b200_debug_evaluate_samples(EchoScene*, const EchoRenderParams*, const int32_t* pixel_xy, const uint32_t* sample_index,
                                         uint64_t n, float* out_rgb);

/* The same with the W lane kept (n x 4 floats): the auxiliary evaluators use it (NormalDepth128's depth). */
int32_t echo_b200_debug_evaluate_samples4(EchoScene*, const EchoRenderParams*, const int32_t* pixel_xy, const uint32_t* sample_index,
                                          uint64_t n, float* out_rgba);

/* Libraries built with -DECHO_BOUNDS_CHECK check every index the kernels derive from scene data or stack pointers; this returns the
 * bit set of checks that failed since commit (0 = clean). Release builds write 0xFFFFFFFF ("not compiled in"). */
int32_t echo_b200_debug_bounds_violations(EchoScene*, uint32_t* out_bits);

/* Microbenchmarks of the on-chip memory system of `device` (csrc/peaks.cu), a few milliseconds each: out3[0] = L2 read bandwidth with
 * coalesced 128-bit loads, out3[1] = L2 bandwidth with one random 32-byte sector per lane (the access shape of an incoherent QBVH
 * node fetch), out3[2] = the same out of L1 (the LSU / L1 data-pipe ceiling), all in GB/s. bench.py sets the traversal kernel's
 * algorithmic bytes against them (`roofline.frac_l2`, `frac_l1_sectors`) beside the HBM fraction. */
int32_t echo_b200_debug_measure_peaks(int32_t device, float* out3);

/* Changes one tuning switch of the wavefront at run time: `name` is the part after ECHO_B200_ of the environment variable that
 * sets its initial value (RENDER_WORKERS, BATCH_PATHS, NARROW_LIMIT, TAIL_LIMIT, RUN_AHEAD, BLOCKING_SYNC; -1 = automatic for the
 * last two). Process-wide; takes effect with the next render call. For A/B runs that keep one uploaded scene. */
int32_t echo_b200_debug_set_option(const char* name, int64_t value);

/* Phases of the calling thread's last echo_b200_build_qbvh that ran the SweepBuilder build (csrc/sweep.cu): out4 = {upload ms, device
 * build ms, download ms, binary levels}, host wall time around synchronised phases. Zeros if no such build ran on this thread. */
int32_t echo_b200_debug_last_build(float* out4);
/* The same for the calling thread's last echo_b200_build_light_tree / echo_b200_scene_build_light_tree (csrc/lightbuild.cu); out4[3] = levels. */
int32_t echo_b200_debug_last_light_build(float* out4);
/* The calling thread's last echo_b200_build_packs / echo_b200_scene_build_packs (csrc/packbuild.cu): out8 = {rounds, QBVH levels read back,
 * light-tree levels read back, synchronising read-backs in all, launches, ms of host wall time for the synchronised build, packs rebuilt one
 * by one after the forest gave up, 0}. Zeros if no such build ran on this thread. */
int32_t echo_b200_debug_last_pack_build(float* out8);

#ifdef __cplusplus
}
#endif
#endif
