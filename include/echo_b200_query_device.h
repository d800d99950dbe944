/*
 * echo_b200_query_device.h — the calls of echo_b200_query.h on device buffers, checked on the device, and the layered trace and
 * occlusion of echo_b200.h on device buffers: what a custom evaluator chains on memory it already holds on the GPU (five to ten
 * calls per bounce), without a copy or a synchronise between them.
 *
 *   echo_b200_interact_batch_device ... echo_b200_evaluate_infinite_batch_device  the eight calls of echo_b200_query.h
 *   echo_b200_trace_batch_hierarchy_device / echo_b200_occlude_batch_hierarchy_device  echo_b200_trace / occlude_batch_hierarchy
 *
 * Each call takes the arguments of its host-buffer form, in the same order, and answers bit for bit what that form answers for
 * the same inputs.
 *
 * Conventions. Every buffer is device memory of the scene's device. The calls are asynchronous on `stream` (a cudaStream_t; NULL
 * is the legacy default stream): they copy nothing and synchronise nothing, and the eight query calls allocate nothing, so a host
 * may capture them in a CUDA graph. (The two hierarchy calls, like echo_b200_trace_batch_device, allocate the work counters of
 * their persistent kernels once per device and stream: make one call on a stream before capturing it.) They need a committed single-device scene (echo_b200_scene_create) like the other *_device entry points; a multi-device
 * scene is refused. n == 0 does nothing. An n that one launch grid cannot cover (more than (2^31 - 1) * 128 queries) is refused.
 * Refused synchronously with ECHO_B200_ERR_INVALID, the message in echo_b200_last_error(): a NULL or uncommitted scene, a scene
 * without materials (interact and scatter calls), a NULL required buffer (d_status included) with n > 0, and a scene without
 * packs (the two hierarchy calls).
 *
 * Validation on the device. The eight query calls accept exactly the inputs the host-buffer calls accept (echo_b200_query.h,
 * "Validation"), but decide per query in the kernel, since tokens and layers that come from outside the library index scene arrays:
 *   - before the call the caller sets *d_status to ECHO_QUERY_STATUS_CLEAR;
 *   - every refused query i writes atomicMin(d_status, (i << 8) | code): once the stream has passed the call, the status holds the
 *     lowest refused index (status >> 8) and its reason (status & 0xFF, see echo_b200_query_reason);
 *   - a refused query reads no scene array with an index that was not accepted, and gets the zeroed record a miss gets (tokens
 *     ECHO_TOKEN_EMPTY, contact material ECHO_TOKEN_EMPTY, pick layers zeroed, pdf 0); every other query is answered normally;
 *   - one status word may collect several calls (a bounce, a frame): it keeps the lowest (index, code) of all of them.
 * The two hierarchy calls take no status: their ignore layers are only compared with the layers of a candidate hit, never used as
 * an index.
 */
#ifndef ECHO_B200_QUERY_DEVICE_H
#define ECHO_B200_QUERY_DEVICE_H

#include "echo_b200_query.h"

#ifdef __cplusplus
extern "C" {
#endif

#define ECHO_QUERY_STATUS_CLEAR 0xFFFFFFFFFFFFFFFFull /* no query refused */

int32_t echo_b200_interact_batch_device(EchoScene*, const EchoRay* rays, const EchoHit* hits, const EchoTokenHierarchy* hit_layers, uint64_t n, EchoContact* out,
                                        uint64_t* d_status, void* stream);
int32_t echo_b200_scatter_sample_batch_device(EchoScene*, const EchoRay* rays, const EchoHit* hits, const EchoTokenHierarchy* hit_layers, const float* samples2,
                                              uint64_t n, EchoScatter* out, uint64_t* d_status, void* stream);
int32_t echo_b200_scatter_evaluate_batch_device(EchoScene*, const EchoRay* rays, const EchoHit* hits, const EchoTokenHierarchy* hit_layers, const float* incident3,
                                                uint64_t n, float* out_rgba, uint64_t* d_status, void* stream);
int32_t echo_b200_light_pick_batch_device(EchoScene*, const EchoSurface* points, const float* samples1, uint64_t n, uint32_t* tokens, EchoTokenHierarchy* layers,
                                          float* pmf, uint64_t* d_status, void* stream);
int32_t echo_b200_light_mass_batch_device(EchoScene*, const uint32_t* tokens, const EchoTokenHierarchy* layers, const EchoSurface* points, uint64_t n, float* pmf,
                                          uint64_t* d_status, void* stream);
int32_t echo_b200_light_sample_batch_device(EchoScene*, const uint32_t* tokens, const EchoTokenHierarchy* layers, const EchoSurface* points, const float* samples2,
                                            uint64_t n, EchoLightSample* out, uint64_t* d_status, void* stream);
int32_t echo_b200_light_pdf_batch_device(EchoScene*, const uint32_t* tokens, const EchoTokenHierarchy* layers, const EchoSurface* points, const float* incident3,
                                         uint64_t n, float* pdf, uint64_t* d_status, void* stream);
int32_t echo_b200_evaluate_infinite_batch_device(EchoScene*, const float* directions3, uint64_t n, int32_t direct, float* out_rgb3, uint64_t* d_status, void* stream);

/* echo_b200_trace_batch_hierarchy / echo_b200_occlude_batch_hierarchy on device buffers (ignore and hit_layers nullable) */
int32_t echo_b200_trace_batch_hierarchy_device(EchoScene*, const EchoRay* rays, const EchoTokenHierarchy* ignore, uint64_t n, EchoHit* hits,
                                               EchoTokenHierarchy* hit_layers, void* stream);
int32_t echo_b200_occlude_batch_hierarchy_device(EchoScene*, const EchoRay* rays, const EchoTokenHierarchy* ignore, uint64_t n, uint8_t* occluded, void* stream);

/* the text of a refusal code (the low 8 bits of a status word); a fixed text for codes that name no refusal */
const char* echo_b200_query_reason(uint32_t code);

#ifdef __cplusplus
}
#endif
#endif
