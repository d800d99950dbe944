/*
 * echo_b200_evaluation.h — one EvaluationOperation (Processes/Evaluation/EvaluationOperation.cs:100-141) driven by a host that
 * brings its own evaluator: the library makes the camera rays, the sample sequence and the per-pixel Accumulator with its noise-driven
 * epoch loop, on device buffers; the host evaluates every sample with the calls of echo_b200_query_device.h in between.
 *
 *   create -> ( next_epoch -> spawn_device, draw_device* -> [the host's evaluator] -> accumulate_device )* -> finish -> destroy
 *
 * These are the kernels the built-in evaluators of echo_b200_render_tiles run, so a host evaluator that computes what a built-in one
 * computes renders the same tiles, bit for bit.
 *
 * Slots. An epoch has `count` slots (next_epoch): active pixels x extend, slot = active-pixel position x extend + s, s = 0 .. extend-1
 * in sample order. Every per-slot buffer (rays, pixels, sample indices, draws, samples) is indexed by slot.
 *
 * Sample sequence. The draws of slot i at dimension d are the draws a built-in evaluator makes for the same pixel and sample index:
 * dimensions 0..3 are the CameraSample (spawn_device), a Next2D occupies d and d + 1. EchoRenderParams.seed picks the sequence,
 * evaluator = ECHO_DISTRIBUTION_STRATIFIED the stratified one. The sample index of slot s of epoch e (from 1) is
 * (epochOffset + e - 1) x extend + s.
 *
 * Epochs. accumulate_device runs Accumulator.Add over every slot of the epoch in sample order per pixel and the stop test of
 * EvaluationOperation.cs:137 (minEpoch, maxEpoch, noiseThreshold); next_epoch then lists the pixels that go on. Call order, refused
 * with ECHO_B200_ERR_INVALID otherwise: spawn, draw and accumulate need an open epoch (opened by next_epoch, closed by accumulate);
 * next_epoch is refused while an epoch is open; finish is refused while an epoch is open and accepted between epochs, which gives a
 * progressive preview.
 *
 * Streams and memory. Every call is enqueued on the stream given to create (a cudaStream_t; NULL = the legacy default stream); the
 * host's own query calls of an epoch go on the same stream. create, next_epoch and finish synchronise it; spawn, draw and accumulate
 * are asynchronous. Every buffer is device memory of the scene's device, except tile_xy and finish's out_rgba. The evaluation owns
 * about 84 bytes per pixel and 12 per slot; the caller owns the rays, draws and samples. Several evaluations may run on one scene at
 * once, on different streams: each owns its buffers and uses none of the scene's. The scene must outlive its evaluations.
 *
 * Refused with ECHO_B200_ERR_INVALID and a message (echo_b200_last_error): a NULL scene or evaluation, an uncommitted or multi-device
 * scene, EchoRenderParams that echo_b200_render_tiles refuses for their sizes, extend or epochs, an evaluator other than 0 or
 * ECHO_DISTRIBUTION_STRATIFIED (bounceLimit and survivability are not read), a negative tile position, more than 2^31 slots
 * (tile_count x tileSize^2 x extend) or 2^30 pixels (split the tiles into several evaluations), components other than 1 or 2, and
 * every call-order violation above.
 */
#ifndef ECHO_B200_EVALUATION_H
#define ECHO_B200_EVALUATION_H

#include "echo_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct EchoEvaluation EchoEvaluation;

/* one EvaluationOperation over tile_count tiles (host buffer tile_xy, as in echo_b200_render_tiles); synchronises `stream` */
int32_t echo_b200_evaluation_create(EchoScene*, const EchoRenderParams* params, const int32_t* tile_xy, uint32_t tile_count, void* stream,
                                    EchoEvaluation** out);
/* closes the previous epoch, if any, and opens the next one: *out_count = its slots, 0 once every pixel has stopped or maxEpoch is
 * reached; synchronises the stream (it reads the active-pixel count) */
int32_t echo_b200_evaluation_next_epoch(EchoEvaluation*, uint64_t* out_count);
/* Camera.SpawnRay of every slot (CameraSample = dimensions 0..3): distance +inf, ignore ECHO_TOKEN_EMPTY; d_pixel_xy (int32 x, y) and
 * d_sample_index (nullable) receive the slot's pixel and sample index */
int32_t echo_b200_evaluation_spawn_device(EchoEvaluation*, EchoRay* d_rays, int32_t* d_pixel_xy, uint32_t* d_sample_index);
/* the draw of every slot at `dimension`: components 1 = Next1D, 2 = Next2D (dimensions d, d + 1); d_out = count x components floats */
int32_t echo_b200_evaluation_draw_device(EchoEvaluation*, uint32_t dimension, uint32_t components, float* d_out);
/* Accumulator.Add of every slot's Float4 (count x 4 floats), in sample order per pixel, then the epoch stop test; closes the epoch */
int32_t echo_b200_evaluation_accumulate_device(EchoEvaluation*, const float* d_samples_rgba);
/* synchronous: out_rgba (host, nullable) = the tiles in echo_b200_render_tiles's layout; d_frame_rgba (device, nullable, width x height
 * Float4) gets (mean * n, n) ADDED as echo_b200_render_frame_device adds it; stats (nullable) = Sample/Evaluated, Sample/Rejected,
 * Pixel/Evaluated and kernelLaunches, every other row zero (those rows belong to the evaluator) */
int32_t echo_b200_evaluation_finish(EchoEvaluation*, float* out_rgba, float* d_frame_rgba, EchoStats* stats);
int32_t echo_b200_evaluation_destroy(EchoEvaluation*);

#ifdef __cplusplus
}
#endif
#endif
