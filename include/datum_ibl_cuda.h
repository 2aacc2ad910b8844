/*
 * libdatum_ibl_cuda — C ABI of the B200 (sm_100a) image-based-lighting bake.
 *
 * Drop-in boundary for the hot path of pniekamp/datum's tools/ibl.cpp.  The
 * reference exposes four C++ free functions in tools/ibl.h:9-15; they take
 * lml/std types, so they cannot be bound directly.  The host shim under
 * datum_b200/host/ keeps those four signatures and forwards plain pointers and
 * sizes to the entry points declared here (see INTEGRATION.md).
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure;
 *     datum_ibl_last_error() then describes the failure (thread-local).
 *     The reference functions return void and never fail; the C++ shim turns a
 *     non-zero status into std::runtime_error, which assetbuilder's main()
 *     already catches (tools/assetbuilder.cpp:968-982).
 *   - there is NO CPU fallback: without a CUDA device datum_ibl_create fails.
 *   - image layout is the reference's: level-major, then face (0 right, 1 left,
 *     2 down, 3 up, 4 forward, 5 back — tools/ibl.cpp:21-26), then rows of
 *     32-bit E5B9G9R9 "rgbe" words (src/math/color.h:154-172);
 *     payload size = sum_i (w>>i)*(h>>i)*6*4 bytes (tools/assetpacker.cpp:488-497).
 *   - a "row" below is a row of the 6*h face-major image of a level; row ranges
 *     let several GPUs split one level.
 *   - host pointers may be pageable; `*_device` entry points take device
 *     pointers and are asynchronous on the context's stream unless stated.
 *   - a context is bound to one device and must be used from one thread at a time.
 */
#ifndef DATUM_IBL_CUDA_H
#define DATUM_IBL_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct datum_ibl_ctx datum_ibl_ctx;

/* texel formats of a level-0 image handed to the SH9 projection, and of float chains (F32, F16) */
#define DATUM_IBL_FORMAT_RGBE 0 /* uint32 E5B9G9R9 words, src/math/color.h:154-172 */
#define DATUM_IBL_FORMAT_F32 1  /* RGBA fp32, the layout of HDRImage::bits (tools/hdr.h:24) */
#define DATUM_IBL_FORMAT_F16 2  /* RGBA IEEE binary16, 8 bytes per texel: VK_FORMAT_R16G16B16A16_SFLOAT */

/* ---- lifetime ------------------------------------------------------------ */

int datum_ibl_create(int device, datum_ibl_ctx **out);
void datum_ibl_destroy(datum_ibl_ctx *ctx);
const char *datum_ibl_last_error(void);

/* the CUDA stream all asynchronous work of the context is issued on (cudaStream_t) */
void *datum_ibl_stream(datum_ibl_ctx *ctx);
int datum_ibl_synchronize(datum_ibl_ctx *ctx);

/* kernels launched by this context since creation (bench.py's gpu_launches) */
uint64_t datum_ibl_launch_count(datum_ibl_ctx *ctx);

/* prefilter kernel variant: 0 = automatic (default); 51-54, 70-73, 80 pin one of the shipped kernels (tests); others exist in the tools build only */
int datum_ibl_set_prefilter_variant(datum_ibl_ctx *ctx, int variant);

/*
 * Development knobs (A/B timing; defaults are what the library measured best): "prefilter_variant" (as above),
 * "sh9_kernel" (0 = column strips, 1 = the row-segment kernel), "sh9_rows_per_item" (0 = automatic).
 */
int datum_ibl_set_tuning(datum_ibl_ctx *ctx, const char *key, int value);

/* bytes of a `levels`-deep cube chain; tools/assetpacker.cpp:488-497 with layers = 6 */
size_t datum_ibl_chain_bytes(int width, int height, int levels);

/* ---- GGX prefilter chain: tools/ibl.cpp:242-279 ----------------------------- */

/*
 * Replaces image_buildmips_cube_ibl(width, height, levels, bits) (tools/ibl.h:9,
 * tools/ibl.cpp:242).  `bits` is the caller's payload (tools/assetbuilder.cpp:439,
 * 484): level 0 pre-filled, levels 1..levels-1 written in place.  Synchronous;
 * includes the host->device copy of level 0 and the device->host copy of the
 * computed levels.  `samples` is the reference's kSamples (tools/ibl.cpp:162: 1024).
 */
int datum_ibl_buildmips_cube_ibl(datum_ibl_ctx *ctx, int width, int height, int levels, int samples, void *bits);

/*
 * A batch of independent bakes (SURVEY.md 8b/8e: "batched probes"; the reference bakes one
 * skybox per write_skybox_asset call, tools/assetbuilder.cpp:416-491).  bits[i] is the i-th
 * caller payload, all of the same width/height/levels, level 0 pre-filled, used exactly like
 * the `bits` of datum_ibl_buildmips_cube_ibl.  `sh` (optional, may be NULL) receives the SH9
 * projection (data/project.comp) of every level 0, count x float[9][3].  Results are those
 * of `count` single calls; the uploads, the kernels and the downloads of consecutive probes
 * overlap on three streams over two device payloads.  Pinned host payloads overlap fully;
 * pageable ones are staged by the driver.  Synchronous.
 */
int datum_ibl_bake_probes(datum_ibl_ctx *ctx, int count, int width, int height, int levels, int samples, void *const *bits, float *sh);

/*
 * Same chain on a device-resident payload.  `d_f32` (optional, may be NULL)
 * receives the fp32 rgb triples handed to rgbe() at tools/ibl.cpp:269 for levels
 * >= 1, level-major starting at level 1 (3 floats per texel).  Asynchronous.
 */
int datum_ibl_buildmips_cube_ibl_device(datum_ibl_ctx *ctx, int width, int height, int levels, int samples, uint32_t *d_bits, float *d_f32);

/*
 * One level of the chain, for a slab of rows: the body of the level loop at
 * tools/ibl.cpp:247-278.  `d_src` is the full (ws x hs x 6) source level, the
 * destination level is (ws/2 x hs/2 x 6); rows [row_begin,row_end) of its
 * 6*(hs/2) rows are written.  `d_dst_words` / `d_dst_f32` point at the START of
 * the destination level (either may be NULL).  roughness = level/(levels-1)
 * (tools/ibl.cpp:251).  Asynchronous.
 */
int datum_ibl_prefilter_level_device(datum_ibl_ctx *ctx, uint32_t const *d_src, int ws, int hs, int level, int levels, int samples, int row_begin, int row_end, uint32_t *d_dst_words, float *d_dst_f32);

/* ---- one probe shared by several GPUs of a node (SURVEY.md 8e "one probe split") ------------ */

/*
 * The reference has no counterpart (its bake is one thread, tools/ibl.cpp:263-272).  Inside a
 * level every destination row is independent, but level L reads all of level L-1
 * (tools/ibl.cpp:249, 274): the GPUs sharing a probe each compute a slab of rows and need the
 * whole level before the next one.  Here the prefilter kernel's epilogue writes its slab into
 * every peer's payload over NVLink (peer stores); the CTA of the launch that finishes last then
 * bumps an arrival counter in every peer's flag block, and each GPU's stream waits on its own
 * counter with a stream memory operation (cuStreamWaitValue32) before the next level: compute,
 * exchange and synchronisation are ONE kernel launch per level, no collective library call.
 *
 * Flag block: DATUM_IBL_PEER_FLAG_BYTES zeroed bytes owned by each rank (the first two 32-bit
 * words are the arrival counters), peer-mapped like the payload.  An "event" is one exchange or
 * barrier; every rank issues the same events in the same order with epochs 1, 2, 3, ...
 *
 * datum_ibl_peer_alloc: zeroed device memory other PROCESSES can map; `handle` receives the 64
 * bytes of its cudaIpcMemHandle_t, to be sent to the peers by any means (torch.distributed in
 * dist.py).  datum_ibl_peer_open / _close: map / unmap a peer's allocation in this process.
 * Inside ONE process use the device-list entry points below instead (plain peer access).
 */
#define DATUM_IBL_MAX_PEERS 7
#define DATUM_IBL_IPC_HANDLE_BYTES 64
#define DATUM_IBL_PEER_FLAG_BYTES 256
int datum_ibl_peer_alloc(datum_ibl_ctx *ctx, size_t bytes, void **d_ptr, void *handle);
int datum_ibl_peer_free(datum_ibl_ctx *ctx, void *d_ptr);
int datum_ibl_peer_open(datum_ibl_ctx *ctx, void const *handle, void **d_ptr);
int datum_ibl_peer_close(datum_ibl_ctx *ctx, void *d_ptr);

/*
 * datum_ibl_prefilter_level_device for rank `rank` of `world` (<= 8) GPUs sharing the probe:
 * d_dst_words[r] points at the START of the destination level in rank r's payload as mapped HERE
 * (r == rank: the local one); every rgbe word of the slab goes to all of them.  With d_flags
 * (by rank, may be NULL) and epoch > 0 the launch also signals its completion to the peers and the
 * context's stream then waits for the arrivals of all peers: after this call has been issued on every
 * rank, work queued behind it sees the complete level.  Asynchronous.
 */
int datum_ibl_prefilter_level_peers(datum_ibl_ctx *ctx, uint32_t const *d_src, int ws, int hs, int level, int levels, int samples, int row_begin, int row_end, int rank, int world, uint32_t *const *d_dst_words, uint32_t *const *d_flags, uint32_t epoch);

/*
 * Barrier of the `world` (<= 8) GPUs on the context's stream (one tiny signal launch + a stream
 * wait): d_flags[r] = rank r's flag block (d_flags[rank] the local one).  Asynchronous.  A peer that
 * never arrives is detected by datum_ibl_synchronize (datum_ibl_set_peer_timeout_ms, default 60 s),
 * which releases the waits and returns an error; no device-side trap.
 */
int datum_ibl_peer_barrier(datum_ibl_ctx *ctx, int rank, int world, uint32_t *const *d_flags, uint32_t epoch);
int datum_ibl_set_peer_timeout_ms(datum_ibl_ctx *ctx, int milliseconds);

/* ---- device list: several GPUs of a node driven from ONE process (SURVEY.md 8b last row) ------- */

/*
 * tools/assetbuilder.cpp is one process whose main thread calls image_buildmips_cube_ibl once per
 * skybox (:465, :486; write_core :778).  A datum_ibl_multi owns one context per listed device and enables
 * plain peer access between them (cudaDeviceEnablePeerAccess; no IPC handles, no second process).  At most
 * 8 devices; a device may be listed more than once (two contexts on one GPU — how the exchange path is
 * tested on a one-GPU box).  Every call is synchronous and must come from one thread at a time.
 */
typedef struct datum_ibl_multi datum_ibl_multi;

int datum_ibl_multi_create(int ndev, int const *devices, datum_ibl_multi **out);
void datum_ibl_multi_destroy(datum_ibl_multi *multi);
int datum_ibl_multi_device_count(datum_ibl_multi *multi);
datum_ibl_ctx *datum_ibl_multi_context(datum_ibl_multi *multi, int index);   /* the context of devices[index] (owned by multi) */

/*
 * datum_ibl_buildmips_cube_ibl with ONE probe shared by the devices (BASELINE config 3): the rows of every
 * level above 6x16^2 texels are split evenly, each device's prefilter launch stores its slab into all
 * payloads over NVLink and signals the peers, the streams wait on the arrival counters; smaller levels are
 * computed by every device.  Level 0 is uploaded once and copied device to device; the result comes back
 * from the first device.  Words equal the single-device bake's up to the re-cut tiles (>= 99.99 % identical).
 */
int datum_ibl_multi_buildmips_cube_ibl(datum_ibl_multi *multi, int width, int height, int levels, int samples, void *bits);

/* datum_ibl_bake_probes with probe p on devices[p % ndev] (BASELINE config 4); results identical to one device's */
int datum_ibl_multi_bake_probes(datum_ibl_multi *multi, int count, int width, int height, int levels, int samples, void *const *bits, float *sh);

/* datum_ibl_project_sh9 with the cube's rows split over the devices (BASELINE config 5); slabs are added in device order on the host */
int datum_ibl_multi_project_sh9(datum_ibl_multi *multi, void const *level0, int format, int width, int height, float *sh);

/* the first two with the device list passed per call; the library keeps one datum_ibl_multi per distinct list */
int datum_ibl_buildmips_cube_ibl_devices(int ndev, int const *devices, int width, int height, int levels, int samples, void *bits);
int datum_ibl_bake_probes_devices(int ndev, int const *devices, int count, int width, int height, int levels, int samples, void *const *bits, float *sh);

/* ---- equirectangular HDR image -> cube: tools/hdr.cpp:331-359, tools/ibl.cpp:283-288 ---- */

/*
 * Replaces image_pack_cube(image, width, height, 1, bits) (tools/hdr.h:39,
 * tools/hdr.cpp:331) as the IBL path uses it (levels == 1): per cube texel the
 * box-filtered bilinear equirect lookup of HDRImage::sample (hdr.cpp:44-74),
 * rgbe(), then image_blend_edges (hdr.cpp:173-318).  `pixels` = HDRImage::bits,
 * imgwidth*imgheight RGBA fp32 on the host; `bits` receives 6*width*height words.
 * Synchronous.
 */
int datum_ibl_pack_cube(datum_ibl_ctx *ctx, int imgwidth, int imgheight, float const *pixels, int width, int height, void *bits);

/*
 * Replaces image_pack_cube_ibl(image, width, height, levels, bits) (tools/ibl.h:11,
 * tools/ibl.cpp:283-288): the resample above, then the prefilter chain; the whole
 * payload (level 0 included) is written to the host buffer `bits`.  Synchronous.
 */
int datum_ibl_pack_cube_ibl(datum_ibl_ctx *ctx, int imgwidth, int imgheight, float const *pixels, int width, int height, int levels, int samples, void *bits);

/* ---- six face images -> cube: tools/assetbuilder.cpp:416-470 ------------------------ */

/*
 * Replaces the per-image loop of write_skybox_asset(fout, id, paths)
 * (tools/assetbuilder.cpp:443-462): for each of the six QImage::Format_ARGB32
 * images (0xAARRGGBB pixels, `argb` = 6*width*height of them on the host, faces in
 * the caller's order rt, lf, dn, up, fr, bk) setPixel(rgbe(srgba(pixel)))
 * (src/math/color.h:125-128, 154-162), QImage::mirrored() and the memcpy into
 * level 0 of the payload.  `bits` receives 6*width*height words.  Synchronous.
 */
int datum_ibl_ingest_cube_argb32(datum_ibl_ctx *ctx, int width, int height, uint32_t const *argb, void *bits);

/*
 * The whole of write_skybox_asset(fout, id, paths) between image loading and
 * write_imag_asset (tools/assetbuilder.cpp:443-465): the ingest above followed by
 * image_buildmips_cube_ibl, level 0 never leaving the device in between.  `bits`
 * receives the full payload of image_datasize(width, height, 6, levels) bytes.
 * Synchronous.
 */
int datum_ibl_ingest_cube_argb32_ibl(datum_ibl_ctx *ctx, int width, int height, int levels, int samples, uint32_t const *argb, void *bits);

/* ---- SH9 irradiance projection: data/project.comp:23-106 -------------------- */

/*
 * Partial sums of the projection over rows [row_begin,row_end) of a level-0
 * cube: 27 unnormalised coefficients in [k][rgb] order (k as in
 * data/project.comp:64-92) followed by the sum of solid-angle weights.
 * `d_partial` = 28 doubles on the device; ranks sharing one probe all-reduce
 * them before datum_ibl_sh9_finish.  Asynchronous.
 */
int datum_ibl_sh9_partial_device(datum_ibl_ctx *ctx, void const *d_level0, int format, int width, int height, int row_begin, int row_end, double *d_partial);

/*
 * The same for a cube shared by `world` (<= 8) GPUs of a node without a collective: d_slots[r] is rank r's
 * peer-mapped array of world x 28 doubles (d_slots[rank] the local one).  The slab's 28 sums are written to
 * row [rank] of EVERY array by the block that finishes last (NVLink peer stores), which then signals the
 * peers' flag blocks (d_flags, epoch as above; NULL: no signal, no wait); the stream waits for all arrivals,
 * after which every rank holds all rows and adds them in rank order.  One launch.  Asynchronous.
 */
int datum_ibl_sh9_partial_peers(datum_ibl_ctx *ctx, void const *d_level0, int format, int width, int height, int row_begin, int row_end, int rank, int world, double *const *d_slots, uint32_t *const *d_flags, uint32_t epoch);

/* data/project.comp:99-105: sh[k] = partial[k] * 4*pi / partial[27]; host arithmetic on 28 numbers */
void datum_ibl_sh9_finish(double const *partial, float *sh);

/*
 * Whole projection of a host-resident level-0 cube; `sh` = float[9][3], the
 * layout of `Irradiance` (src/renderer/envmap.h:112-115).  Synchronous.
 */
int datum_ibl_project_sh9(datum_ibl_ctx *ctx, void const *level0, int format, int width, int height, float *sh);

/*
 * Diffuse irradiance cube from SH9: E(n) of data/lighting.inc:351-366, 371
 * (cosine-lobe band factors, max(.,0)) at the texel directions of
 * tools/ibl.cpp:269.  Writes rgbe words and/or fp32 rgb triples (either may be
 * NULL) for a (width x height x 6) cube on the host.  Synchronous.
 */
int datum_ibl_sh9_irradiance_cube(datum_ibl_ctx *ctx, float const *sh, int width, int height, uint32_t *words, float *f32);

/* ---- 2D LUTs of tools/ibl.h ---------------------------------------------------- */

/* Replaces image_pack_envbrdf(width, height, bits) (tools/ibl.h:13, tools/ibl.cpp:292-308); host buffer. */
int datum_ibl_pack_envbrdf(datum_ibl_ctx *ctx, int width, int height, int samples, void *bits);

/* Replaces image_pack_watercolor(...) (tools/ibl.h:15, tools/ibl.cpp:312-329); colours are float[3]; host buffer. */
int datum_ibl_pack_watercolor(datum_ibl_ctx *ctx, float const *deepcolor, float const *shallowcolor, float depthscale, float const *fresnelcolor, float fresnelbias, float fresnelpower, int width, int height, void *bits);

/* ---- measurement helpers -------------------------------------------------------- */

/*
 * FP32 FMA throughput of the device in TFLOP/s (2 flop per FMA), measured with
 * a register-resident FFMA chain kernel timed with CUDA events; the denominator
 * of the prefilter kernel's roofline fraction.
 */
int datum_ibl_measure_fp32_peak(datum_ibl_ctx *ctx, double *tflops);

/* the same measurement issued as packed two-wide fma.rn.f32x2 (SASS FFMA2, new on sm_100) */
int datum_ibl_measure_fp32x2_peak(datum_ibl_ctx *ctx, double *tflops);

/*
 * CUDA-event timings of the dominant kernel (the level-1 prefilter launch of
 * every chain since the last reset, at most 512): number of launches averaged,
 * their mean duration, and the texel-samples one such launch processes.
 * Synchronises the context's stream.
 */
int datum_ibl_dominant_kernel_stats(datum_ibl_ctx *ctx, int reset, int *launches, double *avg_ms, double *texel_samples_per_launch);

/* milliseconds the device spent in the prefilter kernels of the last chain call (CUDA events) */
int datum_ibl_last_prefilter_ms(datum_ibl_ctx *ctx, float *ms);

/* ---- GGX prefilter of float chains: RGBA32F / RGBA16F, no rgbe re-quantisation ---------- */

/*
 * The chain of datum_ibl_buildmips_cube_ibl on a cube of float texels: `format` is DATUM_IBL_FORMAT_F32
 * (16 bytes per texel) or DATUM_IBL_FORMAT_F16 (8 bytes).  Same layout (level-major, then face 0..5, then
 * rows; the texel offsets of datum_ibl_chain_bytes' levels, texel size of the format), level 0 pre-filled.
 * Level L is convolved from level L-1 as stored in the chain (binary16 widened to fp32) with the arithmetic
 * of tools/ibl.cpp:160-187; input alpha is ignored, output alpha is 1.0.  F32 stores the fp32 result,
 * F16 stores min(x, 65504) rounded to nearest-even.  Level-0 texels must be finite and non-negative; every
 * binary16 value works, fp32 values up to 2^52 (4.5e15).  `samples` 1..4096.
 * Host chain (pageable or pinned), synchronous.
 */
int datum_ibl_buildmips_cube_float(datum_ibl_ctx *ctx, int format, int width, int height, int levels, int samples, void *chain);

/*
 * The same on a device-resident chain (aligned to the texel size); asynchronous on the context's stream.
 * `d_f32` (optional) receives the fp32 rgb of levels >= 1 before rounding, in the layout of
 * datum_ibl_buildmips_cube_ibl_device's d_f32.
 */
int datum_ibl_buildmips_cube_float_device(datum_ibl_ctx *ctx, int format, int width, int height, int levels, int samples, void *d_chain, float *d_f32);

/* One level of a float chain, rows [row_begin, row_end) of the destination; device pointers, asynchronous. */
int datum_ibl_prefilter_level_float_device(datum_ibl_ctx *ctx, int format, void const *d_src, int ws, int hs, int level, int levels, int samples, int row_begin, int row_end, void *d_dst, float *d_dst_f32);

/*
 * datum_ibl_bake_probes for float chains: chains[i] is the i-th host chain (pageable or pinned), all of the same
 * format, width/height/levels, laid out and level 0 pre-filled as for datum_ibl_buildmips_cube_float.  `sh`
 * (optional, may be NULL) receives the SH9 projection of every level 0 as read in the chain's format,
 * count x float[9][3].  Every chain's bytes are those of a single datum_ibl_buildmips_cube_float call; small
 * probes share launches and the uploads, kernels and downloads of consecutive groups overlap as in
 * datum_ibl_bake_probes.  Synchronous.
 */
int datum_ibl_bake_probes_float(datum_ibl_ctx *ctx, int format, int count, int width, int height, int levels, int samples, void *const *chains, float *sh);

/* datum_ibl_bake_probes_float with probe p on devices[p % ndev] (see datum_ibl_multi_bake_probes); results identical to one device's */
int datum_ibl_multi_bake_probes_float(datum_ibl_multi *multi, int format, int count, int width, int height, int levels, int samples, void *const *chains, float *sh);

/*
 * datum_ibl_prefilter_level_peers for a float chain: rank `rank` of `world` (<= 8) GPUs sharing the probe
 * computes rows [row_begin, row_end) of the level and stores every texel of the format into d_dst[r], the START
 * of the destination level in rank r's chain as mapped HERE (r == rank: the local one).  With d_flags (flag
 * blocks by rank, may be NULL: no signal, no wait) and epoch > 0 the launch signals its completion to the peers
 * (an empty slab still arrives) and the context's stream then waits for the arrivals of all peers.  Pointers
 * aligned to the texel size, `samples` 1..4096.  Asynchronous.
 */
int datum_ibl_prefilter_level_float_peers(datum_ibl_ctx *ctx, int format, void const *d_src, int ws, int hs, int level, int levels, int samples, int row_begin, int row_end, int rank, int world, void *const *d_dst, uint32_t *const *d_flags, uint32_t epoch);

/*
 * datum_ibl_buildmips_cube_float with ONE probe shared by the devices, the float counterpart of
 * datum_ibl_multi_buildmips_cube_ibl: the same split of rows, peer stores, arrival counters and uploads.  Level 0
 * of the result is the caller's; the other levels equal the single-device chain's up to the re-cut tiles
 * (F32 within 1e-4 of a texel's largest channel, F16 within 1 ulp).  One device: datum_ibl_buildmips_cube_float.
 * Host chain, synchronous.
 */
int datum_ibl_multi_buildmips_cube_float(datum_ibl_multi *multi, int format, int width, int height, int levels, int samples, void *chain);

/* ---- equirect HDR image or six face images -> level 0 (+ chain) of a float chain ---------------- */

/*
 * datum_ibl_pack_cube with level 0 stored in `format` (DATUM_IBL_FORMAT_F32 or DATUM_IBL_FORMAT_F16) instead of
 * rgbe words.  Per cube texel the arithmetic of the rgbe resample up to sum / totalweight (the same box of
 * bilinear taps, fp32 loop counters), then the format's texel: F32 stores the fp32 rgb, F16 stores min(x, 65504)
 * rounded to nearest-even; alpha is 1.0.  The edge blend then runs the reference's twelve loops in order with the
 * same 0.3/0.4/0.3 arithmetic; each loop reads the texels as stored (halves widened, corners written by earlier
 * loops included) and stores its results in the format, so an F16 corner is rounded once per loop that writes
 * it, as an rgbe corner is re-encoded.  Pixel rgb must be finite and non-negative, and below 2^52 for F32 (the
 * level-0 rules of datum_ibl_buildmips_cube_float; not checked); F16 clamps texels above 65504.  `pixels` =
 * imgwidth*imgheight RGBA fp32 on the host; `texels` receives the 6*width*height texels of level 0 (host,
 * pageable or pinned).  Synchronous.
 */
int datum_ibl_pack_cube_float(datum_ibl_ctx *ctx, int format, int imgwidth, int imgheight, float const *pixels, int width, int height, void *texels);

/*
 * The level 0 above followed by the chain of datum_ibl_buildmips_cube_float, level 0 never leaving the device in
 * between.  `chain` (host, pageable or pinned) receives the whole chain, level 0 included, in the layout of
 * datum_ibl_buildmips_cube_float; its levels >= 1 are those datum_ibl_buildmips_cube_float makes from that
 * level 0.  `samples` 1..4096.  Synchronous.
 */
int datum_ibl_pack_cube_float_ibl(datum_ibl_ctx *ctx, int format, int imgwidth, int imgheight, float const *pixels, int width, int height, int levels, int samples, void *chain);

/*
 * datum_ibl_ingest_cube_argb32 with level 0 stored in `format`: per pixel the linear rgb of srgba(pixel)
 * (pow(c/255, 2.2f), the same 256 values the rgbe ingest encodes) stored as F32 or F16 texels with alpha 1.0,
 * rows mirrored vertically, faces in argument order.  `texels` receives 6*width*height texels (host, pageable
 * or pinned).  Synchronous.
 */
int datum_ibl_ingest_cube_argb32_float(datum_ibl_ctx *ctx, int format, int width, int height, uint32_t const *argb, void *texels);

/* The ingest above followed by the chain of datum_ibl_buildmips_cube_float, as datum_ibl_pack_cube_float_ibl. */
int datum_ibl_ingest_cube_argb32_float_ibl(datum_ibl_ctx *ctx, int format, int width, int height, int levels, int samples, uint32_t const *argb, void *chain);

#ifdef __cplusplus
}
#endif

#endif
