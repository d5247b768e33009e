/* strolle_b200 — C ABI of the B200-native Strolle hot path.
 *
 * Drop-in boundary for the per-pixel GI path of Patryk27/strolle: the functions
 * below are what a Rust `extern "C"` shim behind `strolle::Engine<P>` binds in
 * place of the wgpu compute dispatches (CameraComputePass::run,
 * strolle/src/camera_controller/pass.rs:33-63) and buffer flushes
 * (strolle/src/buffers/mapped_storage_buffer.rs:108-140).  Each entry point
 * cites the reference method it replaces.  Plain pointers and sizes only; no
 * torch / CUDA types.  See INTEGRATION.md for the reference-side binding.
 *
 * Conventions: every function returns ST_OK (0) or a negative error code and
 * never aborts across the ABI; st_last_error() gives the message (the
 * reference panics instead, e.g. strolle/src/triangles.rs:44-53).  Handles are
 * caller-chosen opaque u64 (the reference's Params associated types,
 * strolle/src/lib.rs:402-409).  Mutating calls are externally synchronised
 * (single writer), like `ResMut<Engine>` in bevy-strolle.
 */
#ifndef STROLLE_B200_H
#define STROLLE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct st_engine st_engine;
typedef uint64_t st_handle;
typedef int32_t st_camera_handle;

enum { ST_OK = 0, ST_ERR_CUDA = -1, ST_ERR_INVALID = -2, ST_ERR_NOT_FOUND = -3, ST_ERR_LIMIT = -4 };

/* strolle::MeshTriangle (strolle/src/mesh_triangle.rs:7-12), object space */
typedef struct st_mesh_triangle {
    float positions[3][3];
    float normals[3][3];
    float uvs[3][2];
    float tangents[3][4];
} st_mesh_triangle;

/* strolle::Material (strolle/src/material.rs:8-23); textures are a later row (SURVEY §8f-3) */
typedef struct st_material {
    float base_color[4];
    float emissive[4];
    float perceptual_roughness;
    float metallic;
    float reflectance;
    float ior;
    int32_t alpha_blend; /* AlphaMode::Blend != 0 (strolle/src/material.rs:76-91) */
} st_material;

/* strolle::Light::{Point,Spot} (strolle/src/light.rs:6-22) */
enum { ST_LIGHT_POINT = 1, ST_LIGHT_SPOT = 2 };
typedef struct st_light {
    int32_t kind;
    float position[3];
    float radius;
    float color[3];
    float range;
    float direction[3]; /* spot only */
    float angle;        /* spot only */
} st_light;

/* strolle::CameraMode (strolle/src/camera.rs:83-105) */
enum {
    ST_MODE_IMAGE = 0, ST_MODE_DI_DIFFUSE = 1, ST_MODE_DI_SPECULAR = 2, ST_MODE_GI_DIFFUSE = 3,
    ST_MODE_GI_SPECULAR = 4, ST_MODE_BVH_HEATMAP = 5, ST_MODE_REFERENCE = 6
};
/* strolle::Camera (strolle/src/camera.rs:8-14); matrices column-major like glam::Mat4 */
typedef struct st_camera {
    int32_t mode;
    int32_t denoise;   /* CameraMode::*{denoise} */
    int32_t ref_depth; /* CameraMode::Reference{depth} */
    uint32_t width, height; /* CameraViewport::size */
    float transform[16];
    float projection[16];
} st_camera;

/* Output pixel formats for st_render_camera (the reference composes into the caller's
 * TextureView of CameraViewport::format, strolle/src/camera.rs:170-185).  RGBA32F: 16 B/px, the composed
 * frame as is.  RGBA8_SRGB: 4 B/px, Rgba8UnormSrgb (clamp, sRGB OETF, round to nearest), alpha 255.  RGBA16F:
 * 8 B/px, IEEE binary16 per channel with round-to-nearest-even (what a render-target store to Rgba16Float does:
 * above 65504 becomes inf, NaN stays NaN), alpha 1.0 (0x3C00); the format of Bevy's HDR view target. */
enum { ST_FORMAT_RGBA32F = 0, ST_FORMAT_RGBA8_SRGB = 1, ST_FORMAT_RGBA16F = 2 };

const char* st_last_error(void);

/* Engine::new (strolle/src/lib.rs:132-158).  `device` = CUDA ordinal. */
int st_engine_create(int device, st_engine** out);
void st_engine_destroy(st_engine* e);

/* Engine::insert_mesh / remove_mesh (lib.rs:161-171) */
int st_insert_mesh(st_engine* e, st_handle mesh, const st_mesh_triangle* triangles, size_t count);
int st_remove_mesh(st_engine* e, st_handle mesh);
/* Engine::insert_material / has_material / remove_material (lib.rs:174-195) */
int st_insert_material(st_engine* e, st_handle material, const st_material* m);
int st_has_material(st_engine* e, st_handle material);
int st_remove_material(st_engine* e, st_handle material);
/* Engine::insert_image / remove_image (lib.rs:198-214), ImageData::Raw only: tightly packed RGBA8 pixels in
 * the atlas format Rgba8UnormSrgb (strolle/src/images.rs:38-43).  ST_ERR_LIMIT when the 8192^2 atlas is full
 * (the reference warns and drops the image, images.rs:71-79). */
int st_insert_image(st_engine* e, st_handle image, const uint8_t* rgba8, uint32_t width, uint32_t height);
int st_remove_image(st_engine* e, st_handle image);
/* ImageData::Texture { is_dynamic: true } (strolle/src/images.rs:97-102): an image whose texels live in a caller-owned surface of width x height
 * RGBA8 texels in the atlas format Rgba8UnormSrgb (what a camera renders with ST_FORMAT_RGBA8_SRGB), rows `pitch_bytes` apart (0 = packed).
 * The image gets its atlas rectangle as st_insert_image would place it (a handle that has one of the same size keeps it); this call copies
 * nothing.  Each st_tick then copies every dynamic image's surface into its rectangle (Images::flush, images.rs:189-214), enqueued on the
 * engine's stream before anything else the tick enqueues, and after every write this engine has queued to the surface (its kernel stores,
 * its output copies under ST_OPT_ASYNC_OUTPUT, and in a strip group every member's rows); writes from other streams are the caller's to
 * order.  So every camera rendered after a tick sees the same snapshot, and a frame a camera writes into the surface is seen by the
 * cameras of the next frame.  `src` may be memory of this engine's device, of a device it can reach by peer access, managed memory, or
 * page-locked host memory (read through its device pointer); it must stay valid while the image is dynamic.  st_remove_image,
 * st_insert_image on the same handle, or st_insert_dynamic_image with another surface end the refresh, and synchronise the engine's
 * stream before returning, so the old surface may be freed then.  ST_ERR_INVALID for a NULL src, a zero size, a pitch below 4 * width, an
 * address or pitch not a multiple of 4, pageable host memory, or device memory this device cannot reach; ST_ERR_LIMIT when the atlas is
 * full.  A refused call changes nothing: an image already on the handle keeps its rectangle, its texels and its refresh. */
int st_insert_dynamic_image(st_engine* e, st_handle image, const void* src, size_t pitch_bytes, uint32_t width, uint32_t height);
/* The Option<ImageHandle> fields of strolle::Material (strolle/src/material.rs:13-22); bit i of `mask` = texture i set
 * (0 base_color, 1 emissive, 2 metallic_roughness, 3 normal_map — the last is carried but unused, as in the reference). */
typedef struct st_material_textures { st_handle base_color, emissive, metallic_roughness, normal_map; uint32_t mask; } st_material_textures;
int st_set_material_textures(st_engine* e, st_handle material, const st_material_textures* textures);
/* Engine::insert_instance / remove_instance (lib.rs:217-229); affine = glam::Affine3A as
 * matrix3 columns x,y,z then translation (12 floats) */
int st_insert_instance(st_engine* e, st_handle instance, st_handle mesh, st_handle material, const float affine[12]);
int st_remove_instance(st_engine* e, st_handle instance);
/* Engine::insert_light / remove_light (lib.rs:232-239) */
int st_insert_light(st_engine* e, st_handle light, const st_light* l);
int st_remove_light(st_engine* e, st_handle light);
/* Engine::update_sun (lib.rs:242-245) */
int st_update_sun(st_engine* e, float azimuth, float altitude);

/* Engine::create_camera / update_camera / delete_camera (lib.rs:252-294) */
int st_create_camera(st_engine* e, const st_camera* camera, st_camera_handle* out);
int st_update_camera(st_engine* e, st_camera_handle camera, const st_camera* desc);
int st_delete_camera(st_engine* e, st_camera_handle camera);

/* Engine::tick (lib.rs:301-395): bakes dirty instances, rebuilds + uploads the BVH, lights,
 * materials, world; must precede st_render_camera each frame. */
int st_tick(st_engine* e);

/* Engine::render_camera (lib.rs:279-286 -> CameraController::render,
 * strolle/src/camera_controller.rs:87-174): runs the frame's pass schedule on the engine's
 * stream.  If `host_out` is non-NULL the composed frame (width*height pixels of `format`) is
 * copied to it and the call returns when the copy is done; with NULL the call only enqueues
 * (use st_synchronize). */
int st_render_camera(st_engine* e, st_camera_handle camera, void* host_out, int format);
/* Converts the camera's composed frame to `format` and copies it to host memory (what
 * st_render_camera does when host_out != NULL), without re-running the passes. */
int st_copy_output(st_engine* e, st_camera_handle camera, void* host_out, int format);
/* Engine::render_camera into a caller-owned surface (frame_composition.rs pass: scissor at viewport.position, LoadOp::Load,
 * strolle/src/camera_controller/passes/frame_composition.rs:108-131).
 * `dst` = address of the camera's pixel (0,0) inside the surface; `pitch_bytes` = bytes between rows (0 = width * bytes per pixel).
 * dst may be device memory (this engine's device, or a device it can reach by peer access, or managed memory) or host memory
 * (pinned or pageable); the kind is found with cudaPointerGetAttributes.  Only the width x height rectangle is written.
 * Device memory: one kernel on the engine's stream stores straight into dst (no staging, no host round trip); the call returns
 * once enqueued (order with st_synchronize or st_set_stream).  Host memory: as st_render_camera with host_out (blocking unless
 * ST_OPT_ASYNC_OUTPUT).  ST_ERR_INVALID, before any pass runs and with nothing written, for a NULL dst, an unknown format, a
 * nonzero pitch below width * bytes per pixel, a dst or pitch that is not a multiple of the bytes per pixel (16 / 8 / 4), or device
 * memory this engine's device cannot reach. */
int st_render_camera_to(st_engine* e, st_camera_handle camera, void* dst, size_t pitch_bytes, int format);
int st_synchronize(st_engine* e);

/* ---- several cameras per frame (no reference counterpart: the reference renders one camera per call) ---- */
/* Renders `n` cameras of this engine for the current frame.  The result is, camera for camera, what st_render_camera_to(e, cameras[i],
 * dsts[i], pitch_bytes[i], format) gives when called for i = 0..n-1 in order: bit-identical buffers and output bytes.  Cameras with the
 * same width, height, mode, denoise and ref_depth run as ONE launch per pass (the view index is blockIdx.z); groups run in the order of
 * their first camera in the list, a group larger than one launch holds runs as several launches per pass.  dsts == NULL, or
 * dsts[i] == NULL: no output for that camera (enqueue only, as st_render_camera with NULL).  pitch_bytes may be NULL (all packed).
 * Device surfaces only enqueue (one store launch per group); host surfaces get one copy each and the call blocks unless
 * ST_OPT_ASYNC_OUTPUT.  Everything is checked before any pass runs; on a refusal nothing is rendered or written: ST_ERR_NOT_FOUND for an
 * unknown or deleted camera, ST_ERR_INVALID for n <= 0, a camera listed twice, a camera restricted to a row strip
 * (st_camera_set_strip) or linked into a strip group, a surface st_render_camera_to refuses, or a call before the first st_tick. */
int st_render_cameras(st_engine* e, const st_camera_handle* cameras, int n, void* const* dsts, const size_t* pitch_bytes, int format);

/* ---- hooks that the reference does not have (SURVEY §8b) -------------------------------- */
/* Explicit per-dispatch seeds: seed(frame f, dispatch k) = pcg(base ^ (f*64 + k)); the reference
 * draws rand::thread_rng() per dispatch (camera_controller.rs:189-194) and is not reproducible. */
int st_set_seed_base(st_engine* e, uint32_t base);
/* 256x256 RGBA8 blue-noise tile (strolle/src/noise.rs:30-66 embeds a PNG; here the host passes bytes) */
int st_set_blue_noise(st_engine* e, const uint8_t* rgba8_256x256);
/* Copies a per-camera buffer (names = fields of CameraBuffers, strolle/src/camera_controller/
 * buffers.rs:9-51; double-buffered ones take _a/_b) to host.  Returns #floats available via
 * *count; copies min(cap, count). */
int st_read_buffer(st_engine* e, st_camera_handle camera, const char* name, float* dst, size_t cap_floats, size_t* count);
/* Scene buffers as uploaded: "triangles", "bvh", "materials", "lights", "world", "transmittance_lut",
 * "scattering_lut", "sky_lut". */
int st_read_scene(st_engine* e, const char* name, float* dst, size_t cap_floats, size_t* count);
/* An image's atlas rectangle (static or dynamic), tightly packed RGBA8, after the work queued on the engine's stream: *bytes = width *
 * height * 4; with dst == NULL only the size is returned, cap_bytes below it is ST_ERR_LIMIT.  ST_ERR_NOT_FOUND for an unknown image. */
int st_read_image(st_engine* e, st_handle image, uint8_t* dst, size_t cap_bytes, size_t* bytes);
int st_bvh_depth(st_engine* e, int* depth);
uint32_t st_frame(st_engine* e);
/* Sets the id of the frame the next st_tick prepares (ids start at 1, strolle/src/lib.rs:152).  Used by the
 * sample-parallel reference mode: rank g renders accumulations g+1, g+1+N, ... (SURVEY §8e, config C5). */
int st_set_frame(st_engine* e, uint32_t frame);
/* Ray-stream entry points (the ref_tracing / *_spatial_resampling::trace shape): `rays` = n x 8
 * host floats (origin.xyz, len, dir.xyz, pad).  closest: out = n x 12 floats (packed hit d0, d1
 * as in strolle-gpu/src/hit.rs:112-120, then distance, triangle id bits, material id bits,
 * used_memory).  any: out = n u32 flags.  `device_ms` (optional) receives kernel time. */
int st_trace_closest(st_engine* e, const float* rays, size_t n, float* out, float* device_ms);
int st_trace_any(st_engine* e, const float* rays, size_t n, uint32_t* out, float* device_ms);
/* elementary functions as evaluated on the device (op: 0 sin, 1 cos, 2 acos, 3 atan2, 4 exp, 5 pow, 6 glam's acos_approx) */
int st_device_math(st_engine* e, int op, const float* a, const float* b, float* out, size_t n);
/* Per-pass device time (ms, CUDA events) accumulated since the last reset; `ms`/`launches`
 * have ST_PASS_COUNT entries indexed by st_pass_name(). */
#define ST_PASS_COUNT 27
int st_enable_timing(st_engine* e, int enabled);
int st_pass_times(st_engine* e, float* ms, uint32_t* launches, int reset);
const char* st_pass_name(int pass);
/* K22 frame_denoising::wavelet per à-trous iteration i (stride 2^i, strolle/src/camera_controller/passes/frame_denoising.rs:161-189):
 * device time (ms) and launches accumulated while timing is enabled; 5 entries each. */
int st_wavelet_times(st_engine* e, float* ms5, uint32_t* launches5, int reset);
/* Engine options.  ST_OPT_SVGF_FAST_MATH (default 1): the SVGF edge-stopping weights (K21/K22) use the
 * GPU's SFU approximations (ex2/sqrt/rcp.approx, <= 2 ulp) and fused multiply-adds, like a GLSL compiler
 * does for the reference's shaders; 0 selects strict IEEE arithmetic with polynomial exp, which makes the
 * denoiser bit-identical to the CPU oracle (everything else is bit-identical in both modes). */
enum { ST_OPT_SVGF_FAST_MATH = 1, ST_OPT_ASYNC_OUTPUT = 2, ST_OPT_HALO_NCCL = 3, ST_OPT_WAVELET_TILED = 4, ST_OPT_WAVELET_TILE_CFG = 5, ST_OPT_FUSE_REPROJECT = 6, ST_OPT_BVH_REUSE = 7, ST_OPT_VARIANCE_TILED = 8, ST_OPT_SHADING_FAST_MATH = 9, ST_OPT_STRIP_FUSED = 10, ST_OPT_FUSED_PASSES = 11, ST_OPT_STRIP_DMA = 12, ST_OPT_WAVELET_PAIRED = 13 };
/* ST_OPT_WAVELET_PAIRED (default 1; only with ST_OPT_SVGF_FAST_MATH, and never under the exchange-point strip transports, which ship the
 * named buffers between iterations): the wide-stride à-trous iterations, whose taps are scattered by the per-pixel jitter, read the DI and
 * GI signal as one interleaved 32-byte record per pixel (private scratch; one full sector and one 256-bit load per tap instead of two
 * half-used sectors).  1 = the stride-16 iteration reads records written by the stride-8 iteration; 2 = strides 8 and 16 both do (the
 * stride-4 iteration writes the records, the stride-8 iteration runs the gather kernel, which measured slower than the tile-staged one:
 * 65.6 vs 61.8 us at 1080p); 0 = planar buffers throughout.  Stride 16: 78.1 -> 70.0 us (Cornell), 113.5 -> 98.7 us (dungeon).  Same values in
 * every layout; `*_diff_stash` then keeps the output of the last planar iteration. */
#define ST_WAVELET_PAIRED_DEFAULT 1
/* ST_OPT_STRIP_DMA (fused strip transport only): which halos travel by copy engine (one side stream per neighbour, flag raised behind the
 * copy) instead of the producing kernel's own mirror stores.  1 = the 128-row halos of gi_reservoirs[1] / [2] (64 B per pixel, the bulk of
 * what travels), pushed right after the kernel that produced them and overlapping the DI passes that follow; 2 = also the 128 G-buffer rows
 * (prim_gbuffer_d0 / d1, surface map, surface_nd: 64 B per pixel) next to each strip edge right after the primary pass, instead of every
 * strip recomputing its neighbours' rows (which costs an inner strip of an 8-GPU frame two thirds of a G-buffer pass); 3 = also
 * di_reservoirs[1] and the preview pass's gi_reservoirs[3] (measured slower at 2 GPUs: 1.398 vs 1.351 ms — the flags behind the copies
 * arrive later than the in-kernel stores did); 0 = every halo is mirrored in-kernel and the G-buffer rows are recomputed.
 * Default -1: level 1 for two strips, level 2 from three strips on (the configurations measured at 2 and at 8 GPUs). */
#define ST_STRIP_DMA_DEFAULT (-1)
/* ST_OPT_FUSED_PASSES (default 1): reference passes whose hand-over is private to a pixel or to a checkerboard pair run as ONE launch:
 * K5+K6 (di_sampling + di_temporal_resampling), K7+K8+K9 (di_spatial_resampling pick / trace / sample), K12+K13 (gi_sampling a + b),
 * K11 inside K14 on tracing frames (gi_reprojection + gi_temporal_resampling), K15+K16+K17 (gi_spatial_resampling) and the second
 * gi_preview_resampling pass + K19 gi_resolving.  Reservoirs, samples and every later buffer are bit-identical to the one-launch-per-
 * pass schedule; only the scratch textures between the fused members (and the intermediate gi_reservoirs entries they replaced) are no
 * longer written.  0 = one launch per reference dispatch (every buffer comparable with the oracle). */
#define ST_FUSED_PASSES_DEFAULT 1
/* ST_OPT_STRIP_FUSED (default 1): strip-partitioned frames use the fused transport (producer kernels store boundary rows straight
 * into the neighbours' buffers, neighbour-only sequence flags, halo rows of the G-buffer and of the SVGF chain recomputed instead of
 * shipped, DI / GI chains interleaved so that rows in flight overlap compute, temporal rows pulled on demand); 0 = one push +
 * all-rank barrier kernel per exchange point.  Needs strips of >= 128 rows. */
/* ST_OPT_SHADING_FAST_MATH (default 1): the ReSTIR DI/GI kernels K5-K19 (strolle-shaders/src/di_*.rs, gi_*.rs) run in their
 * fast-shading build: FMA contraction, approximate division / square root and SFU sin/cos/ex2/lg2 for radiance, BRDF, pdf
 * and MIS evaluation - the arithmetic a GPU shader compiler emits for the reference's SPIR-V.  BVH traversal, the ray/box and
 * ray/triangle tests, the alpha test and the RNG are identical in both builds (same hit for the same ray, bit for bit); the
 * frame stays inside the 1e-3 relative per-channel L2 tolerance.  0 = strict IEEE everywhere (bit-identical to the oracle). */
#define ST_SHADING_FAST_DEFAULT 1
/* ST_OPT_VARIANCE_TILED: 1 = K21 frame_denoising::estimate_variance (frame_denoising.rs:81-217) reads its 6x5 window from a
 * shared-memory tile filled by TMA tensor copies (identical results). */
#define ST_VARIANCE_TILED_DEFAULT 1
/* ST_OPT_BVH_REUSE (default 1): a BVH refresh takes over the subtrees of the previous tree whose primitive-centre
 * sequence is unchanged, as the reference does (strolle/src/bvh/builder.rs:245-275, hash = primitive.rs:27-37);
 * 0 = every refresh builds from scratch.  Both give the same tree unless a primitive changed while its centre did
 * not (e.g. only the instance's material): the reference keeps the old primitive in the reused leaf then (quirk C-20). */
/* ST_OPT_WAVELET_TILED: bit i set = à-trous iteration i (stride 2^i, K22 frame_denoising::wavelet,
 * strolle-shaders/src/frame_denoising.rs:220-361) runs the tile-staged kernel (pixel neighbourhood brought into
 * shared memory by TMA tensor copies) instead of the per-tap gather kernel; both produce identical bits.
 * ST_OPT_WAVELET_TILE_CFG: 4 bits per iteration, output-tile shape (0: 32x8, 1: 32x16, 2: 64x4, 3: 64x8 pixels). */
/* Defaults measured on a B200 at 1920x1080 (tools/wavelet_tune.py, profiles/r1i_wavelet_tune.txt): strides 1, 2, 4, 8
 * tile-staged (32x8, 32x8, 32x8, 32x16 output tiles), stride 16 gathers (its jittered 3x3 footprint does not fit a tile). */
#define ST_WAVELET_TILED_DEFAULT 15
#define ST_WAVELET_CFG_DEFAULT 0x01000
/* ST_OPT_FUSE_REPROJECT: 1 = K20 frame_denoising::reproject (frame_denoising.rs:4-78) handles the DI and the GI
 * signal in one launch (the reference dispatches it twice, passes/frame_denoising.rs:143-160); identical results. */
#define ST_FUSE_REPROJECT_DEFAULT 1
/* ST_OPT_HALO_NCCL (default 0): 1 keeps NCCL send/recv for the halo rows even when peer memory is linked. */
/* ST_OPT_ASYNC_OUTPUT (default 0): st_render_camera / st_copy_output only enqueue the device->host copy of
 * the composed frame and return; the caller keeps `host_out` (pinned) untouched until st_synchronize, and
 * alternates between two host buffers to pipeline frame N's copy with frame N+1's passes. */
int st_set_option(st_engine* e, int option, int value);
/* Engine statistics (development / test aid): tile-staged wavelet launches since creation, and how many of its
 * CTAs gave up waiting for their tensor copies (must stay 0). */
enum { ST_STAT_WAVELET_TILED_LAUNCHES = 1, ST_STAT_WAVELET_TILED_ERRORS = 2, ST_STAT_BVH_GRAFTED_SUBTREES = 3, ST_STAT_VARIANCE_TILED_LAUNCHES = 4,
       ST_STAT_STRIP_PULLED_ROWS = 5 /* rows x buffers fetched from other ranks by the temporal pull since linking */, ST_STAT_LAST_FRAME_FUSED_STRIPS = 6 /* 1 = the last strip frame used the fused transport */,
       ST_STAT_STRIP_FIRST_TIMEOUT = 7 /* 0, or 0x80000000 | slot << 16 | awaited rank << 8 | sequence & 0xff of the first strip flag wait that gave up */ };
int st_get_stat(st_engine* e, int stat, uint64_t* value);
/* The host-side BVH builder on its own (no device needed): binned-SAH build (strolle/src/bvh/builder.rs:17-319) + DFS
 * serialisation (serializer.rs:20-110) over `n` primitives of 11 floats each (triangle id bits, material id bits,
 * centre xyz, bounds min xyz, bounds max xyz; centre.x == FLT_MAX marks a dead primitive, primitive.rs:18-24).  The
 * builder object keeps the previous tree; `reuse` != 0 grafts its unchanged subtrees (builder.rs:245-359).  `out`
 * receives the float4 stream the GPU traverses (`*n_floats` floats); with out == NULL only the size is returned and
 * st_bvh_builder_read copies the stream of that build afterwards. */
typedef struct st_bvh_builder st_bvh_builder;
int st_bvh_builder_create(st_bvh_builder** out);
void st_bvh_builder_destroy(st_bvh_builder* b);
int st_bvh_builder_build(st_bvh_builder* b, const float* prims11, size_t n, int reuse, float* out, size_t cap_floats, size_t* n_floats,
                         uint32_t* grafted_subtrees, int* depth);
int st_bvh_builder_read(st_bvh_builder* b, float* out, size_t cap_floats);
/* external != 0: run the engine on the caller-owned CUDA stream `cuda_stream` (NULL = the legacy default
 * stream), e.g. the host runtime's stream that NCCL halo exchanges are ordered against; external == 0:
 * back to a private non-blocking stream. */
int st_set_stream(st_engine* e, void* cuda_stream, int external);
/* Ray statistics: counts executed Ray::trace / Ray::intersect calls (the Mrays/s numerator, SURVEY §8d). */
int st_count_rays(st_engine* e, int enabled);
int st_ray_count(st_engine* e, uint64_t* rays, int reset);
/* Native strip-parallel frame (SURVEY §8e): one engine per GPU/process, NCCL communicator owned by the engine.
 * rank 0 obtains an id (st_nccl_unique_id), the host runtime broadcasts the 128 bytes, every rank calls
 * st_nccl_init; st_render_strips then runs the frame's passes on this rank's row strip with an NCCL halo
 * exchange (grouped ncclSend/ncclRecv on the engine's stream) before each gathering pass, and, when `gather`
 * is non-zero (same value on every rank), assembles the composed frame on rank 0 in `format` (copied to `host_out`
 * there if non-NULL).  st_plan_frame exposes the exchange plan
 * ("step:buffer:reach;..." text) for tests. */
int st_nccl_unique_id(uint8_t* out128);
int st_nccl_init(st_engine* e, const uint8_t* id128, int rank, int world);
int st_plan_frame(const int* schedule, int n, uint32_t frame, int temporal_reach, char* out, size_t cap);
int st_render_strips(st_engine* e, st_camera_handle camera, void* host_out, int format, int temporal_reach, int gather);
/* The fused strip transport's order of one frame for a given pass schedule (st_frame_schedule), as text for tests:
 * "step:i;signal:SLOT:nb|all;wait:SLOT:nb|all[:prev];pull;push:buffer:SLOT;..." (no device needed).  `dma`: bits 0-1 = ST_OPT_STRIP_DMA (0, 1, 2),
 * bit 2 = a frame on which nothing moved (no temporal pull, no wait for PULL_DONE). */
int st_plan_strip_order(const int* schedule, int n, int dma, char* out, size_t cap);
/* The row partition st_render_strips / st_multi_* use for a frame of `height` rows over `world` ranks: rows_out[2r], rows_out[2r+1] = rank r's
 * [y0, y1).  Equal strips for one or two ranks; from three on the outer strips (one neighbour) get a few rows more than the inner ones
 * (two neighbours' worth of recomputed and mirrored halo rows).  No device needed. */
int st_strip_bounds(int height, int world, int* rows_out);
int st_halo_bytes(st_engine* e, uint64_t* bytes);
/* Peer-memory halo transport (default once linked): every rank exports CUDA IPC handles of the camera's buffers
 * (st_peer_export, ST_PEER_HANDLE_BYTES bytes), the host runtime all-gathers them, st_peer_import maps the other
 * ranks' buffers.  From then on st_render_strips replaces each NCCL exchange with ONE kernel that stores this
 * rank's boundary rows straight into the neighbours' buffers over NVLink, raises a sequence flag in every peer and
 * waits for theirs (a device-side barrier; no host involvement).  st_peer_errors counts barrier time-outs. */
#define ST_PEER_HANDLE_BYTES 192
int st_peer_export(st_engine* e, st_camera_handle camera, uint8_t* out192);
int st_peer_import(st_engine* e, st_camera_handle camera, const uint8_t* all_handles, int rank, int world);
int st_peer_errors(st_engine* e, st_camera_handle camera, uint32_t* count);
/* Device-side stopwatch on the engine's stream (CUDA events): st_mark_begin records, st_mark_end
 * records + waits and returns the elapsed milliseconds between the two. */
int st_mark_begin(st_engine* e);
int st_mark_end(st_engine* e, float* ms);
/* Row-strip partition for multi-GPU runs (SURVEY §8e): this engine computes rows [y0, y1) of the
 * camera's frame; full-frame buffers stay addressable for halo rows. */
int st_camera_set_strip(st_engine* e, st_camera_handle camera, int y0, int y1);
/* Device pointer + byte size of a per-camera buffer (for NCCL halo exchange by the host runtime). */
int st_buffer_device_ptr(st_engine* e, st_camera_handle camera, const char* name, void** ptr, size_t* bytes);
/* Stage-wise rendering for strip-parallel runs: executes passes [first, last] of the frame
 * schedule (indices into the schedule returned by st_frame_schedule). */
int st_frame_schedule(st_engine* e, st_camera_handle camera, int* pass_ids, int cap, int* count);
int st_render_range(st_engine* e, st_camera_handle camera, int first, int last);

/* Links engines of THIS process into one strip group (rank = index): enables peer access between their devices and maps every
 * member's per-camera buffers into the others (what st_peer_export / st_peer_import do between processes).  Members may share a
 * device (the whole protocol then runs on one GPU: how single-GPU boxes test it). */
int st_link_local(st_engine* const* engines, const st_camera_handle* cameras, int n);

/* ---- st_multi: one process, several devices (SURVEY 8b: `Engine::new` over a list of device ordinals) --------------------------
 * The strolle::Engine surface for a row-strip group: scene verbs are replayed on every member (the scene is replicated), a camera
 * exists on every member, st_multi_render_camera renders every member's strip of ONE frame with the fused transport and copies
 * each strip into the caller's frame.  Mirrors the st_* verbs one to one (lib.rs:132-301). */
typedef struct st_multi st_multi;
int st_multi_create(const int* device_ordinals, int n, st_multi** out);
void st_multi_destroy(st_multi* m);
int st_multi_size(st_multi* m);
st_engine* st_multi_engine(st_multi* m, int rank);   /* member access (statistics, options, st_read_buffer on one strip) */
st_camera_handle st_multi_member_camera(st_multi* m, st_camera_handle camera, int rank);
int st_multi_insert_mesh(st_multi* m, st_handle mesh, const st_mesh_triangle* triangles, size_t count);
int st_multi_remove_mesh(st_multi* m, st_handle mesh);
int st_multi_insert_material(st_multi* m, st_handle material, const st_material* mat);
int st_multi_has_material(st_multi* m, st_handle material);
int st_multi_remove_material(st_multi* m, st_handle material);
int st_multi_insert_image(st_multi* m, st_handle image, const uint8_t* rgba8, uint32_t width, uint32_t height);
int st_multi_remove_image(st_multi* m, st_handle image);
/* st_insert_dynamic_image for the group: every member refreshes its own atlas from the same surface, which must be reachable from every
 * member's device (or be page-locked host memory); otherwise it is refused with nothing registered on any member. */
int st_multi_insert_dynamic_image(st_multi* m, st_handle image, const void* src, size_t pitch_bytes, uint32_t width, uint32_t height);
int st_multi_set_material_textures(st_multi* m, st_handle material, const st_material_textures* textures);
int st_multi_insert_instance(st_multi* m, st_handle instance, st_handle mesh, st_handle material, const float affine[12]);
int st_multi_remove_instance(st_multi* m, st_handle instance);
int st_multi_insert_light(st_multi* m, st_handle light, const st_light* l);
int st_multi_remove_light(st_multi* m, st_handle light);
int st_multi_update_sun(st_multi* m, float azimuth, float altitude);
int st_multi_create_camera(st_multi* m, const st_camera* camera, st_camera_handle* out);
int st_multi_update_camera(st_multi* m, st_camera_handle camera, const st_camera* desc);
int st_multi_delete_camera(st_multi* m, st_camera_handle camera);
int st_multi_tick(st_multi* m);
/* host_out: the full frame (width*height pixels of `format`); every member fills its own rows.  NULL = enqueue only. */
int st_multi_render_camera(st_multi* m, st_camera_handle camera, void* host_out, int format);
/* st_render_camera_to for the group: every member stores its own rows [y0, y1) at dst + y0 * pitch_bytes, a kernel of its own for a
 * device surface (a peer store when the surface lives on another member's device), a 2-D copy for a host surface.  A device surface
 * on a device some member cannot reach is refused.  st_multi_render_camera is the tightly packed host case. */
int st_multi_render_camera_to(st_multi* m, st_camera_handle camera, void* dst, size_t pitch_bytes, int format);
int st_multi_synchronize(st_multi* m);
int st_multi_set_option(st_multi* m, int option, int value);
int st_multi_set_seed_base(st_multi* m, uint32_t base);
int st_multi_set_blue_noise(st_multi* m, const uint8_t* rgba8_256x256);
int st_multi_read_buffer(st_multi* m, st_camera_handle camera, const char* name, float* dst, size_t cap_floats, size_t* count);
int st_multi_peer_errors(st_multi* m, st_camera_handle camera, uint32_t* count);

/* ---- view-parallel groups: whole cameras placed on one member each (no reference counterpart) -------------------------------------
 * Many independent views (split screen, camera walls, mirrors and monitors, probes) need no exchange between devices: each renders whole
 * on one member.  Members tick in lockstep, so frame ids, seeds and the BVH are equal on every member, and a placed camera's frames are
 * bit for bit what one st_engine with the same scene and seed base renders.  On a placed camera st_multi_update_camera (a resize
 * re-creates its buffers there only), st_multi_delete_camera, st_multi_render_camera(_to) (the whole frame, as st_render_camera(_to)
 * there), st_multi_read_buffer (the whole frame) and st_multi_peer_errors (always 0) act on its member only; st_multi_member_camera
 * gives -1 on every other member, where it has no buffers at all.  In a group of one member a placed camera is a strip camera. */
enum { ST_PLACE_STRIPS = -1, ST_PLACE_AUTO = -2 };
/* A camera that lives on member `rank` only.  ST_PLACE_AUTO picks the member with the fewest pixels (width * height summed) of placed
 * cameras, the lowest rank on a tie; the choice is made here, once.  ST_ERR_INVALID for another rank outside [0, size). */
int st_multi_create_camera_on(st_multi* m, const st_camera* camera, int rank, st_camera_handle* out);
/* The member a camera lives on, or ST_PLACE_STRIPS for a camera made by st_multi_create_camera.  ST_ERR_NOT_FOUND for an unknown or
 * deleted camera. */
int st_multi_camera_rank(st_multi* m, st_camera_handle camera, int* rank);
/* Moves a placed camera, with all of its temporal state, to member `rank`: waits for the source member's queued work, allocates the
 * camera there and copies its buffers device to device (a peer copy between devices), then frees the source.  The handle stays; the
 * next frame is the one it would have rendered where it was.  Moving to its own member does nothing.  ST_ERR_NOT_FOUND for an unknown
 * camera, ST_ERR_INVALID for a strip camera or a rank outside the group; a refused or failed move leaves the camera where it was. */
int st_multi_move_camera(st_multi* m, st_camera_handle camera, int rank);
/* st_render_cameras for the group: every member renders the listed cameras placed on it as batched groups, all members concurrently
 * (every member's passes and device stores are enqueued before any host copy is issued, and nothing in between waits on the host).
 * Camera for camera the result is what st_render_cameras gives for them on one engine.  A surface is resolved from its camera's member:
 * device memory of any device that member reaches (a peer store otherwise), managed or host memory.  Host surfaces block unless
 * ST_OPT_ASYNC_OUTPUT; device surfaces only enqueue (order with st_multi_synchronize).  In a group of one member this is st_render_cameras
 * on it.  Everything is checked before any member renders: ST_ERR_NOT_FOUND for an unknown or deleted camera; ST_ERR_INVALID for n <= 0,
 * a camera listed twice, a strip camera in a group of several members, a surface st_render_camera_to refuses on the camera's member,
 * or a call before the first st_multi_tick. */
int st_multi_render_cameras(st_multi* m, const st_camera_handle* cameras, int n, void* const* dsts, const size_t* pitch_bytes, int format);

#ifdef __cplusplus
}
#endif
#endif /* STROLLE_B200_H */
