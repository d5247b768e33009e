// strolle_b200 — host-callable launchers for the kernels in kernels.cu.
#pragma once
#include <cuda_runtime.h>
#include <vector>
#include "st_types.h"

namespace st {
typedef uint32_t u32;

// One view of a per-pixel launch.  A launch covers one camera, or several cameras of one size, mode and frame (st_render_cameras),
// blockIdx.z selecting the view.  Buffer pointers passed as launch arguments are those of view 0; every camera arena (and svgf_pairs)
// of one size has the same layout, so view v's buffer lies at the same offset from its own base.
struct ViewDev {
    CameraDev cam;
    long long arena_delta, pair_delta;   // bytes from view 0's camera arena / svgf_pairs to this view's (0 for view 0)
    char* dst; size_t pitch;             // launch_output_store: where pixel (0, 0) of this view's frame goes, and the surface's row pitch
};
// Views per launch.  Kernel parameters may take 32764 bytes (sm_70 and later, CUDA 12.1 and later); the scene and the pass's own
// arguments get the rest.
constexpr int kBatchViews = (32764 - 1024) / (int)sizeof(ViewDev);
template <bool BATCHED> struct ViewBatch { ViewDev v[BATCHED ? kBatchViews : 1]; };
static_assert(sizeof(ViewBatch<true>) + 1024 <= 32764, "a batched launch's parameters must fit the 32764-byte limit");
// The views of one launch (1..kBatchViews).  One view runs the single-camera instantiation of each kernel, which reads the camera at
// fixed parameter offsets; several run the batched one.
typedef std::vector<ViewDev> ViewSet;

void launch_prim_gbuffer(const ViewSet& v, const SceneDev& s, int cur, int with_reprojection, cudaStream_t st);
void launch_frame_reprojection(const ViewSet& v, const SceneDev& s, int cur, cudaStream_t st);
void launch_di_sampling(const ViewSet& v, const SceneDev& s, int cur, u32 seed, u32 frame, cudaStream_t st);
void launch_di_temporal(const ViewSet& v, const SceneDev& s, int cur, u32 seed, cudaStream_t st);
void launch_di_spatial_pick(const ViewSet& v, const SceneDev& s, int cur, u32 seed, u32 frame, cudaStream_t st);
void launch_spatial_trace(const ViewSet& v, const SceneDev& s, const float4* d0, const float4* d1, float4* d2, cudaStream_t st);
void launch_di_spatial_sample(const ViewSet& v, const SceneDev& s, u32 seed, u32 frame, cudaStream_t st);
void launch_di_resolving(const ViewSet& v, const SceneDev& s, int cur, cudaStream_t st);
void launch_gi_reprojection(const ViewSet& v, const SceneDev& s, int cur, cudaStream_t st);
void launch_gi_sampling_a(const ViewSet& v, const SceneDev& s, int cur, u32 seed, u32 frame, cudaStream_t st);
void launch_gi_sampling_b(const ViewSet& v, const SceneDev& s, int cur, u32 seed, u32 frame, cudaStream_t st);
void launch_gi_temporal(const ViewSet& v, const SceneDev& s, int cur, u32 seed, u32 frame, int inline_reprojection, cudaStream_t st);
void launch_gi_spatial_pick(const ViewSet& v, const SceneDev& s, int cur, u32 seed, u32 frame, cudaStream_t st);
void launch_gi_spatial_sample(const ViewSet& v, const SceneDev& s, u32 seed, u32 frame, cudaStream_t st);
void launch_gi_preview(const ViewSet& v, const SceneDev& s, int cur, u32 seed, u32 nth, const float4* in, float4* out, int mirror_reach, cudaStream_t st);
void launch_gi_resolving(const ViewSet& v, const SceneDev& s, int cur, const float4* in, cudaStream_t st);
void launch_di_sample_temporal(const ViewSet& v, const SceneDev& s, int cur, u32 seed_sampling, u32 seed_temporal, u32 frame, cudaStream_t st);
void launch_di_spatial_fused(const ViewSet& v, const SceneDev& s, int cur, u32 seed_pick, u32 seed_sample, u32 frame, cudaStream_t st);
void launch_gi_sampling_fused(const ViewSet& v, const SceneDev& s, int cur, u32 seed_a, u32 seed_b, u32 frame, cudaStream_t st);
void launch_gi_spatial_fused(const ViewSet& v, const SceneDev& s, int cur, u32 seed_pick, u32 seed_sample, u32 frame, cudaStream_t st);
void launch_gi_preview_resolve(const ViewSet& v, const SceneDev& s, int cur, u32 seed, const float4* in, const float4* source, cudaStream_t st);
void launch_denoise_reproject(const ViewSet& v, const SceneDev& s, int cur, const float4* pc, const float4* pm, const float4* smp, float4* col, float4* mom, cudaStream_t st);
void launch_denoise_reproject_pair(const ViewSet& v, const SceneDev& s, int cur, cudaStream_t st);
void launch_denoise_variance(const ViewSet& v, const SceneDev& s, int cur, bool fast, cudaStream_t st);
void launch_denoise_wavelet(const ViewSet& v, const SceneDev& s, int cur, u32 frame, u32 stride, float strength, const float4* di_in, float4* di_out, const float4* gi_in, float4* gi_out, const float4* pair_in, float4* pair_out, bool fast, cudaStream_t st);
bool launch_denoise_wavelet_tiled(const CameraDev& c, const SceneDev& s, u32 frame, u32 stride, float strength, const float4* di_in, float4* di_out, const float4* gi_in, float4* gi_out, float4* pair_out, bool fast, int cfg, u32* errors, cudaStream_t st);
bool launch_denoise_variance_tiled(const CameraDev& c, const SceneDev& s, int cur, bool fast, u32* errors, cudaStream_t st);
void launch_composition(const ViewSet& v, const SceneDev& s, int cur, u32 mode, const float4* di_diff, const float4* gi_diff, cudaStream_t st);
// output pixel formats of launch_output_store, numbered like ST_FORMAT_* (include/strolle_b200.h)
enum OutputFormat { OUT_RGBA32F = 0, OUT_RGBA8_SRGB = 1, OUT_RGBA16F = 2 };
// per view: rows [cam.y0, cam.y1) of cam.output stored at dst + y * pitch (pitch and dst aligned to the format's bytes per pixel)
void launch_output_store(const ViewSet& v, const SceneDev& s, int format, cudaStream_t st);
// Dynamic images (st_insert_dynamic_image): at each tick every image's caller-owned surface is copied into its atlas rectangle.  One record per
// image; a block copies `rows_per_block` rows of one image, and finds its record from the running block offsets (`block0`, ascending).
// Each row is `head` 4-byte texels, `body` 16-byte groups of four, then `tail` 4-byte texels; body > 0 only when the source row and the atlas
// row have the same address modulo 16 on every row (the host sets head = texels up to the atlas row's first 16-byte boundary).
struct AtlasCopy {
    const char* src; unsigned long long pitch;   // source texel (0, 0) (a device, peer, managed or mapped host address) and its row pitch
    u32 x, y, w, h;                               // atlas rectangle
    u32 head, body, tail, rows_per_block, block0;
};
constexpr int kAtlasCopies = 128;   // records per launch (5 KB of parameters); more images run as several launches
struct AtlasCopyBatch { AtlasCopy c[kAtlasCopies]; int n; };
// Splits `copies` into launches of kAtlasCopies records; fills head / body / tail / rows_per_block / block0.  Returns the launch count.
int launch_atlas_refresh(std::vector<AtlasCopy>& copies, uchar4* atlas, cudaStream_t st);
void launch_ref_tracing(const ViewSet& v, const SceneDev& s, u32 depth, cudaStream_t st);
void launch_ref_shading(const ViewSet& v, const SceneDev& s, u32 seed, u32 depth, cudaStream_t st);
void launch_bvh_heatmap(const ViewSet& v, const SceneDev& s, cudaStream_t st);
void launch_trace_stream_closest(const SceneDev& s, const float4* rays, long n, float4* out, cudaStream_t st);
void launch_trace_stream_any(const SceneDev& s, const float4* rays, long n, u32* out, cudaStream_t st);
void launch_math(int op, const float* a, const float* b, float* out, long n, cudaStream_t st);
void launch_material_derive(const GpuMaterial* mats, u32 n, u32* packed, cudaStream_t st);
void launch_srgb_lut(float* lut, cudaStream_t st);
void launch_unpack_lut(float* lut, cudaStream_t st);
void launch_atm_transmittance(float4* out, cudaStream_t st);
void launch_atm_scattering(const float4* tl, float4* out, cudaStream_t st);
void launch_atm_sky(const float4* tl, const float4* sl, float sun_altitude, float4* out, cudaStream_t st);

// Halo rows over NVLink peer memory + device-side barrier (multi-GPU strips, SURVEY §8e)
#define ST_PEER_MAX_SEGMENTS 40
#define ST_PEER_MAX_RANKS 16
struct PeerSegment { const uint4* src; uint4* dst; unsigned long long n; };
struct PeerExchange {
    PeerSegment seg[ST_PEER_MAX_SEGMENTS]; int nseg;
    u32* peer_flags[ST_PEER_MAX_RANKS];   // slot [my rank] of every peer's flag array (mapped peer memory); null for self
    const u32* my_flags;                  // my flag array, slot [r] raised by rank r
    u32* counter; u32* errors;            // block completion counter (self-resetting), barrier time-out count
    int n_ranks, rank; u32 seq; int signal;
};
void launch_peer_exchange(const PeerExchange& x, cudaStream_t st);

// Fused strip transport (engine.cu render_strips_fused): sequence flags between ranks and the temporal pull
enum StripSlot { SLOT_FRAME_DONE = 0, SLOT_PULL_DONE = 1, SLOT_DI1 = 2, SLOT_GI1 = 3, SLOT_GI2 = 4, SLOT_GI3 = 5, SLOT_SVGF = 6, SLOT_GBUF = 7, SLOT_COUNT = 8 };
struct StripSync {
    const u32* my_flags;                  // this rank's flag words, [slot * ST_PEER_MAX_RANKS + source rank]
    u32* peer_flags[ST_PEER_MAX_RANKS];   // every other rank's flag array (mapped peer memory); null for self
    u32* errors;                          // wait time-outs
    int n_ranks, rank;
};
struct StripPullItem { size_t offset; int vec4_per_px; int local_rows; };   // arena byte offset of the buffer, float4 per pixel, rows beyond the strip this rank holds itself
struct StripPull {
    char* arena[ST_PEER_MAX_RANKS]; int bounds[ST_PEER_MAX_RANKS + 1];
    int n_ranks, rank, w, h, own_y0, own_y1;
    const int* need_rows; unsigned long long* pulled_rows;
    StripPullItem items[12]; int nitems;
};
int preload_kernels();   // 0 = every kernel of the strict build is loaded; > 0 = the driver cannot enumerate them (kernels then load at first launch)
void launch_strip_signal(const StripSync& s, int slot, u32 seq, u32 dst_mask, int* reset_need, int h, cudaStream_t st);
void launch_strip_wait(const StripSync& s, int slot, u32 seq, u32 src_mask, cudaStream_t st);
void launch_strip_signal_wait(const StripSync& s, int sig_slot, u32 seq, u32 dst_mask, int wait_slot, u32 wait_seq, u32 src_mask, cudaStream_t st);
void launch_strip_pull(const StripPull& p, cudaStream_t st);
void launch_atm_sun_color(float4* out2, const GpuWorld& world, cudaStream_t st);

}  // namespace st

// The ReSTIR kernels K5-K19 built a second time with FMA contraction and SFU approximations (kernels.cu compiled with
// -DST_FAST=1, see st_math.cuh): same launch interface, selected by ST_OPT_SHADING_FAST_MATH.
namespace stf {
using st::CameraDev; using st::SceneDev; using st::ViewSet; using st::u32;
int preload_kernels();   // the fast-shading build's kernels
void launch_di_sampling(const ViewSet& v, const SceneDev& s, int cur, u32 seed, u32 frame, cudaStream_t st);
void launch_di_temporal(const ViewSet& v, const SceneDev& s, int cur, u32 seed, cudaStream_t st);
void launch_di_spatial_pick(const ViewSet& v, const SceneDev& s, int cur, u32 seed, u32 frame, cudaStream_t st);
void launch_spatial_trace(const ViewSet& v, const SceneDev& s, const float4* d0, const float4* d1, float4* d2, cudaStream_t st);
void launch_di_spatial_sample(const ViewSet& v, const SceneDev& s, u32 seed, u32 frame, cudaStream_t st);
void launch_di_resolving(const ViewSet& v, const SceneDev& s, int cur, cudaStream_t st);
void launch_gi_reprojection(const ViewSet& v, const SceneDev& s, int cur, cudaStream_t st);
void launch_gi_sampling_a(const ViewSet& v, const SceneDev& s, int cur, u32 seed, u32 frame, cudaStream_t st);
void launch_gi_sampling_b(const ViewSet& v, const SceneDev& s, int cur, u32 seed, u32 frame, cudaStream_t st);
void launch_gi_temporal(const ViewSet& v, const SceneDev& s, int cur, u32 seed, u32 frame, int inline_reprojection, cudaStream_t st);
void launch_gi_spatial_pick(const ViewSet& v, const SceneDev& s, int cur, u32 seed, u32 frame, cudaStream_t st);
void launch_gi_spatial_sample(const ViewSet& v, const SceneDev& s, u32 seed, u32 frame, cudaStream_t st);
void launch_gi_preview(const ViewSet& v, const SceneDev& s, int cur, u32 seed, u32 nth, const float4* in, float4* out, int mirror_reach, cudaStream_t st);
void launch_gi_resolving(const ViewSet& v, const SceneDev& s, int cur, const float4* in, cudaStream_t st);
void launch_di_sample_temporal(const ViewSet& v, const SceneDev& s, int cur, u32 seed_sampling, u32 seed_temporal, u32 frame, cudaStream_t st);
void launch_di_spatial_fused(const ViewSet& v, const SceneDev& s, int cur, u32 seed_pick, u32 seed_sample, u32 frame, cudaStream_t st);
void launch_gi_sampling_fused(const ViewSet& v, const SceneDev& s, int cur, u32 seed_a, u32 seed_b, u32 frame, cudaStream_t st);
void launch_gi_spatial_fused(const ViewSet& v, const SceneDev& s, int cur, u32 seed_pick, u32 seed_sample, u32 frame, cudaStream_t st);
void launch_gi_preview_resolve(const ViewSet& v, const SceneDev& s, int cur, u32 seed, const float4* in, const float4* source, cudaStream_t st);
}  // namespace stf
