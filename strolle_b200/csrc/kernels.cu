// strolle_b200 — sm_100a kernels for the per-pixel GI hot path.
//
// One kernel per reference compute entry point (strolle-shaders/src/*.rs, K1–K22 in
// SURVEY.md §2.2) plus the primary-visibility G-buffer kernel that replaces the rasteriser
// and the composition kernel.  All kernels are HBM/latency-bound integer+f32 work: no tensor
// cores.  Mapping: one thread per pixel, CTAs of 128 threads covering a 16x8 pixel tile so
// that a warp reads two 256-byte row segments of every float4 texture (coalesced 16-byte
// loads); BVH nodes / triangles go through the read-only path (ld.global.nc.v4.f32) and the
// traversal stack lives in shared memory, one conflict-free column per thread.
#include <algorithm>
#include <cstdio>
#include <cuda_fp16.h>
#include <cuda.h>   // CUtensorMap (type only; the encoder is reached through cudaGetDriverEntryPoint)
#include <map>
#include <mutex>
#include <tuple>
#include <vector>
#include "st_device.cuh"
#include "kernels.h"

// Compiled twice (strolle_b200/build.py): as namespace st with strict IEEE arithmetic (every kernel), and with -DST_FAST=1 as
// namespace stf, the fast-shading flavour of the ReSTIR kernels K5-K19 only (see st_math.cuh).
#if defined(ST_FAST) && ST_FAST
#define ST_EXACT_ONLY 0
#else
#define ST_EXACT_ONLY 1
#endif

namespace ST_NS {

#define TILE_W 16
#define TILE_H 8

struct Px { u32 x, y; bool in; };
// Row tile of this CTA.  In a strip that mirrors rows into the strip below it, the CTAs are rotated so that the bottom boundary rows are
// computed FIRST (the top boundary rows follow, the interior last): the remote stores of both boundaries drain over NVLink while the
// interior is still computing, instead of at the very end of the kernel.
ST_DEV u32 row_tile(const CameraDev& cam) {
    if (cam.mirror_dn == 0) return blockIdx.y;
    const u32 lead = (u32)(ST_REACH_SPATIAL / TILE_H);
    return gridDim.y > lead ? (blockIdx.y + gridDim.y - lead) % gridDim.y : blockIdx.y;
}
ST_DEV Px pixel_full(const CameraDev& cam) {
    Px p; p.x = blockIdx.x * TILE_W + (threadIdx.x % TILE_W); p.y = (u32)cam.y0 + row_tile(cam) * TILE_H + (threadIdx.x / TILE_W);
    p.in = p.x < (u32)cam.w && p.y < (u32)cam.y1;
    return p;
}
// half-width checkerboard dispatch of the reference: gid.x < 8*(((W+7)/8)/2), gid.y < 8*((H+7)/8)
ST_DEV int half_grid_w(int w) { return 8 * (((w + 7) / 8) / 2); }
ST_DEV Px pixel_half(const CameraDev& cam) {
    Px p; p.x = blockIdx.x * TILE_W + (threadIdx.x % TILE_W); p.y = (u32)cam.y0 + row_tile(cam) * TILE_H + (threadIdx.x / TILE_W);
    p.in = p.x < (u32)half_grid_w(cam.w) && p.y < (u32)cam.y1;
    return p;
}
ST_DEV size_t pix(const CameraDev& cam, u32 x, u32 y) { return (size_t)y * (size_t)cam.w + x; }
ST_DEV size_t screen_idx(const CameraDev& cam, u32 x, u32 y) { return (size_t)(y * to_u32_sat(cam.curr.screen.x) + x); }   // camera.rs:39-41 (u32 arithmetic)
ST_DEV bool in_tex(const CameraDev& cam, u32 x, u32 y) { return x < (u32)cam.w && y < (u32)cam.h; }
ST_DEV float4 tex_or_zero(const float4* __restrict__ t, const CameraDev& cam, u32 x, u32 y) { return in_tex(cam, x, y) ? t[pix(cam, x, y)] : f4zero(); }
ST_DEV void tex_store(float4* __restrict__ t, const CameraDev& cam, u32 x, u32 y, float4 v) { if (in_tex(cam, x, y)) t[pix(cam, x, y)] = v; }
ST_DEV Hit load_hit(const GpuCamera& c, const float4* __restrict__ d0, const float4* __restrict__ d1, const CameraDev& cam, u32 x, u32 y) {
    return hit_make(cam_ray(c, x, y), gbuf_unpack(tex_or_zero(d0, cam, x, y), tex_or_zero(d1, cam, x, y)));
}
// variant whose base colour comes from the byte table (kernels that consume hit.g.base_color)
ST_DEV Hit load_hit_lut(const SceneDev& sc, const GpuCamera& c, const float4* __restrict__ d0, const float4* __restrict__ d1, const CameraDev& cam, u32 x, u32 y) {
    return hit_make(cam_ray(c, x, y), gbuf_unpack(sc, tex_or_zero(d0, cam, x, y), tex_or_zero(d1, cam, x, y)));
}
#define ST_TRACE_STACK()                                          \
    __shared__ u32 s_stack[ST_BVH_STACK * ST_BLOCK];              \
    TraceStack stk; stk.base = s_stack + threadIdx.x;

#define KPARAMS const __grid_constant__ CameraDev cam, const __grid_constant__ SceneDev sc
// The per-pixel kernels are instantiated twice: BATCHED = false reads its one camera at fixed parameter offsets (every single-camera
// frame runs this), BATCHED = true takes the view from blockIdx.z (st_render_cameras).  The choice follows the launch's view count.
#define VPARAMS const __grid_constant__ ViewBatch<BATCHED> views, const __grid_constant__ SceneDev sc
#define VIEW const ViewDev& view = views.v[BATCHED ? blockIdx.z : 0]; const CameraDev& cam = view.cam
#define VIEW_ARENA(p) p = arena_ptr<BATCHED>(p, view)
// a buffer pointer passed as a launch argument (view 0's) moved to the same buffer of this thread's view
template <bool BATCHED, class T> ST_DEV T* arena_ptr(T* p, const ViewDev& v) { return (BATCHED && p) ? (T*)((char*)p + v.arena_delta) : p; }
template <bool BATCHED, class T> ST_DEV T* pair_ptr(T* p, const ViewDev& v) { return (BATCHED && p) ? (T*)((char*)p + v.pair_delta) : p; }

// Launch bounds per kernel: ST_LB_<KERNEL> is __launch_bounds__(128) (ptxas' own register choice) unless a minimum number
// of resident CTAs per SM is set (ST_MINB_<KERNEL> = N caps registers at 65536 / (128 N)); values tuned on a B200 with
// tools/occupancy_tune.py.  -DST_MINB_ALL=N overrides every kernel at once (tuning builds).
#define ST_LB_N(N) __launch_bounds__(ST_BLOCK, N)
// measured (profiles/r1j_occupancy_tune.txt): capping these five at 64 registers (8 CTAs/SM) is worth 80 us per 1080p frame
#if !defined(ST_MINB_ALL)
#define ST_MINB_GI_PREVIEW 8
#define ST_MINB_GI_TEMPORAL 8
#define ST_MINB_GI_SAMPLING_B 8
#define ST_MINB_GI_SPATIAL_PICK 8
#define ST_MINB_DI_TEMPORAL 12
#endif
// ST_LB_<K>: -DST_MINB_ALL=N beats a per-kernel ST_MINB_<K>, which beats ptxas' own choice.  The preprocessor cannot test a macro whose
// name is pasted together, so the three-way choice is spelled once per kernel through ST_LB_PICK (0 = "no minimum").
#define ST_LB_PICK(per_kernel) ST_LB_CHOOSE(ST_MINB_ALL_OR_0, per_kernel)
#if defined(ST_MINB_ALL)
#define ST_MINB_ALL_OR_0 ST_MINB_ALL
#else
#define ST_MINB_ALL_OR_0 0
#endif
// The caps hold for the single-camera instantiations.  A batched instantiation (BATCHED, see VPARAMS) reads the camera through register-
// indexed constant loads, which need registers of their own; under the same cap it would spill, so ptxas chooses its registers.
template <int ALL, int ONE> struct LbMin { static constexpr int value = ALL > 0 ? ALL : ONE; };
#define ST_LB_CHOOSE(all, one) __launch_bounds__(ST_BLOCK, (!BATCHED && LbMin<all, one>::value > 0 ? LbMin<all, one>::value : 1))
#ifndef ST_MINB_PRIM_GBUFFER
#define ST_MINB_PRIM_GBUFFER 0
#endif
#define ST_LB_PRIM_GBUFFER ST_LB_PICK(ST_MINB_PRIM_GBUFFER)
#ifndef ST_MINB_DI_SAMPLING
#define ST_MINB_DI_SAMPLING 0
#endif
#define ST_LB_DI_SAMPLING ST_LB_PICK(ST_MINB_DI_SAMPLING)
#ifndef ST_MINB_DI_TEMPORAL
#define ST_MINB_DI_TEMPORAL 0
#endif
#define ST_LB_DI_TEMPORAL ST_LB_PICK(ST_MINB_DI_TEMPORAL)
#ifndef ST_MINB_DI_SPATIAL_PICK
#define ST_MINB_DI_SPATIAL_PICK 0
#endif
#define ST_LB_DI_SPATIAL_PICK ST_LB_PICK(ST_MINB_DI_SPATIAL_PICK)
#ifndef ST_MINB_SPATIAL_TRACE
#define ST_MINB_SPATIAL_TRACE 0
#endif
#define ST_LB_SPATIAL_TRACE ST_LB_PICK(ST_MINB_SPATIAL_TRACE)
#ifndef ST_MINB_DI_RESOLVING
#define ST_MINB_DI_RESOLVING 0
#endif
#define ST_LB_DI_RESOLVING ST_LB_PICK(ST_MINB_DI_RESOLVING)
#ifndef ST_MINB_GI_SAMPLING_A
#define ST_MINB_GI_SAMPLING_A 0
#endif
#define ST_LB_GI_SAMPLING_A ST_LB_PICK(ST_MINB_GI_SAMPLING_A)
#ifndef ST_MINB_GI_SAMPLING_B
#define ST_MINB_GI_SAMPLING_B 0
#endif
#define ST_LB_GI_SAMPLING_B ST_LB_PICK(ST_MINB_GI_SAMPLING_B)
#ifndef ST_MINB_GI_TEMPORAL
#define ST_MINB_GI_TEMPORAL 0
#endif
#define ST_LB_GI_TEMPORAL ST_LB_PICK(ST_MINB_GI_TEMPORAL)
#ifndef ST_MINB_GI_SPATIAL_PICK
#define ST_MINB_GI_SPATIAL_PICK 0
#endif
#define ST_LB_GI_SPATIAL_PICK ST_LB_PICK(ST_MINB_GI_SPATIAL_PICK)
#ifndef ST_MINB_GI_SPATIAL_SAMPLE
#define ST_MINB_GI_SPATIAL_SAMPLE 0
#endif
#define ST_LB_GI_SPATIAL_SAMPLE ST_LB_PICK(ST_MINB_GI_SPATIAL_SAMPLE)
#ifndef ST_MINB_GI_PREVIEW
#define ST_MINB_GI_PREVIEW 0
#endif
#define ST_LB_GI_PREVIEW ST_LB_PICK(ST_MINB_GI_PREVIEW)
#ifndef ST_MINB_GI_RESOLVING
#define ST_MINB_GI_RESOLVING 0
#endif
#define ST_LB_GI_RESOLVING ST_LB_PICK(ST_MINB_GI_RESOLVING)

#if ST_EXACT_ONLY
// ---------------------------------------------------------------------------------------------
// Primary-visibility G-buffer (stands in for strolle-shaders/src/prim_raster.rs:41-128; SURVEY §8f-1)
// ---------------------------------------------------------------------------------------------
ST_DEV float4 frame_reprojection_px(const CameraDev& cam, int cur, Px p, float4 surface_texel, float4 vel);
// `with_reprojection` (ST_OPT_FUSED_PASSES; single GPU, or a strip on a frame where nothing moved): K4 runs in this launch too — its inputs for the pixel are still in registers
template <bool BATCHED>
__global__ void ST_LB_PRIM_GBUFFER k_prim_gbuffer(VPARAMS, int cur, int with_reprojection) {
    VIEW;
    ST_TRACE_STACK();
    Px p = pixel_full(cam);
    if (!p.in) return;
    Ray ray = cam_ray(cam.curr, p.x, p.y);
    TriHit th = trace_closest(ray, sc, stk);
    if ((int)p.y < cam.own_y0 || (int)p.y >= cam.own_y1) uncount_ray(sc);   // a neighbour's row, recomputed here: not counted as a ray of the frame
    float4 g0 = f4zero(), g1 = f4zero(), surf = f4zero(), vel = f4zero(), tid = f4(bitsf(0xffffffffu), 0.f, 0.f, 0.f), nd = f4zero();
    if (trihit_some(th)) {
        const GpuMaterial m = sc.materials[th.material_id];
        GBuf g;
        float2 mr = mat_metallic_roughness(sc, m, th.uv);
        g.base_color = mat_base_color(sc, m, th.uv); g.normal = th.normal; g.metallic = mr.x; g.emissive = mat_emissive(sc, m, th.uv);
        g.roughness = mr.y; g.reflectance = m.reflectance; g.depth = dist(ray.o, th.point);
        // untextured base colour: its gamma-encoded bytes come from the per-material table
        gbuf_pack_pre(g, all_zero(m.base_color_texture) ? __ldg(sc.material_packed + th.material_id) : gbuf_pack_color(g.base_color), &g0, &g1);
        float2 n = oct_encode(th.normal);
        surf = f4(n.x, n.y, g.depth, m.roughness);
        nd = f4(oct_decode(n), g.depth);   // what every consumer of the surface map decodes, computed once
        // prim_raster::vs (prim_raster.rs:25-34): where this surface point was last frame, per instance
        const float4* xf = sc.instance_xforms + 6u * (size_t)__ldg(sc.tri_instance + th.triangle_id);
        float4 c0 = ldg4(xf), c1 = ldg4(xf + 1), c2 = ldg4(xf + 2), q0 = ldg4(xf + 3), q1 = ldg4(xf + 4), q2 = ldg4(xf + 5);
        float3 local = ((xyz(c0) * th.point.x + xyz(c1) * th.point.y) + xyz(c2) * th.point.z) + f3(c0.w, c1.w, c2.w);
        float3 prev_point = ((xyz(q0) * local.x + xyz(q1) * local.y) + xyz(q2) * local.z) + f3(q0.w, q1.w, q2.w);
        float2 v = cam_world_to_screen(cam.curr, th.point) - cam_world_to_screen(cam.prev, prev_point);
        if (len2(v) >= 0.001f) vel = f4(v.x, v.y, 0.f, 0.f);
        tid.x = bitsf(th.triangle_id);
        // strip partition: which rows of LAST frame's buffers the temporal passes (K4, K6, K11, K14, K20) of this strip will read:
        // they fetch at prev = pixel - velocity (rounded, or its floor/ceil corners).  Only pixels whose reprojection leaves the
        // owned rows report; the pull kernel that follows brings exactly those rows in from their owners.
        if (cam.need_rows != nullptr && vel.y != 0.0f && (int)p.y >= cam.own_y0 && (int)p.y < cam.own_y1) {
            float py = (float)p.y - vel.y;
            int lo = max(0, min(cam.h - 1, to_i32_sat(floorf(py)))), hi = max(0, min(cam.h - 1, to_i32_sat(ceilf(py))));
            if (lo < cam.own_y0) atomicMin(cam.need_rows, lo);
            if (hi >= cam.own_y1) atomicMax(cam.need_rows + 1, hi);
        }
    }
    size_t i = pix(cam, p.x, p.y);
    cam.prim_gbuffer_d0[cur][i] = g0; cam.prim_gbuffer_d1[cur][i] = g1; cam.prim_surface_map[cur][i] = surf;
    cam.velocity_map[i] = vel; cam.prim_triangle_ids[i] = tid; cam.surface_nd[i] = nd;
    if (with_reprojection && (int)p.y >= cam.own_y0 && (int)p.y < cam.own_y1) cam.reprojection_map[i] = frame_reprojection_px(cam, cur, p, surf, vel);   // not for the rows a strip recomputes beyond its own
}

// K4 frame_reprojection::main (frame_reprojection.rs:7-95): where the pixel was last frame and how far that can be trusted
ST_DEV float4 frame_reprojection_px(const CameraDev& cam, int cur, Px p, float4 surface_texel, float4 vel) {
    const float4* sp_ = cam.prim_surface_map[cur ^ 1];
    Reproj rp; rp.px = 0.f; rp.py = 0.f; rp.confidence = 0.f; rp.validity = 0u;
    Surf surface = surf_decode(surface_texel);
    if (surface.depth == 0.0f) return reproj_encode(rp);
    float2 prev = f2((float)p.x, (float)p.y) - f2(vel.x, vel.y);
    float2 pr = f2(roundf(prev.x), roundf(prev.y));
    if (cam_contains_f(cam.prev, pr)) {
        Surf ps = surf_decode(tex_or_zero(sp_, cam, to_u32_sat(pr.x), to_u32_sat(pr.y)));
        float conf = surf_similarity(ps, surface);
        if (conf > 0.0f) { rp.px = prev.x; rp.py = prev.y; rp.confidence = conf; rp.validity = 0u; }
    }
    if (reproj_some(rp)) {
        int x0 = to_i32_sat(floorf(rp.px)), x1 = to_i32_sat(ceilf(rp.px)), y0 = to_i32_sat(floorf(rp.py)), y1 = to_i32_sat(ceilf(rp.py));
        int xs[4] = {x0, x1, x0, x1}, ys[4] = {y0, y0, y1, y1};
#pragma unroll
        for (int k = 0; k < 4; k++) {
            if (!cam_contains_i(cam.curr, xs[k], ys[k])) continue;
            if (surf_similarity(surf_decode(sp_[pix(cam, (u32)xs[k], (u32)ys[k])]), surface) >= 0.25f) rp.validity |= (1u << k);
        }
    }
    return reproj_encode(rp);
}
template <bool BATCHED>
__global__ void __launch_bounds__(ST_BLOCK) k_frame_reprojection(VPARAMS, int cur) {
    VIEW;
    Px p = pixel_full(cam);
    if (!p.in) return;
    size_t i = pix(cam, p.x, p.y);
    cam.reprojection_map[i] = frame_reprojection_px(cam, cur, p, cam.prim_surface_map[cur][i], cam.velocity_map[i]);
}
#endif   // ST_EXACT_ONLY

// K5 di_sampling::main (di_sampling.rs:4-94): the initial sample of a pixel whose primary hit is `hit`
ST_DEV DiRes di_sampling_px(const CameraDev& cam, const SceneDev& sc, const TraceStack& stk, const Hit& hit, u32 seed, u32 frame, Px p) {
    Rng rng = rng_make(seed, p.x, p.y);
    EphRes res = ephemeral_build(rng, sc, hit);
    DiRes out = di_zero();
    if (res.m > 0.0f) {
        float4 bn = blue_noise(sc, p.x, p.y, frame);
        Ray ray = light_ray_bnoise(light_load(sc, res.light_id), f2(bn.x, bn.y), hit.point);
        bool occ = trace_any(ray, sc, stk);
        if (occ) res.w = 0.0f;
        out.pdf = 0.f; out.confidence = 0.f; out.light_id = res.light_id; out.light_point = ray.o; out.occluded = occ; out.m = 1.0f; out.w = res.w;
    }
    return out;
}
template <bool BATCHED>
__global__ void ST_LB_DI_SAMPLING k_di_sampling(VPARAMS, int cur, u32 seed, u32 frame) {
    VIEW;
    ST_TRACE_STACK();
    Px p = pixel_full(cam);
    if (!p.in) return;
    Hit hit = load_hit_lut(sc, cam.curr, cam.prim_gbuffer_d0[cur], cam.prim_gbuffer_d1[cur], cam, p.x, p.y);
    if (!hit_some(hit)) return;
    di_store(di_sampling_px(cam, sc, stk, hit, seed, frame, p), cam.di_reservoirs[1], screen_idx(cam, p.x, p.y));
}

// K6 di_temporal_resampling::main (di_temporal_resampling.rs:4-112): merges this frame's sample `lhs` with last frame's reservoir at
// the reprojected position
ST_DEV DiRes di_temporal_px(const CameraDev& cam, const SceneDev& sc, int cur, u32 seed, Px p, const Hit& lhs_hit, DiRes lhs) {
    size_t npx = (size_t)cam.w * cam.h;
    Rng rng = rng_make(seed, p.x, p.y);
    if (lhs.m != 0.0f) lhs.pdf = di_pdf_with(lhs, light_load(sc, lhs.light_id), lhs_hit);
    DiRes rhs = di_zero();
    Hit rhs_hit = hit_zero();
    bool killed = false;
    Reproj rp = reproj_decode(cam.reprojection_map[pix(cam, p.x, p.y)]);
    if (reproj_some(rp)) {
        uint2 rpos = reproj_round(rp);
        size_t ridx = screen_idx(cam, rpos.x, rpos.y);
        if (ridx < npx) rhs = di_load(cam.di_reservoirs[0], ridx);
        rhs.m = rmin(rhs.m, 64.0f);
        if (rhs.m != 0.0f) {
            GpuLight rl = light_load(sc, rhs.light_id);
            u32 slot = fbits(rl.d3.x);
            if (slot == 0xcafebabeu) { rhs.w = 0.0f; killed = true; }
            else if (slot > 0u) rhs.light_id = slot - 1u;
            rhs_hit = load_hit_lut(sc, cam.prev, cam.prim_gbuffer_d0[cur ^ 1], cam.prim_gbuffer_d1[cur ^ 1], cam, rpos.x, rpos.y);
        }
    }
    MisIn mi;
    mi.lhs_m = lhs.m; mi.rhs_m = rhs.m; mi.rhs_jacobian = 1.0f; mi.lhs_lhs_pdf = lhs.pdf; mi.rhs_rhs_pdf = rhs.pdf;
    mi.lhs_rhs_pdf = ((lhs.m > 0.0f) & hit_some(rhs_hit)) ? di_pdf_with(lhs, light_prev(light_load(sc, lhs.light_id)), rhs_hit) : 0.0f;
    mi.rhs_lhs_pdf = ((rhs.m > 0.0f) & !killed) ? di_pdf_with(rhs, light_load(sc, rhs.light_id), lhs_hit) : 0.0f;
    MisOut mo = mis_eval(mi);
    DiRes main_ = di_zero();
    float main_pdf = 0.0f;
    if (di_update(main_, rng, lhs, mo.lhs_mis * mo.lhs_pdf * lhs.w)) main_pdf = mo.lhs_pdf;
    if (di_update(main_, rng, rhs, mo.rhs_mis * mo.rhs_pdf * rhs.w)) main_pdf = mo.rhs_pdf;
    main_.m = lhs.m + mo.m;
    main_.pdf = main_pdf;
    main_.confidence = killed ? 0.0f : 1.0f;
    main_.w = res_norm(main_.w, main_pdf, 1.0f, 1.0f);
    return main_;
}
template <bool BATCHED>
__global__ void ST_LB_DI_TEMPORAL k_di_temporal(VPARAMS, int cur, u32 seed) {
    VIEW;
    Px p = pixel_full(cam);
    if (!p.in) return;
    size_t lhs_idx = screen_idx(cam, p.x, p.y);
    Hit lhs_hit = load_hit_lut(sc, cam.curr, cam.prim_gbuffer_d0[cur], cam.prim_gbuffer_d1[cur], cam, p.x, p.y);
    if (!hit_some(lhs_hit)) return;
    di_store_m(cam, di_temporal_px(cam, sc, cur, seed, p, lhs_hit, di_load(cam.di_reservoirs[1], lhs_idx)), cam.di_reservoirs[1], lhs_idx, p.y, cam.di_mirror_reach);
}
// K5 + K6 in one launch (ST_OPT_FUSED_PASSES): the pixel's fresh sample goes from K5 to K6 in registers instead of through di_reservoirs[1]
// (the hit is decoded once).  What di_store / di_load would do to the sample on the way (confidence -> byte) is the identity for K5's
// output (confidence 0), so the result is the two-launch result bit for bit.
template <bool BATCHED>
__global__ void ST_LB_DI_SAMPLING k_di_sample_temporal(VPARAMS, int cur, u32 seed_sampling, u32 seed_temporal, u32 frame) {
    VIEW;
    ST_TRACE_STACK();
    Px p = pixel_full(cam);
    if (!p.in) return;
    Hit hit = load_hit_lut(sc, cam.curr, cam.prim_gbuffer_d0[cur], cam.prim_gbuffer_d1[cur], cam, p.x, p.y);
    if (!hit_some(hit)) return;
    DiRes fresh = di_sampling_px(cam, sc, stk, hit, seed_sampling, frame, p);
    di_store_m(cam, di_temporal_px(cam, sc, cur, seed_temporal, p, hit, fresh), cam.di_reservoirs[1], screen_idx(cam, p.x, p.y), p.y, cam.di_mirror_reach);
}

// The four scratch texels of one checkerboard pair: (d0, d1) of texel a = (2gx, gy) and texel b = (2gx + 1, gy).
// state 0: the pair has no left-hand pixel on the screen, nothing is written; 1: only the two d1 texels are cleared; 2: all four.
struct PairTexels { float4 a0, a1, b0, b1; int state; };

// K7 di_spatial_resampling::pick (di_spatial_resampling.rs:4-147); scratch buf_d0 = di_diff_samples,
// buf_d1 = di_diff_curr_colors (passes/di_spatial_resampling.rs:24-28).  Sky pixels clear buf_d1
// (the reference leaves stale texels there and later reads out of bounds — SURVEY Appendix C-15).
ST_DEV PairTexels di_spatial_pick_pair(const CameraDev& cam, const SceneDev& sc, int cur, u32 seed, u32 frame, Px g) {
    PairTexels o; o.a0 = o.a1 = o.b0 = o.b1 = f4zero(); o.state = 0;
    uint2 lp = checker(g.x, g.y, frame / 2u + 1u);
    if (!cam_contains_u(cam.curr, lp.x, lp.y)) return o;
    o.state = 1;
    size_t lhs_idx = screen_idx(cam, lp.x, lp.y);
    Rng rng = rng_make(seed, lp.x, lp.y);
    const float4* gd0 = cam.prim_gbuffer_d0[cur]; const float4* gd1 = cam.prim_gbuffer_d1[cur];
    Hit lhs_hit = load_hit_lut(sc, cam.curr, gd0, gd1, cam, lp.x, lp.y);
    if (!hit_some(lhs_hit)) return o;
    DiRes lhs = di_load(cam.di_reservoirs[1], lhs_idx);
    DiRes rhs = di_zero();
    size_t rhs_idx = 0;
    Hit rhs_hit = hit_zero();
    float max_radius = 128.0f;
    for (u32 nth = 0u; nth < 8u; nth++) {
        float2 off = rng_disk(rng) * max_radius;
        float2 fp = f2((float)lp.x, (float)lp.y) + off;
        uint2 rpos = cam_contain(cam.curr, to_i32_sat(fp.x), to_i32_sat(fp.y));
        if (rpos.x == lp.x && rpos.y == lp.y) continue;
        // the rejection tests only need the neighbour's depth and normal: one (normal, depth) float4
        float4 nd = tex_or_zero(cam.surface_nd, cam, rpos.x, rpos.y);
        if (nd.w == 0.0f) { max_radius = rmax(max_radius * 0.5f, 5.0f); continue; }
        if (fabs_(nd.w - lhs_hit.g.depth) > 0.33f * lhs_hit.g.depth) { max_radius = rmax(max_radius * 0.5f, 5.0f); continue; }
        if (dot(xyz(nd), lhs_hit.g.normal) < 0.33f) { max_radius = rmax(max_radius * 0.5f, 5.0f); continue; }
        rhs_idx = screen_idx(cam, rpos.x, rpos.y);
        rhs = di_load(cam.di_reservoirs[1], rhs_idx);
        if (rhs.m != 0.0f) { rhs_hit = load_hit_lut(sc, cam.curr, gd0, gd1, cam, rpos.x, rpos.y); break; }
    }
    if (rhs.m == 0.0f) return o;
    float lhs_rhs_pdf = di_pdf_with(lhs, light_load(sc, lhs.light_id), rhs_hit);
    float rhs_lhs_pdf = di_pdf_with(rhs, light_load(sc, rhs.light_id), lhs_hit);
    Ray ra = (lhs_rhs_pdf > 0.0f) ? di_ray(lhs, rhs_hit.point) : ray_zero();
    Ray rb = (rhs_lhs_pdf > 0.0f) ? di_ray(rhs, lhs_hit.point) : ray_zero();
    float2 na = oct_encode(ra.d), nb = oct_encode(rb.d);
    o.a0 = f4(ra.o, ra.len); o.a1 = f4(na.x, na.y, bitsf((u32)rhs_idx + 1u), 0.0f);
    o.b0 = f4(rb.o, rb.len); o.b1 = f4(nb.x, nb.y, lhs_rhs_pdf, rhs_lhs_pdf);
    o.state = 2;
    return o;
}
ST_DEV void store_pair_texels(const CameraDev& cam, const PairTexels& o, float4* buf_d0, float4* buf_d1, Px g) {
    if (o.state == 0) return;
    u32 ax = g.x * 2u, bx = g.x * 2u + 1u;
    if (o.state == 2) { tex_store(buf_d0, cam, ax, g.y, o.a0); tex_store(buf_d0, cam, bx, g.y, o.b0); }
    tex_store(buf_d1, cam, ax, g.y, o.a1); tex_store(buf_d1, cam, bx, g.y, o.b1);
}
template <bool BATCHED>
__global__ void ST_LB_DI_SPATIAL_PICK k_di_spatial_pick(VPARAMS, int cur, u32 seed, u32 frame) {
    VIEW;
    Px g = pixel_half(cam);
    if (!g.in) return;
    store_pair_texels(cam, di_spatial_pick_pair(cam, sc, cur, seed, frame, g), cam.di_diff_samples, cam.di_diff_curr_colors, g);
}

// K8 / K16 *_spatial_resampling::trace (di_spatial_resampling.rs:150-209, gi_spatial_resampling.rs:163-222): one scratch texel
ST_DEV float4 spatial_trace_texel(const SceneDev& sc, const TraceStack& stk, float4 d0, float4 d1) {
    if (all_zero(d1)) return f4zero();
    Ray ray = ray_make(xyz(d0), oct_decode(f2(d1.x, d1.y)), d0.w);
    bool occ = trace_any(ray, sc, stk);
    return f4(occ ? 0.0f : 1.0f, d1.z, d1.w, 0.0f);
}
template <bool BATCHED>
__global__ void ST_LB_SPATIAL_TRACE k_spatial_trace(VPARAMS, const float4* __restrict__ buf_d0, const float4* __restrict__ buf_d1, float4* __restrict__ buf_d2) {
    VIEW; VIEW_ARENA(buf_d0); VIEW_ARENA(buf_d1); VIEW_ARENA(buf_d2);
    ST_TRACE_STACK();
    Px p = pixel_full(cam);
    if (!p.in) return;
    size_t i = pix(cam, p.x, p.y);
    buf_d2[i] = spatial_trace_texel(sc, stk, buf_d0[i], buf_d1[i]);
}
// the two visibility texels of a pair as K8 / K16 would leave them for K9 / K17 (a texel outside the texture reads as zero)
ST_DEV void trace_pair_texels(const CameraDev& cam, const SceneDev& sc, const TraceStack& stk, const PairTexels& o, Px g, float4* d2a, float4* d2b) {
    u32 ax = g.x * 2u, bx = g.x * 2u + 1u;
    *d2a = (o.state == 2 && in_tex(cam, ax, g.y)) ? spatial_trace_texel(sc, stk, o.a0, o.a1) : f4zero();
    *d2b = (o.state == 2 && in_tex(cam, bx, g.y)) ? spatial_trace_texel(sc, stk, o.b0, o.b1) : f4zero();
}

// K9 di_spatial_resampling::sample (di_spatial_resampling.rs:212-297); d0 / d1 = the pair's two visibility texels
ST_DEV void di_spatial_sample_pair(const CameraDev& cam, u32 seed, u32 frame, Px g, float4 d0, float4 d1) {
    uint2 lp = checker(g.x, g.y, frame / 2u + 1u);
    if (!cam_contains_u(cam.curr, lp.x, lp.y)) return;
    size_t npx = (size_t)cam.w * cam.h;
    size_t lhs_idx = screen_idx(cam, lp.x, lp.y);
    Rng rng = rng_make(seed, lp.x, lp.y);
    const float4* in = cam.di_reservoirs[1]; float4* out = cam.di_reservoirs[2];
    float lhs_rhs_vis = d0.x; u32 rhs_idx = fbits(d0.y);
    float rhs_lhs_vis = d1.x, lhs_rhs_pdf = d1.y, rhs_lhs_pdf = d1.z;
    DiRes lhs = di_load(in, lhs_idx);
    if (rhs_idx > 0u && (size_t)rhs_idx - 1 < npx) {
        DiRes rhs = di_load(in, (size_t)rhs_idx - 1);
        MisIn mi;
        mi.lhs_m = lhs.m; mi.rhs_m = rhs.m; mi.rhs_jacobian = 1.0f; mi.lhs_lhs_pdf = lhs.pdf;
        mi.lhs_rhs_pdf = lhs_rhs_pdf * lhs_rhs_vis; mi.rhs_lhs_pdf = rhs_lhs_pdf * rhs_lhs_vis; mi.rhs_rhs_pdf = rhs.pdf;
        MisOut mo = mis_eval(mi);
        DiRes main_ = di_zero();
        float main_pdf = 0.0f;
        if (di_update(main_, rng, lhs, mo.lhs_mis * mo.lhs_pdf * lhs.w)) main_pdf = mo.lhs_pdf;
        if (di_update(main_, rng, rhs, mo.rhs_mis * mo.rhs_pdf * rhs.w)) { main_pdf = mo.rhs_pdf; main_.occluded = lhs_rhs_vis == 0.0f; }
        main_.m = lhs.m + mo.m;
        main_.pdf = main_pdf;
        main_.w = res_norm(main_.w, main_pdf, 1.0f, 1.0f);
        di_store(main_, out, lhs_idx);
    } else di_store(lhs, out, lhs_idx);
    uint2 op = checker(g.x, g.y, frame / 2u);
    if (cam_contains_u(cam.curr, op.x, op.y)) { size_t oi = screen_idx(cam, op.x, op.y); di_store(di_load(in, oi), out, oi); }
}
template <bool BATCHED>
__global__ void __launch_bounds__(ST_BLOCK) k_di_spatial_sample(VPARAMS, u32 seed, u32 frame) {
    VIEW;
    Px g = pixel_half(cam);
    if (!g.in) return;
    di_spatial_sample_pair(cam, seed, frame, g, tex_or_zero(cam.di_diff_stash, cam, g.x * 2u, g.y), tex_or_zero(cam.di_diff_stash, cam, g.x * 2u + 1u, g.y));
}
// K7 + K8 + K9 in one launch (ST_OPT_FUSED_PASSES): one thread per checkerboard pair picks the neighbour, traces the pair's two shadow
// rays and merges — the three scratch textures (48 B per pixel written and read back) never leave the registers.  Same draws, same rays
// (direction through the same octahedral round trip), same merge as the three-launch sequence.
template <bool BATCHED>
__global__ void ST_LB_DI_SPATIAL_PICK k_di_spatial_fused(VPARAMS, int cur, u32 seed_pick, u32 seed_sample, u32 frame) {
    VIEW;
    ST_TRACE_STACK();
    Px g = pixel_half(cam);
    if (!g.in) return;
    PairTexels o = di_spatial_pick_pair(cam, sc, cur, seed_pick, frame, g);
    if (o.state == 0) return;
    float4 d2a, d2b; trace_pair_texels(cam, sc, stk, o, g, &d2a, &d2b);
    di_spatial_sample_pair(cam, seed_sample, frame, g, d2a, d2b);
}

// K10 di_resolving::main (di_resolving.rs:4-119)
template <bool BATCHED>
__global__ void ST_LB_DI_RESOLVING k_di_resolving(VPARAMS, int cur) {
    VIEW;
    ST_TRACE_STACK();
    Px p = pixel_full(cam);
    if (!p.in) return;
    size_t idx = screen_idx(cam, p.x, p.y);
    Hit hit = load_hit_lut(sc, cam.curr, cam.prim_gbuffer_d0[cur], cam.prim_gbuffer_d1[cur], cam, p.x, p.y);
    DiRes res = di_load(cam.di_reservoirs[2], idx);
    float confidence;
    LightRad rad;
    if (hit_some(hit)) {
        bool occ = trace_any(di_ray(res, hit.point), sc, stk);
        confidence = (res.occluded == occ) ? res.confidence : 0.0f;
        res.confidence = 1.0f;
        res.occluded = occ;
        if (occ) rad = lightrad_zero();
        else { rad = light_radiance(light_load(sc, res.light_id), hit); rad.radiance = rad.radiance * res.w; }
    } else {
        confidence = 1.0f;
        rad.radiance = atmosphere_sample(sc, world_sun_dir(sc.world), hit.dir);
        rad.diff = f3s(1.0f); rad.spec = f3s(0.0f);
    }
    float diff_brdf = (1.0f - hit.g.metallic) / kPi;
    size_t i = pix(cam, p.x, p.y);
    cam.di_diff_samples[i] = f4(rad.radiance * diff_brdf, confidence);
    cam.di_spec_samples[i] = f4(rad.radiance * rad.spec, confidence);
    di_store(res, cam.di_reservoirs[0], idx);
}

// K11 gi_reprojection::main (gi_reprojection.rs:4-51)
ST_DEV GiRes gi_reprojection_px(const CameraDev& cam, const Hit& hit, const Reproj& rp) {
    size_t npx = (size_t)cam.w * cam.h;
    GiRes res = gi_zero();
    if (reproj_some(rp)) {
        uint2 rpos = reproj_round(rp);
        size_t ridx = screen_idx(cam, rpos.x, rpos.y);
        if (ridx < npx) res = gi_load(cam.gi_reservoirs[0], ridx);
    }
    res.confidence = 1.0f;
    res.v1 = hit.point;
    return res;
}
template <bool BATCHED>
__global__ void __launch_bounds__(ST_BLOCK) k_gi_reprojection(VPARAMS, int cur) {
    VIEW;
    Px p = pixel_full(cam);
    if (!p.in) return;
    Hit hit = load_hit_lut(sc, cam.curr, cam.prim_gbuffer_d0[cur], cam.prim_gbuffer_d1[cur], cam, p.x, p.y);
    if (!hit_some(hit)) return;
    // strips: the columns the checkerboard passes do not cover (widths whose (W + 7) / 8 is odd) keep this entry as the spatial pass's
    // output, so there it is one of the rows a neighbouring strip's preview pass gathers
    gi_store_m(cam, gi_reprojection_px(cam, hit, reproj_decode(cam.reprojection_map[pix(cam, p.x, p.y)])), cam.gi_reservoirs[2], screen_idx(cam, p.x, p.y), p.y,
               (int)p.x >= 2 * half_grid_w(cam.w) ? cam.gi_mirror_reach : 0);
}

// K12 gi_sampling_a::main (gi_sampling_a.rs:4-122)
// returns false where the kernel leaves without writing its three scratch texels (gi_d0: ray direction + pdf, gi_d1/gi_d2: the packed
// G-buffer entry of what the ray hit)
ST_DEV bool gi_sampling_a_pair(const CameraDev& cam, const SceneDev& sc, const TraceStack& stk, int cur, u32 seed, u32 frame, Px g, float4* t0, float4* t1, float4* t2) {
    bool tracing = gi_tracing_frame(frame);
    uint2 sp = tracing ? checker(g.x, g.y, frame / 2u) : checker(g.x, g.y, frame);
    if (!cam_contains_u(cam.curr, sp.x, sp.y)) return false;
    size_t idx = screen_idx(cam, sp.x, sp.y);
    Ray gi_r; float gi_pdf_;
    if (tracing) {
        Rng rng = rng_make(seed, sp.x, sp.y);
        Hit hit = load_hit_lut(sc, cam.curr, cam.prim_gbuffer_d0[cur], cam.prim_gbuffer_d1[cur], cam, sp.x, sp.y);
        if (!hit_some(hit)) return false;
        BrdfS s = brdf_layered_sample(hit.g, rng, -hit.dir);
        gi_r = ray_make(hit.point, s.dir);
        gi_pdf_ = s.pdf;
    } else {
        GiRes res = gi_load(cam.gi_reservoirs[2], idx);
        if (res.m == 0.0f) return false;
        gi_r = ray_make(res.v1, gi_dir(res, res.v1));
        gi_pdf_ = 1.0f;
    }
    TriHit gh = trace_closest(gi_r, sc, stk);
    GBuf gg = gbuf_zero();
    u32 gi_color_bits = 0u;
    if (trihit_some(gh)) {
        GpuMaterial m = sc.materials[gh.material_id];
        m.roughness = rmax(m.roughness, 0.75f * 0.75f);   // Material::regularize (material.rs:25-27)
        gg.base_color = mat_base_color(sc, m, gh.uv); gg.normal = gh.normal; gg.metallic = m.metallic; gg.emissive = mat_emissive(sc, m, gh.uv);
        gi_color_bits = all_zero(m.base_color_texture) ? __ldg(sc.material_packed + gh.material_id) : gbuf_pack_color(gg.base_color);
        gg.roughness = m.roughness; gg.reflectance = m.reflectance; gg.depth = dist(gi_r.o, gh.point);
    }
    gbuf_pack_pre(gg, gi_color_bits, t1, t2);
    *t0 = f4(gi_r.d, gi_pdf_);
    return true;
}
template <bool BATCHED>
__global__ void ST_LB_GI_SAMPLING_A k_gi_sampling_a(VPARAMS, int cur, u32 seed, u32 frame) {
    VIEW;
    ST_TRACE_STACK();
    Px g = pixel_half(cam);
    if (!g.in) return;
    float4 t0, t1, t2;
    if (!gi_sampling_a_pair(cam, sc, stk, cur, seed, frame, g, &t0, &t1, &t2)) return;
    size_t gi = pix(cam, g.x, g.y);
    cam.gi_d0[gi] = t0; cam.gi_d1[gi] = t1; cam.gi_d2[gi] = t2;
}

// K13 gi_sampling_b::main (gi_sampling_b.rs:4-235)
ST_DEV void gi_sampling_b_pair(const CameraDev& cam, const SceneDev& sc, const TraceStack& stk, int cur, u32 seed, u32 frame, Px g, float4 d0, float4 d1, float4 d2) {
    bool tracing = gi_tracing_frame(frame);
    uint2 sp = tracing ? checker(g.x, g.y, frame / 2u) : checker(g.x, g.y, frame);
    if (!cam_contains_u(cam.curr, sp.x, sp.y)) return;
    size_t idx = screen_idx(cam, sp.x, sp.y);
    Hit prim = load_hit_lut(sc, cam.curr, cam.prim_gbuffer_d0[cur], cam.prim_gbuffer_d1[cur], cam, sp.x, sp.y);
    if (!hit_some(prim)) return;
    Rng rng; Hit gh; float gi_pdf_;
    if (tracing) {
        rng = rng_make(seed, sp.x, sp.y);
        gh = hit_make(ray_make(prim.point, xyz(d0)), gbuf_unpack(sc, d1, d2));
        gi_pdf_ = d0.w;
    } else {
        GiRes res = gi_load(cam.gi_reservoirs[2], idx);
        if (res.m == 0.0f) return;
        rng.s = res.rng;
        gh = hit_make(ray_make(res.v1, xyz(d0)), gbuf_unpack(sc, d1, d2));
        gi_pdf_ = 1.0f;
    }
    u32 rng_state = rng.s;
    const u32 SKY = 0xffffffffu;
    float3 sun_dir = world_sun_dir(sc.world);
    u32 light_id; float light_pdf; float3 light_rad; float3 light_dir = f3s(0.f);
    if (!hit_some(gh)) { light_id = SKY; light_pdf = 1.0f; light_rad = atmosphere_sample(sc, sun_dir, gh.dir); }
    else {
        float atm_pdf = (sc.world.sun_altitude <= -1.0f) ? 0.0f : 0.25f;
        if (sc.world.light_count == 0u || rng_f(rng) < atm_pdf) {
            light_id = SKY; light_pdf = atm_pdf;
            light_dir = rng_hemisphere(rng, gh.g.normal);
            light_rad = atmosphere_sample(sc, sun_dir, light_dir) * dot(gh.g.normal, light_dir);
        } else {
            EphRes er = ephemeral_build(rng, sc, gh);
            if (er.w > 0.0f) { light_id = er.light_id; light_pdf = (1.0f / er.w) * (1.0f - atm_pdf); light_rad = er.rad.radiance * (f3s(1.0f) + er.rad.spec); }
            else { light_id = 0u; light_pdf = 1.0f; light_rad = f3s(0.f); }
        }
    }
    float3 radiance;
    if (light_pdf > 0.0f) {
        float vis;
        if (hit_some(gh)) {
            Ray r = (light_id == SKY) ? ray_make(gh.point, light_dir) : light_ray_wnoise(light_load(sc, light_id), rng, gh.point);
            vis = trace_any(r, sc, stk) ? 0.0f : 1.0f;
        } else vis = 1.0f;
        radiance = light_rad * vis / light_pdf;
    } else radiance = f3s(0.f);
    if (hit_some(gh)) { radiance = radiance * (xyz(gh.g.base_color) / kPi); radiance = radiance + gh.g.emissive; }
    GiRes res = gi_zero();
    if (gi_pdf_ > 0.0f) {
        res.rng = rng_state; res.radiance = radiance; res.v1 = prim.point;
        if (hit_some(gh)) { res.v2 = gh.point; res.v2n = gh.g.normal; }
        else { res.v2 = prim.point + gh.dir * 1000.0f; res.v2n = -gh.dir; }
        res.m = 1.0f; res.w = 1.0f / gi_pdf_;
        res.pdf = 0.0f;
        res.pdf = gi_pdf(res, prim);
    }
    gi_store(res, cam.gi_reservoirs[1], idx);
}
template <bool BATCHED>
__global__ void ST_LB_GI_SAMPLING_B k_gi_sampling_b(VPARAMS, int cur, u32 seed, u32 frame) {
    VIEW;
    ST_TRACE_STACK();
    Px g = pixel_half(cam);
    if (!g.in) return;
    size_t gi = pix(cam, g.x, g.y);
    gi_sampling_b_pair(cam, sc, stk, cur, seed, frame, g, cam.gi_d0[gi], cam.gi_d1[gi], cam.gi_d2[gi]);
}
// K12 + K13 in one launch (ST_OPT_FUSED_PASSES): the bounce ray is traced and shaded by the same thread; the hit still goes through
// GBufferEntry's pack / unpack (its 8-bit quantisation is part of the result), just not through memory.
template <bool BATCHED>
__global__ void ST_LB_GI_SAMPLING_B k_gi_sampling_fused(VPARAMS, int cur, u32 seed_a, u32 seed_b, u32 frame) {
    VIEW;
    ST_TRACE_STACK();
    Px g = pixel_half(cam);
    if (!g.in) return;
    float4 t0, t1, t2;
    if (!gi_sampling_a_pair(cam, sc, stk, cur, seed_a, frame, g, &t0, &t1, &t2)) return;
    gi_sampling_b_pair(cam, sc, stk, cur, seed_b, frame, g, t0, t1, t2);
}

// K14 gi_temporal_resampling::main (gi_temporal_resampling.rs:4-156)
// `inline_reprojection` (ST_OPT_FUSED_PASSES, tracing frames): K11 is evaluated here instead of in its own launch — last frame's
// reservoir is fetched from gi_reservoirs[0] at the reprojected position directly, and handed on as K11 would have left it in
// gi_reservoirs[2] (its normal goes through the same octahedral store / load round trip).  gi_reservoirs[2] itself is then only written
// for the columns a later pass still reads there (those the checkerboard passes do not cover when the width is odd).
template <bool BATCHED>
__global__ void ST_LB_GI_TEMPORAL k_gi_temporal(VPARAMS, int cur, u32 seed, u32 frame, int inline_reprojection) {
    VIEW;
    Px p = pixel_full(cam);
    if (!p.in) return;
    bool tracing = gi_tracing_frame(frame);
    size_t lhs_idx = screen_idx(cam, p.x, p.y);
    Rng rng = rng_make(seed, p.x, p.y);
    Hit lhs_hit = load_hit_lut(sc, cam.curr, cam.prim_gbuffer_d0[cur], cam.prim_gbuffer_d1[cur], cam, p.x, p.y);
    float4* curr = cam.gi_reservoirs[1];
    if (!hit_some(lhs_hit)) { gi_store_m(cam, gi_zero(), curr, lhs_idx, p.y, cam.gi_mirror_reach); return; }
    bool got = tracing ? (frame % 2u == 0u && checker_at(p.x, p.y, frame / 2u)) : checker_at(p.x, p.y, frame);
    GiRes lhs = got ? gi_load(curr, lhs_idx) : gi_zero();
    GiRes rhs = gi_zero();
    Hit rhs_hit = hit_zero();
    Reproj rp = reproj_decode(cam.reprojection_map[pix(cam, p.x, p.y)]);
    if (inline_reprojection) {
        GiRes r11 = gi_reprojection_px(cam, lhs_hit, rp);
        if ((int)p.x >= 2 * half_grid_w(cam.w)) gi_store_m(cam, r11, cam.gi_reservoirs[2], lhs_idx, p.y, cam.gi_mirror_reach);
        if (reproj_some(rp)) { rhs = r11; rhs.v2n = oct_decode(oct_encode(r11.v2n)); }
    } else if (reproj_some(rp)) rhs = gi_load(cam.gi_reservoirs[2], lhs_idx);
    if (reproj_some(rp)) {
        rhs.confidence = 1.0f;
        rhs.m = rmin(rhs.m, 128.0f);
        if (!tracing && lhs.m != 0.0f && rhs.m != 0.0f && gi_exists(rhs)) {
            if (dist(lhs.radiance, rhs.radiance) > 0.33f) rhs.confidence = 0.0f;
            rhs.radiance = lhs.radiance; rhs.v2 = lhs.v2; rhs.v2n = lhs.v2n;
        }
        if (rhs.m != 0.0f) {
            uint2 rpos = reproj_round(rp);
            rhs_hit = load_hit_lut(sc, cam.prev, cam.prim_gbuffer_d0[cur ^ 1], cam.prim_gbuffer_d1[cur ^ 1], cam, rpos.x, rpos.y);
        }
    }
    GiRes main_ = gi_zero();
    float main_pdf = 0.0f;
    if (tracing) {
        MisIn mi;
        mi.lhs_m = lhs.m; mi.rhs_m = rhs.m; mi.rhs_jacobian = 1.0f; mi.lhs_lhs_pdf = lhs.pdf; mi.rhs_rhs_pdf = rhs.pdf;
        mi.lhs_rhs_pdf = ((lhs.m > 0.0f) & hit_some(rhs_hit)) ? gi_pdf(lhs, rhs_hit) : 0.0f;
        mi.rhs_lhs_pdf = (rhs.m > 0.0f) ? gi_pdf(rhs, lhs_hit) : 0.0f;
        MisOut mo = mis_eval(mi);
        if (gi_update(main_, rng, lhs, mo.lhs_mis * mo.lhs_pdf * lhs.w)) main_pdf = mo.lhs_pdf;
        if (gi_update(main_, rng, rhs, mo.rhs_mis * mo.rhs_pdf * rhs.w)) main_pdf = mo.rhs_pdf;
        main_.m = lhs.m + mo.m;
        main_.confidence = 1.0f;
        main_.w = res_norm(main_.w, main_pdf, 1.0f, 1.0f);
    } else {
        if (gi_merge(main_, rng, rhs, rhs.pdf)) main_pdf = rhs.pdf;
        main_.confidence = rhs.confidence;
        main_.w = res_norm(main_.w, main_pdf, 1.0f, main_.m);
    }
    main_.pdf = main_pdf;
    main_.v1 = lhs_hit.point;
    main_.w = rmin(main_.w, 5.0f);
    gi_store_m(cam, main_, curr, lhs_idx, p.y, cam.gi_mirror_reach);
}

// K15 gi_spatial_resampling::pick (gi_spatial_resampling.rs:4-160); scratch = gi_d0, gi_d1
ST_DEV PairTexels gi_spatial_pick_pair(const CameraDev& cam, const SceneDev& sc, int cur, u32 seed, u32 frame, Px g) {
    PairTexels o; o.a0 = o.a1 = o.b0 = o.b1 = f4zero(); o.state = 0;
    uint2 lp = checker(g.x, g.y, frame / 2u + 1u);
    if (!cam_contains_u(cam.curr, lp.x, lp.y)) return o;
    o.state = 1;
    size_t lhs_idx = screen_idx(cam, lp.x, lp.y);
    Rng rng = rng_make(seed, lp.x, lp.y);
    const float4* gd0 = cam.prim_gbuffer_d0[cur]; const float4* gd1 = cam.prim_gbuffer_d1[cur];
    const float4* reservoirs = cam.gi_reservoirs[1];
    Hit lhs_hit = load_hit_lut(sc, cam.curr, gd0, gd1, cam, lp.x, lp.y);
    GiRes lhs = gi_load(reservoirs, lhs_idx);
    if (!hit_some(lhs_hit) || lhs.m == 0.0f) return o;
    GiRes rhs = gi_zero();
    size_t rhs_idx = 0;
    Hit rhs_hit = hit_zero();
    float rhs_jac = 0.0f;
    float max_radius = 128.0f;
    for (u32 nth = 0u; nth < 8u; nth++) {
        float2 off = rng_disk(rng) * max_radius;
        float2 fp = f2((float)lp.x, (float)lp.y) + off;
        uint2 rpos = cam_contain(cam.curr, to_i32_sat(fp.x), to_i32_sat(fp.y));
        if (rpos.x == lp.x && rpos.y == lp.y) continue;
        float4 nd = tex_or_zero(cam.surface_nd, cam, rpos.x, rpos.y);
        if (nd.w == 0.0f) { max_radius = rmax(max_radius * 0.5f, 5.0f); continue; }
        if (fabs_(nd.w - lhs_hit.g.depth) > 0.33f * lhs_hit.g.depth) { max_radius = rmax(max_radius * 0.5f, 5.0f); continue; }
        if (dot(xyz(nd), lhs_hit.g.normal) < 0.33f) { max_radius = rmax(max_radius * 0.5f, 5.0f); continue; }
        rhs_idx = screen_idx(cam, rpos.x, rpos.y);
        rhs = gi_load(reservoirs, rhs_idx);
        if (rhs.m == 0.0f) continue;
        rhs_jac = gi_jacobian(rhs, lhs_hit.point);
        if (rhs_jac < 1.0f / 10.0f || rhs_jac > 10.0f) { rhs.m = 0.0f; continue; }
        rhs_jac = rclamp(rhs_jac, 1.0f / 3.0f, 3.0f);
        rhs_hit = load_hit_lut(sc, cam.curr, gd0, gd1, cam, rpos.x, rpos.y);
        break;
    }
    if (rhs.m == 0.0f || !hit_some(rhs_hit)) return o;
    float lhs_rhs_pdf = gi_pdf(lhs, rhs_hit);
    float rhs_lhs_pdf = gi_pdf(rhs, lhs_hit);
    Ray ra = (lhs_rhs_pdf > 0.0f) ? gi_ray(lhs, rhs_hit.point) : ray_zero();
    Ray rb = (rhs_lhs_pdf > 0.0f) ? gi_ray(rhs, lhs_hit.point) : ray_zero();
    float2 na = oct_encode(ra.d), nb = oct_encode(rb.d);
    o.a0 = f4(ra.o, ra.len); o.a1 = f4(na.x, na.y, bitsf((u32)rhs_idx + 1u), rhs_jac);
    o.b0 = f4(rb.o, rb.len); o.b1 = f4(nb.x, nb.y, lhs_rhs_pdf, rhs_lhs_pdf);
    o.state = 2;
    return o;
}
template <bool BATCHED>
__global__ void ST_LB_GI_SPATIAL_PICK k_gi_spatial_pick(VPARAMS, int cur, u32 seed, u32 frame) {
    VIEW;
    Px g = pixel_half(cam);
    if (!g.in) return;
    store_pair_texels(cam, gi_spatial_pick_pair(cam, sc, cur, seed, frame, g), cam.gi_d0, cam.gi_d1, g);
}

// K17 gi_spatial_resampling::sample (gi_spatial_resampling.rs:225-314)
ST_DEV void gi_spatial_sample_pair(const CameraDev& cam, u32 seed, u32 frame, Px g, float4 d0, float4 d1) {
    uint2 sp = checker(g.x, g.y, frame / 2u + 1u);
    if (!cam_contains_u(cam.curr, sp.x, sp.y)) return;
    size_t npx = (size_t)cam.w * cam.h;
    size_t idx = screen_idx(cam, sp.x, sp.y);
    Rng rng = rng_make(seed, sp.x, sp.y);
    const float4* in = cam.gi_reservoirs[1]; float4* out = cam.gi_reservoirs[2];
    float lhs_rhs_vis = d0.x; u32 rhs_idx = fbits(d0.y); float rhs_jac = d0.z;
    float rhs_lhs_vis = d1.x, lhs_rhs_pdf = d1.y, rhs_lhs_pdf = d1.z;
    GiRes lhs = gi_load(in, idx);
    if (rhs_idx > 0u && (size_t)rhs_idx - 1 < npx) {
        GiRes rhs = gi_load(in, (size_t)rhs_idx - 1);
        MisIn mi;
        mi.lhs_m = lhs.m; mi.rhs_m = rhs.m; mi.rhs_jacobian = rhs_jac; mi.lhs_lhs_pdf = lhs.pdf;
        mi.lhs_rhs_pdf = lhs_rhs_pdf * lhs_rhs_vis; mi.rhs_lhs_pdf = rhs_lhs_pdf * rhs_lhs_vis; mi.rhs_rhs_pdf = rhs.pdf;
        MisOut mo = mis_eval(mi);
        GiRes main_ = gi_zero();
        float main_pdf = 0.0f;
        if (gi_update(main_, rng, lhs, mo.lhs_mis * mo.lhs_pdf * lhs.w)) main_pdf = mo.lhs_pdf;
        if (gi_update(main_, rng, rhs, mo.rhs_mis * mo.rhs_pdf * rhs.w * rhs_jac)) main_pdf = mo.rhs_pdf;
        main_.m = lhs.m + mo.m;
        main_.confidence = 1.0f;
        main_.pdf = main_pdf;
        main_.v1 = lhs.v1;
        main_.w = res_norm(main_.w, main_pdf, 1.0f, 1.0f);
        main_.w = rmin(main_.w, 5.0f);
        gi_store_m(cam, main_, out, idx, sp.y, cam.gi_mirror_reach);
    } else gi_store_m(cam, lhs, out, idx, sp.y, cam.gi_mirror_reach);
    uint2 op = checker(g.x, g.y, frame / 2u);
    if (cam_contains_u(cam.curr, op.x, op.y)) { size_t oi = screen_idx(cam, op.x, op.y); gi_store_m(cam, gi_load(in, oi), out, oi, op.y, cam.gi_mirror_reach); }
}
template <bool BATCHED>
__global__ void ST_LB_GI_SPATIAL_SAMPLE k_gi_spatial_sample(VPARAMS, u32 seed, u32 frame) {
    VIEW;
    Px g = pixel_half(cam);
    if (!g.in) return;
    gi_spatial_sample_pair(cam, seed, frame, g, tex_or_zero(cam.gi_d2, cam, g.x * 2u, g.y), tex_or_zero(cam.gi_d2, cam, g.x * 2u + 1u, g.y));
}
// K15 + K16 + K17 in one launch (ST_OPT_FUSED_PASSES), like k_di_spatial_fused
template <bool BATCHED>
__global__ void ST_LB_GI_SPATIAL_PICK k_gi_spatial_fused(VPARAMS, int cur, u32 seed_pick, u32 seed_sample, u32 frame) {
    VIEW;
    ST_TRACE_STACK();
    Px g = pixel_half(cam);
    if (!g.in) return;
    PairTexels o = gi_spatial_pick_pair(cam, sc, cur, seed_pick, frame, g);
    if (o.state == 0) return;
    float4 d2a, d2b; trace_pair_texels(cam, sc, stk, o, g, &d2a, &d2b);
    gi_spatial_sample_pair(cam, seed_sample, frame, g, d2a, d2b);
}

// K18 gi_preview_resampling::main (gi_preview_resampling.rs:4-138).  Returns false where the kernel exits without writing (quirk C-6).
ST_DEV bool gi_preview_px(const CameraDev& cam, const SceneDev& sc, const Hit& chit, u32 seed, u32 nth, const float4* __restrict__ in, Px p, GiRes* result) {
    size_t cidx = screen_idx(cam, p.x, p.y);
    Rng rng = rng_make(seed, p.x, p.y);
    if (!hit_some(chit)) { *result = gi_zero(); return true; }
    GiRes main_ = gi_zero();
    float main_pdf = 0.0f;
    GiRes center = gi_load(in, cidx);
    if (gi_merge(main_, rng, center, center.pdf)) main_pdf = center.pdf;
    u32 max_samples = to_u32_sat(lerpc(8.0f, 0.0f, main_.m / 8.0f));
    float max_radius = (nth == 0u) ? 128.0f : 64.0f;
    const float4* __restrict__ surf = cam.surface_nd;
    for (u32 k = 0u; k < max_samples; k++) {
        float2 off = rng_disk(rng) * max_radius;
        float2 fp = f2((float)p.x, (float)p.y) + off;
        uint2 sp = cam_contain(cam.curr, to_i32_sat(fp.x), to_i32_sat(fp.y));
        if (sp.x == p.x && sp.y == p.y) return false;   // quirk C-6: the kernel exits without writing
        if (!cam_contains_u(cam.curr, sp.x, sp.y)) continue;
        float4 nd = surf[pix(cam, sp.x, sp.y)];
        if (nd.w == 0.0f) continue;
        if (fabs_(nd.w - chit.g.depth) > 0.25f * chit.g.depth) continue;
        if (dot(xyz(nd), chit.g.normal) < 0.5f) continue;
        GiRes s = gi_load(in, screen_idx(cam, sp.x, sp.y));
        if (s.m == 0.0f) continue;
        float s_pdf = gi_pdf(s, chit);
        float s_jac = gi_jacobian(s, chit.point);
        if (s_jac < 1.0f / 10.0f || s_jac > 10.0f) continue;
        s_jac = rclamp(s_jac, 1.0f / 3.0f, 3.0f);
        if (gi_merge(main_, rng, s, s_pdf * s_jac)) main_pdf = s_pdf;
    }
    main_.confidence = center.confidence;
    main_.pdf = main_pdf;
    main_.v1 = center.v1;
    main_.w = res_norm(main_.w, main_pdf, 1.0f, main_.m);
    main_.w = rmin(main_.w, 5.0f);
    *result = main_;
    return true;
}
template <bool BATCHED>
__global__ void ST_LB_GI_PREVIEW k_gi_preview(VPARAMS, int cur, u32 seed, u32 nth, const float4* __restrict__ in, float4* __restrict__ out, int reach) {
    VIEW; VIEW_ARENA(in); VIEW_ARENA(out);
    Px p = pixel_full(cam);
    if (!p.in) return;
    Hit chit = load_hit_lut(sc, cam.curr, cam.prim_gbuffer_d0[cur], cam.prim_gbuffer_d1[cur], cam, p.x, p.y);
    GiRes r;
    if (gi_preview_px(cam, sc, chit, seed, nth, in, p, &r)) gi_store_m(cam, r, out, screen_idx(cam, p.x, p.y), p.y, reach);
}

// K19 gi_resolving::main (gi_resolving.rs:4-67): shades the pixel from `res` (the entry the second preview pass left in gi_reservoirs[0]),
// then replaces that entry with the frame's source reservoir
ST_DEV void gi_resolving_px(const CameraDev& cam, const Hit& hit, const GiRes& res, const float4* __restrict__ in, Px p) {
    size_t idx = screen_idx(cam, p.x, p.y);
    float confidence; float3 radiance;
    if (hit_some(hit)) { confidence = res.confidence; radiance = res.w * gi_cosine(res, hit) * res.radiance; }
    else { confidence = 1.0f; radiance = f3s(0.f); }
    float diff_brdf = (1.0f - hit.g.metallic) / kPi;
    float3 spec = gi_spec(res, hit);
    size_t i = pix(cam, p.x, p.y);
    cam.gi_diff_samples[i] = f4(radiance * diff_brdf, confidence);
    cam.gi_spec_samples[i] = f4(radiance * spec, confidence);
    gi_store(gi_load(in, idx), cam.gi_reservoirs[0], idx);
}
template <bool BATCHED>
__global__ void ST_LB_GI_RESOLVING k_gi_resolving(VPARAMS, int cur, const float4* __restrict__ in) {
    VIEW; VIEW_ARENA(in);
    Px p = pixel_full(cam);
    if (!p.in) return;
    Hit hit = load_hit_lut(sc, cam.curr, cam.prim_gbuffer_d0[cur], cam.prim_gbuffer_d1[cur], cam, p.x, p.y);
    gi_resolving_px(cam, hit, gi_load(cam.gi_reservoirs[0], screen_idx(cam, p.x, p.y)), in, p);
}
// second preview pass + K19 in one launch (ST_OPT_FUSED_PASSES): the pass's result is shaded straight away instead of going through
// gi_reservoirs[0] (K19 only consumes fields that a store / load leaves untouched); where the pass exits without writing (quirk C-6) K19
// sees last frame's entry, which is what is loaded here then.
template <bool BATCHED>
__global__ void ST_LB_GI_PREVIEW k_gi_preview_resolve(VPARAMS, int cur, u32 seed, const float4* __restrict__ in, const float4* __restrict__ source) {
    VIEW; VIEW_ARENA(in); VIEW_ARENA(source);
    Px p = pixel_full(cam);
    if (!p.in) return;
    Hit chit = load_hit_lut(sc, cam.curr, cam.prim_gbuffer_d0[cur], cam.prim_gbuffer_d1[cur], cam, p.x, p.y);
    GiRes r;
    if (!gi_preview_px(cam, sc, chit, seed, 1u, in, p, &r)) r = gi_load(cam.gi_reservoirs[0], screen_idx(cam, p.x, p.y));
    gi_resolving_px(cam, chit, r, source, p);
}

#if ST_EXACT_ONLY
// K20 frame_denoising::reproject (frame_denoising.rs:4-78)
template <bool BATCHED>
__global__ void __launch_bounds__(ST_BLOCK) k_denoise_reproject(VPARAMS, int cur, const float4* __restrict__ prev_colors, const float4* __restrict__ prev_moments,
                                                                const float4* __restrict__ samples, float4* __restrict__ colors, float4* __restrict__ moments) {
    VIEW; VIEW_ARENA(prev_colors); VIEW_ARENA(prev_moments); VIEW_ARENA(samples); VIEW_ARENA(colors); VIEW_ARENA(moments);
    Px p = pixel_full(cam);
    if (!p.in) return;
    size_t i = pix(cam, p.x, p.y);
    float4 sample = samples[i];
    if (cam.prim_surface_map[cur][i].z == 0.0f) { store4m(cam, colors + i, sample, p.y, ST_REACH_SVGF); return; }
    float sl = luma(xyz(sample));
    Reproj rp = reproj_decode(cam.reprojection_map[i]);
    float3 color, moment;
    if (reproj_some(rp) && sample.w > 0.0f) {
        float4 pc = history_fetch(rp, prev_colors, cam.w, cam.h);
        float4 pm = history_fetch(rp, prev_moments, cam.w, cam.h);
        float hist = rmin(pm.x + 1.0f, 16.0f);
        float alpha = 1.0f / hist;
        color = lerpc(xyz(pc), xyz(sample), alpha);
        moment = f3(hist, lerpc(pm.y, sl, alpha), lerpc(pm.z, sl * sl, alpha));
    } else { color = xyz(sample); moment = f3(1.0f, sl, sl * sl); }
    store4m(cam, colors + i, f4(color, 0.0f), p.y, ST_REACH_SVGF);
    store4m(cam, moments + i, f4(moment, 0.0f), p.y, ST_REACH_SVGF);
}

// K20 for the DI and the GI signal in one launch: the surface depth and the reprojection entry are read once
// (192 instead of 2 x 112 B/px); per signal exactly the arithmetic of k_denoise_reproject.
struct ReprojectSignal { const float4* prev_colors; const float4* prev_moments; const float4* samples; float4* colors; float4* moments; };
ST_DEV void denoise_reproject_signal(const CameraDev& cam, size_t i, u32 y, float4 sample, const Reproj& rp, bool has_rp, const ReprojectSignal& g) {
    float sl = luma(xyz(sample));
    float3 color, moment;
    if (has_rp && sample.w > 0.0f) {
        float4 pc = history_fetch(rp, g.prev_colors, cam.w, cam.h);
        float4 pm = history_fetch(rp, g.prev_moments, cam.w, cam.h);
        float hist = rmin(pm.x + 1.0f, 16.0f);
        float alpha = 1.0f / hist;
        color = lerpc(xyz(pc), xyz(sample), alpha);
        moment = f3(hist, lerpc(pm.y, sl, alpha), lerpc(pm.z, sl * sl, alpha));
    } else { color = xyz(sample); moment = f3(1.0f, sl, sl * sl); }
    store4m(cam, g.colors + i, f4(color, 0.0f), y, ST_REACH_SVGF);
    store4m(cam, g.moments + i, f4(moment, 0.0f), y, ST_REACH_SVGF);
}
ST_DEV void denoise_reproject_pair_px(const CameraDev& cam, int cur, Px p, const ReprojectSignal& di, const ReprojectSignal& gi) {
    size_t i = pix(cam, p.x, p.y);
    float4 sd = di.samples[i], sg = gi.samples[i];
    if (cam.prim_surface_map[cur][i].z == 0.0f) { store4m(cam, di.colors + i, sd, p.y, ST_REACH_SVGF); store4m(cam, gi.colors + i, sg, p.y, ST_REACH_SVGF); return; }
    Reproj rp = reproj_decode(cam.reprojection_map[i]);
    bool has_rp = reproj_some(rp);
    denoise_reproject_signal(cam, i, p.y, sd, rp, has_rp, di);
    denoise_reproject_signal(cam, i, p.y, sg, rp, has_rp, gi);
}
ST_DEV ReprojectSignal signal_in_view(const ReprojectSignal& g, const ViewDev& v) {
    return {arena_ptr<true>(g.prev_colors, v), arena_ptr<true>(g.prev_moments, v), arena_ptr<true>(g.samples, v), arena_ptr<true>(g.colors, v), arena_ptr<true>(g.moments, v)};
}
template <bool BATCHED>
__global__ void __launch_bounds__(ST_BLOCK) k_denoise_reproject_pair(VPARAMS, int cur, const __grid_constant__ ReprojectSignal di, const __grid_constant__ ReprojectSignal gi) {
    VIEW;
    Px p = pixel_full(cam);
    if (!p.in) return;
    if (BATCHED) denoise_reproject_pair_px(cam, cur, p, signal_in_view(di, view), signal_in_view(gi, view));
    else denoise_reproject_pair_px(cam, cur, p, di, gi);
}

// frame_denoising::sample_weight (frame_denoising.rs:363-392), split into the part that is common to
// the DI and GI signals (depth ramp, normal^64) and the per-signal luminance term:
//   weight = exp(-|sqrt(lc) - sqrt(ls)| * luma_sigma) * depth_weight * normal_weight
// A zero depth or normal factor makes the product 0 (or NaN), never > 0, so the caller may skip the tap.
//
// Two arithmetic flavours (template parameter FAST):
//   FAST = false  strict IEEE f32 with the polynomial exp: bit-identical to the CPU oracle.
//   FAST = true   the SFU approximations a GPU shader compiler emits for GLSL exp/sqrt/div
//                 (ex2.approx, sqrt.approx, rcp.approx; <= 2 ulp each) and fused multiply-adds.  Only the
//                 edge-stopping weights / normalisation of the denoiser use it; reservoirs, hits and every
//                 other buffer stay bit-exact, the denoised colours stay inside north_star's 1e-3 tolerance.
ST_DEV float sfu_ex2(float x) { float r; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
ST_DEV float sfu_sqrt(float x) { float r; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
ST_DEV float sfu_rcp(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
template <bool FAST> ST_DEV float sv_sqrt(float x) { return FAST ? sfu_sqrt(x) : sqrtf(x); }
template <bool FAST> ST_DEV float sv_luma(float3 c) { return FAST ? __fmaf_rn(c.z, 0.0722f, __fmaf_rn(c.y, 0.7152f, c.x * 0.2126f)) : luma(c); }
template <bool FAST> ST_DEV float svgf_depth_weight(float c_depth, float s_depth, float depth_sigma) {
    float leeway = c_depth * depth_sigma;
    float diff = fabs_(s_depth - c_depth);
    if (diff >= leeway) return 0.0f;
    return FAST ? __fmaf_rn(-diff, sfu_rcp(leeway), 1.0f) : 1.0f - diff / leeway;
}
template <bool FAST> ST_DEV float svgf_normal_weight(float3 c_normal, float3 s_normal) {
    float d = FAST ? __fmaf_rn(s_normal.z, c_normal.z, __fmaf_rn(s_normal.y, c_normal.y, s_normal.x * c_normal.x)) : dot(s_normal, c_normal);
    return pow_det(rmax(d, 0.0f), 64.0f);   // six squarings
}
template <bool FAST> ST_DEV float svgf_luma_weight(float sqrt_center_luma, float sample_luma, float luma_sigma) {
    float lw = fabs_(sqrt_center_luma - sv_sqrt<FAST>(sample_luma)) * luma_sigma;
    return FAST ? sfu_ex2(lw * -1.44269504088896341f) : exp_det(-lw);
}

// K21 frame_denoising::estimate_variance (frame_denoising.rs:81-217)
template <bool BATCHED, bool FAST>
__global__ void __launch_bounds__(ST_BLOCK) k_denoise_variance(VPARAMS, int cur) {
    VIEW;
    Px p = pixel_full(cam);
    if (!p.in) return;
    size_t i = pix(cam, p.x, p.y);
    const float4* __restrict__ snd = cam.surface_nd;
    const float4* __restrict__ di_colors = cam.di_diff_curr_colors; const float4* __restrict__ gi_colors = cam.gi_diff_curr_colors;
    float4 cnd = snd[i];
    float4 cdi = di_colors[i], cgi = gi_colors[i];
    if (cnd.w == 0.0f) { cam.di_diff_stash[i] = cdi; cam.gi_diff_stash[i] = cgi; return; }
    float4 mdi = cam.di_diff_moments[cur][i], mgi = cam.gi_diff_moments[cur][i];
    float di_var, gi_var;
    if (mdi.x >= 4.0f) { di_var = mdi.z - sq(mdi.y); gi_var = mgi.z - sq(mgi.y); }
    else {
        float3 cn = xyz(cnd);
        float scdl = sv_sqrt<FAST>(sv_luma<FAST>(xyz(cdi))), scgl = sv_sqrt<FAST>(sv_luma<FAST>(xyz(cgi)));
        float3 sdi = f3s(0.f), sgi = f3s(0.f);
        int ox = -2, oy = -2;
        for (;;) {   // quirk C-3: row -2 spans x in [-2,2], rows -1..2 span x in [-3,2]
            int sx = (int)p.x + ox, sy = (int)p.y + oy;
            if (cam_contains_i(cam.curr, sx, sy)) {
                size_t si = pix(cam, (u32)sx, (u32)sy);
                float4 nds = snd[si];
                if (nds.w != 0.0f) {
                    float common = svgf_depth_weight<FAST>(cnd.w, nds.w, 0.2f);
                    float nw = svgf_normal_weight<FAST>(cn, xyz(nds));
                    float sl = sv_luma<FAST>(xyz(di_colors[si]));
                    float w = svgf_luma_weight<FAST>(scdl, sl, 1.0f) * common * nw;
                    sdi = sdi + f3(sl, sl * sl, 1.0f) * f3s(w);
                    float gl = sv_luma<FAST>(xyz(gi_colors[si]));
                    float wg = svgf_luma_weight<FAST>(scgl, gl, 1.0f) * common * nw;
                    sgi = sgi + f3(gl, gl * gl, 1.0f) * f3s(wg);
                }
            }
            ox += 1;
            if (ox == 3) { ox = -3; oy += 1; if (oy == 3) break; }
        }
        { float m1 = sdi.x / sdi.z, m2 = sdi.y / sdi.z; di_var = fabs_(m2 - m1 * m1) * 4.0f; }
        { float m1 = sgi.x / sgi.z, m2 = sgi.y / sgi.z; gi_var = fabs_(m2 - m1 * m1) * 4.0f; }
    }
    di_var = rmax(di_var, 0.0f); gi_var = rmax(gi_var, 0.0f);
    cam.di_diff_stash[i] = f4(xyz(cdi), di_var);
    cam.gi_diff_stash[i] = f4(xyz(cgi), gi_var);
}

// K22 frame_denoising::wavelet (frame_denoising.rs:220-361): 3x3 à-trous, DI and GI together.
// Per tap: one (normal, depth) float4 + the two signal float4s; the depth ramp and normal^64 factors are
// evaluated once and shared by both signals, taps whose shared factor is 0 are skipped (weight cannot be > 0).
#ifndef ST_WAVELET_MIN_BLOCKS
#define ST_WAVELET_MIN_BLOCKS 10
#endif
// PAIR_IN: the two signals arrive interleaved, {DI, GI} = one 32-byte record per pixel (`pair_in`, written by the previous iteration
// through `pair_out`), so that a jittered tap of the wide strides is one full sector and one 256-bit load instead of two half-used
// sectors; `pair_out` != nullptr writes that layout.  Values and arithmetic are those of the planar layout.
template <bool BATCHED, bool FAST, bool PAIR_IN>
__global__ void __launch_bounds__(ST_BLOCK, ST_WAVELET_MIN_BLOCKS) k_denoise_wavelet(VPARAMS, int cur, u32 frame, u32 stride, float strength,
                                                              const float4* __restrict__ di_in, float4* __restrict__ di_out,
                                                              const float4* __restrict__ gi_in, float4* __restrict__ gi_out,
                                                              const float4* __restrict__ pair_in, float4* __restrict__ pair_out) {
    VIEW; VIEW_ARENA(di_in); VIEW_ARENA(di_out); VIEW_ARENA(gi_in); VIEW_ARENA(gi_out);
    pair_in = pair_ptr<BATCHED>(pair_in, view); pair_out = pair_ptr<BATCHED>(pair_out, view);
    Px p = pixel_full(cam);
    if (!p.in) return;
    size_t i = pix(cam, p.x, p.y);
    const float4* __restrict__ snd = cam.surface_nd;
    float4 cnd = snd[i];
    float4 cdi, cgi;
    if (PAIR_IN) { F8 c = ld8(pair_in + 2 * i); cdi = c.a; cgi = c.b; } else cdi = di_in[i];
    float3 cdc = xyz(cdi); float cdv = cdi.w;
    if (cnd.w == 0.0f) { if (pair_out) pair_out[2 * i] = f4(cdc, cdv); else di_out[i] = f4(cdc, cdv); return; }
    float4 bn = blue_noise(sc, p.x, p.y, frame);
    if (!PAIR_IN) cgi = gi_in[i];
    float3 cgc = xyz(cgi); float cgv = cgi.w;
    float3 cn = xyz(cnd);
    float scdl = sv_sqrt<FAST>(sv_luma<FAST>(cdc)), scgl = sv_sqrt<FAST>(sv_luma<FAST>(cgc));
    float ls_di = lerpc(2.5f, 0.5f, sv_sqrt<FAST>(cdv));
    float ls_gi = lerpc(1.0f, 0.0f, sv_sqrt<FAST>(cgv));
    float depth_sigma = 0.33f / strength;   // same for DI and GI (frame_denoising.rs:264,267)
    float2 jf = (f2(bn.z, bn.w) - f2(0.5f, 0.5f)) * ((float)stride - 1.0f) * 0.5f;
    int jx = to_i32_sat(jf.x), jy = to_i32_sat(jf.y);
    float sdw = 1.0f; float3 sdc = cdc; float sdv = cdv;
    float sgw = 1.0f; float3 sgc = cgc; float sgv = cgv;
#pragma unroll
    for (int oy = -1; oy <= 1; oy++) {
#pragma unroll
        for (int ox = -1; ox <= 1; ox++) {
            if (ox == 0 && oy == 0) continue;
            int sx = (int)p.x + jx + ox * (int)stride, sy = (int)p.y + jy + oy * (int)stride;
            if (!cam_contains_i(cam.curr, sx, sy)) continue;
            size_t si = pix(cam, (u32)sx, (u32)sy);
            float4 nds = snd[si];
            if (nds.w == 0.0f) continue;
            float dw = svgf_depth_weight<FAST>(cnd.w, nds.w, depth_sigma);
            float nw = svgf_normal_weight<FAST>(cn, xyz(nds));
            if (dw == 0.0f || nw == 0.0f) continue;
            float dnw = dw * nw;
            float4 sdi, sgi;
            if (PAIR_IN) { F8 t = ld8(pair_in + 2 * si); sdi = t.a; sgi = t.b; } else { sdi = di_in[si]; sgi = gi_in[si]; }
            if (FAST) {
                float wd = svgf_luma_weight<true>(scdl, sv_luma<true>(xyz(sdi)), ls_di) * dnw;
                if (wd > 0.0f) { sdw += wd; sdc = f3(__fmaf_rn(wd, sdi.x, sdc.x), __fmaf_rn(wd, sdi.y, sdc.y), __fmaf_rn(wd, sdi.z, sdc.z)); sdv = __fmaf_rn(wd * wd, sdi.w, sdv); }
                float wg = svgf_luma_weight<true>(scgl, sv_luma<true>(xyz(sgi)), ls_gi) * dnw;
                if (wg > 0.0f) { sgw += wg; sgc = f3(__fmaf_rn(wg, sgi.x, sgc.x), __fmaf_rn(wg, sgi.y, sgc.y), __fmaf_rn(wg, sgi.z, sgc.z)); sgv = __fmaf_rn(wg * wg, sgi.w, sgv); }
            } else {
                float wd = svgf_luma_weight<false>(scdl, luma(xyz(sdi)), ls_di) * dw * nw;
                if (wd > 0.0f) { sdw += wd; sdc = sdc + wd * xyz(sdi); sdv += sq(wd) * sdi.w; }
                float wg = svgf_luma_weight<false>(scgl, luma(xyz(sgi)), ls_gi) * dw * nw;
                if (wg > 0.0f) { sgw += wg; sgc = sgc + wg * xyz(sgi); sgv += sq(wg) * sgi.w; }
            }
        }
    }
    float4 odi, ogi;
    if (FAST) {
        float rd = sfu_rcp(sdw), rg = sfu_rcp(sgw);
        odi = f4(sdc * rd, sdv * (rd * rd));
        ogi = f4(sgc * rg, sgv * (rg * rg));
    } else {
        odi = f4(sdc / sdw, sdv / (sdw * sdw));
        ogi = f4(sgc / sgw, sgv / (sgw * sgw));
    }
    if (pair_out) st8(pair_out + 2 * i, odi, ogi);
    else { di_out[i] = odi; gi_out[i] = ogi; }
}

// ---------------------------------------------------------------------------------------------
// K22, tile-staged variant: the (TW+2·HL) x (TH+2·HL) pixel neighbourhood of a TW x TH output tile is
// brought into shared memory by three TMA tensor copies (surface_nd, DI colours, GI colours; one elected
// thread, one mbarrier), out-of-frame texels arrive as zeros (= the reference's `contains` test, because a
// zero depth skips the tap), and the 3x3 à-trous taps become LDS.128 at compile-time offsets.  HL = S + J,
// J = the largest |jitter| the blue-noise term can produce for stride S (0 for S <= 4, 1 for 8, 3 for 16).
// Same taps, same order, same arithmetic as k_denoise_wavelet: the two kernels are bit-identical in both
// arithmetic flavours (tests/test_gpu_parity.py::test_tiled_wavelet_matches_gather).
// ---------------------------------------------------------------------------------------------
ST_DEV u32 smem_addr(const void* p) { return (u32)__cvta_generic_to_shared(p); }
ST_DEV void mbar_init(u32 bar, u32 count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory"); }
ST_DEV void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
ST_DEV void mbar_expect_tx(u32 bar, u32 bytes) { asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory"); }
ST_DEV bool mbar_try_wait(u32 bar, u32 parity) {
    u32 ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0u;
}
ST_DEV void tma_load_2d(u32 dst, const CUtensorMap* tm, int c0, int c1, u32 bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(dst), "l"(reinterpret_cast<unsigned long long>(tm)), "r"(c0), "r"(c1), "r"(bar) : "memory");
}

// Per-centre state of K22: the terms of frame_denoising::sample_weight (frame_denoising.rs:363-392) that depend on the centre
// pixel only are evaluated once (1 / leeway of the depth ramp, sqrt of the centre luminances, the luminance sigmas); `geometry`
// is the part of a tap's weight shared by the DI and the GI signal, `add` the per-signal luminance term and the accumulation.
// Same expressions, same order as k_denoise_wavelet (both arithmetic flavours): bit-identical results.
template <bool FAST> struct WaveletCentre {
    float3 n; float depth, leeway, rcp_leeway, scdl, scgl, ls_di, ls_gi;
    float sdw; float3 sdc; float sdv; float sgw; float3 sgc; float sgv;
    ST_DEV void init(float4 cnd, float4 cdi, float4 cgi, float depth_sigma) {
        n = xyz(cnd); depth = cnd.w; leeway = cnd.w * depth_sigma; rcp_leeway = FAST ? sfu_rcp(leeway) : 0.0f;
        float3 cdc = xyz(cdi), cgc = xyz(cgi);
        scdl = sv_sqrt<FAST>(sv_luma<FAST>(cdc)); scgl = sv_sqrt<FAST>(sv_luma<FAST>(cgc));
        ls_di = lerpc(2.5f, 0.5f, sv_sqrt<FAST>(cdi.w)); ls_gi = lerpc(1.0f, 0.0f, sv_sqrt<FAST>(cgi.w));
        sdw = 1.0f; sdc = cdc; sdv = cdi.w; sgw = 1.0f; sgc = cgc; sgv = cgi.w;
    }
    // depth ramp and normal^64 of one tap (svgf_depth_weight / svgf_normal_weight); false = the tap cannot contribute
    ST_DEV bool geometry(float4 nds, float* dw, float* nw) const {
        float diff = fabs_(nds.w - depth);
        if (diff >= leeway) return false;
        *dw = FAST ? __fmaf_rn(-diff, rcp_leeway, 1.0f) : 1.0f - diff / leeway;
        *nw = svgf_normal_weight<FAST>(n, xyz(nds));
        return !(*dw == 0.0f || *nw == 0.0f);
    }
    ST_DEV void add(float dw, float nw, float4 sdi, float4 sgi) {
        if (FAST) {
            float dnw = dw * nw;
            float wd = svgf_luma_weight<true>(scdl, sv_luma<true>(xyz(sdi)), ls_di) * dnw;
            if (wd > 0.0f) { sdw += wd; sdc = f3(__fmaf_rn(wd, sdi.x, sdc.x), __fmaf_rn(wd, sdi.y, sdc.y), __fmaf_rn(wd, sdi.z, sdc.z)); sdv = __fmaf_rn(wd * wd, sdi.w, sdv); }
            float wg = svgf_luma_weight<true>(scgl, sv_luma<true>(xyz(sgi)), ls_gi) * dnw;
            if (wg > 0.0f) { sgw += wg; sgc = f3(__fmaf_rn(wg, sgi.x, sgc.x), __fmaf_rn(wg, sgi.y, sgc.y), __fmaf_rn(wg, sgi.z, sgc.z)); sgv = __fmaf_rn(wg * wg, sgi.w, sgv); }
        } else {
            float wd = svgf_luma_weight<false>(scdl, luma(xyz(sdi)), ls_di) * dw * nw;
            if (wd > 0.0f) { sdw += wd; sdc = sdc + wd * xyz(sdi); sdv += sq(wd) * sdi.w; }
            float wg = svgf_luma_weight<false>(scgl, luma(xyz(sgi)), ls_gi) * dw * nw;
            if (wg > 0.0f) { sgw += wg; sgc = sgc + wg * xyz(sgi); sgv += sq(wg) * sgi.w; }
        }
    }
    ST_DEV void store(float4* __restrict__ di_out, float4* __restrict__ gi_out, float4* __restrict__ pair_out, size_t i) const {
        float4 odi, ogi;
        if (FAST) {
            float rd = sfu_rcp(sdw), rg = sfu_rcp(sgw);
            odi = f4(sdc * rd, sdv * (rd * rd));
            ogi = f4(sgc * rg, sgv * (rg * rg));
        } else {
            odi = f4(sdc / sdw, sdv / (sdw * sdw));
            ogi = f4(sgc / sgw, sgv / (sgw * sgw));
        }
        if (pair_out) st8(pair_out + 2 * i, odi, ogi);   // interleaved {DI, GI} record for the wide-stride iterations (see k_denoise_wavelet)
        else { di_out[i] = odi; gi_out[i] = ogi; }
    }
};

template <int S, int J, int TW, int TH> struct WaveletTile {
    static constexpr int HL = S + J, BW = TW + 2 * HL, BH = TH + 2 * HL;
    static constexpr u32 BOX_BYTES = (u32)(BW * BH * 16);
    static constexpr u32 PLANE = (BOX_BYTES + 127u) & ~127u;
    static constexpr u32 SMEM = 3u * PLANE + 128u;   // + slack to align the first plane to 128 B
};

#ifndef ST_WAVELET_TILED_MINB
#define ST_WAVELET_TILED_MINB 1
#endif
template <bool FAST, int S, int J, int TW, int TH>
__global__ void __launch_bounds__(TW * TH, (TW * TH <= 256 && S <= 8) ? ST_WAVELET_TILED_MINB : 1) k_denoise_wavelet_tiled(KPARAMS, u32 frame, float strength,
                                                                   const __grid_constant__ CUtensorMap tm_nd, const __grid_constant__ CUtensorMap tm_di,
                                                                   const __grid_constant__ CUtensorMap tm_gi,
                                                                   float4* __restrict__ di_out, float4* __restrict__ gi_out, float4* __restrict__ pair_out,
                                                                   u32* __restrict__ errors) {
    typedef WaveletTile<S, J, TW, TH> T;
    extern __shared__ unsigned char s_raw[];
    __shared__ __align__(8) unsigned long long s_bar;
    const int tx = (int)threadIdx.x % TW, ty = (int)threadIdx.x / TW;
    const int x0 = (int)blockIdx.x * TW, y0 = cam.y0 + (int)blockIdx.y * TH;
    const u32 bar = smem_addr(&s_bar);
    const u32 raw = smem_addr(s_raw);
    const u32 base = (raw + 127u) & ~127u;
    if (threadIdx.x == 0) { mbar_init(bar, 1u); mbar_fence_init(); }
    __syncthreads();
    if (threadIdx.x == 0) {
        mbar_expect_tx(bar, 3u * T::BOX_BYTES);   // tensor coordinates: x in 8-byte elements (see wavelet_tensor_map), y in rows
        tma_load_2d(base, &tm_nd, (x0 - T::HL) * 2, y0 - T::HL, bar);
        tma_load_2d(base + T::PLANE, &tm_di, (x0 - T::HL) * 2, y0 - T::HL, bar);
        tma_load_2d(base + 2u * T::PLANE, &tm_gi, (x0 - T::HL) * 2, y0 - T::HL, bar);
    }
    const u32 px = (u32)(x0 + tx), py = (u32)(y0 + ty);
    const bool in = px < (u32)cam.w && py < (u32)cam.y1;
    int jo = 0;
    if (J > 0 && in) {   // the jitter only needs the blue-noise texel: fetched while the tile is in flight
        float4 bn = blue_noise(sc, px, py, frame);
        float2 jf = (f2(bn.z, bn.w) - f2(0.5f, 0.5f)) * ((float)S - 1.0f) * 0.5f;
        jo = to_i32_sat(jf.y) * T::BW + to_i32_sat(jf.x);
    }
    {   // every thread waits (the CTA's shared memory must stay allocated until the copies have landed)
        bool done = false;
        for (u32 spin = 0; spin < (1u << 20) && !done; spin++) done = mbar_try_wait(bar, 0u);
        if (!done) { if (threadIdx.x == 0) atomicAdd(errors, 1u); return; }
    }
    if (!in) return;
    const float4* __restrict__ t_nd = reinterpret_cast<const float4*>(s_raw + (base - raw));
    const float4* __restrict__ t_di = reinterpret_cast<const float4*>(s_raw + (base - raw) + T::PLANE);
    const float4* __restrict__ t_gi = reinterpret_cast<const float4*>(s_raw + (base - raw) + 2u * T::PLANE);
    const int c = (ty + T::HL) * T::BW + (tx + T::HL);
    const size_t i = pix(cam, px, py);
    float4 cnd = t_nd[c];
    float4 cdi = t_di[c];
    if (cnd.w == 0.0f) { if (pair_out) pair_out[2 * i] = f4(xyz(cdi), cdi.w); else di_out[i] = f4(xyz(cdi), cdi.w); return; }   // sky: DI passes through, GI is not written (frame_denoising.rs:248-254)
    WaveletCentre<FAST> ctr;
    ctr.init(cnd, cdi, t_gi[c], 0.33f / strength);   // depth sigma is the same for DI and GI (frame_denoising.rs:264,267)
    const int cj = c + jo;
#pragma unroll
    for (int oy = -1; oy <= 1; oy++) {
#pragma unroll
        for (int ox = -1; ox <= 1; ox++) {
            if (ox == 0 && oy == 0) continue;
            const int k = cj + oy * S * T::BW + ox * S;
            float4 nds = t_nd[k];
            if (nds.w == 0.0f) continue;   // sky, or outside the frame (zero-filled by the tensor copy)
            float dw, nw;
            if (!ctr.geometry(nds, &dw, &nw)) continue;
            ctr.add(dw, nw, t_di[k], t_gi[k]);
        }
    }
    ctr.store(di_out, gi_out, pair_out, i);
}

// R2 frame_composition::fs (frame_composition.rs:19-82), linear HDR out
template <bool BATCHED>
__global__ void __launch_bounds__(ST_BLOCK) k_composition(VPARAMS, int cur, u32 mode, const float4* __restrict__ di_diff, const float4* __restrict__ gi_diff) {
    VIEW; VIEW_ARENA(di_diff); VIEW_ARENA(gi_diff);
    Px p = pixel_full(cam);
    if (!p.in) return;
    size_t i = pix(cam, p.x, p.y);
    float3 color;
    if (mode == 0u) {
        GBuf g = gbuf_unpack(sc, cam.prim_gbuffer_d0[cur][i], cam.prim_gbuffer_d1[cur][i]);
        float3 dd = xyz(di_diff[i]), ds = xyz(cam.di_spec_samples[i]), gd = xyz(gi_diff[i]), gs = xyz(cam.gi_spec_samples[i]);
        if (g.depth != 0.0f) color = g.emissive + (dd + gd) * xyz(g.base_color) + ds + gs;
        else color = dd;
    } else if (mode == 1u) color = xyz(di_diff[i]);
    else if (mode == 2u) color = xyz(cam.di_spec_samples[i]);
    else if (mode == 3u) color = xyz(gi_diff[i]);
    else if (mode == 4u) color = xyz(cam.gi_spec_samples[i]);
    else if (mode == 5u) color = xyz(cam.ref_colors[i]);
    else if (mode == 6u) { float4 c = cam.ref_colors[i]; color = xyz(c) / c.w; }
    else color = f3s(0.f);
    cam.output[i] = f4(color, 1.0f);
}


// One channel of an Rgba8UnormSrgb render-target store (the reference's default CameraViewport::format,
// strolle/src/camera.rs:177-185): clamp to [0,1], sRGB OETF, round to nearest.
ST_DEV u32 srgb8_encode(float v) {
    float x = sat(v);
    float e = (x <= 0.0031308f) ? 12.92f * x : 1.055f * pow_det(x, 1.0f / 2.4f) - 0.055f;
    return to_u32_sat(sat(e) * 255.0f + 0.5f);
}

// Store of rows [y0, y1) of the composed frame into a surface of format FMT (CameraViewport::format): pixel (x, y) goes to
// dst + y * pitch + x * bytes per pixel, one aligned store per pixel; nothing else of the surface is touched (LoadOp::Load).
// RGBA32F copies `output`; RGBA16F converts each channel with round-to-nearest-even (what a store to an Rgba16Float target does),
// alpha 1.0; RGBA8 is the sRGB encode above.
template <bool BATCHED, int FMT>
__global__ void __launch_bounds__(ST_BLOCK) k_output_store(VPARAMS) {
    VIEW;
    char* __restrict__ dst = view.dst; const size_t pitch = view.pitch;
    Px p = pixel_full(cam);
    if (!p.in) return;
    float4 c = cam.output[pix(cam, p.x, p.y)];
    char* row = dst + (size_t)p.y * pitch;
    if (FMT == OUT_RGBA32F) {
        reinterpret_cast<float4*>(row)[p.x] = c;
    } else if (FMT == OUT_RGBA16F) {
        const u32 r = __half_as_ushort(__float2half_rn(c.x)), g = __half_as_ushort(__float2half_rn(c.y)), b = __half_as_ushort(__float2half_rn(c.z));
        reinterpret_cast<uint2*>(row)[p.x] = make_uint2(r | (g << 16), b | (0x3C00u << 16));
    } else {
        reinterpret_cast<uchar4*>(row)[p.x] = make_uchar4((unsigned char)srgb8_encode(c.x), (unsigned char)srgb8_encode(c.y), (unsigned char)srgb8_encode(c.z), 255);
    }
}

// K1 ref_tracing::main (ref_tracing.rs:4-60)
template <bool BATCHED>
__global__ void __launch_bounds__(ST_BLOCK) k_ref_tracing(VPARAMS, u32 depth) {
    VIEW;
    ST_TRACE_STACK();
    Px p = pixel_full(cam);
    if (!p.in) return;
    size_t idx = screen_idx(cam, p.x, p.y);
    Ray ray;
    if (depth == 0u) ray = cam_ray(cam.curr, p.x, p.y);
    else {
        float4 d0 = cam.ref_rays[3 * idx], d1 = cam.ref_rays[3 * idx + 1];
        if (all_zero(d1)) return;
        ray = ray_make(xyz(d0), xyz(d1));
    }
    TriHit h = trace_closest(ray, sc, stk);
    float4 h0, h1; trihit_pack(h, &h0, &h1);
    cam.ref_hits[2 * idx] = h0; cam.ref_hits[2 * idx + 1] = h1;
}

// K2 ref_shading::main (ref_shading.rs:4-177)
template <bool BATCHED>
__global__ void __launch_bounds__(ST_BLOCK) k_ref_shading(VPARAMS, u32 seed, u32 depth) {
    VIEW;
    ST_TRACE_STACK();
    Px p = pixel_full(cam);
    if (!p.in) return;
    size_t idx = screen_idx(cam, p.x, p.y);
    Rng rng = rng_make(seed, p.x, p.y);
    float4* rays = cam.ref_rays;
    if (depth == 255u) {
        size_t i = pix(cam, p.x, p.y);
        float4 prev = cam_is_eq(cam.curr, cam.prev) ? cam.ref_colors[i] : f4zero();
        cam.ref_colors[i] = prev + f4(xyz(rays[3 * idx + 2]), 1.0f);
        return;
    }
    Ray ray; float3 color, thr;
    if (depth == 0u) { ray = cam_ray(cam.curr, p.x, p.y); color = f3s(0.f); thr = f3s(1.0f); }
    else {
        float4 d0 = rays[3 * idx], d1 = rays[3 * idx + 1], d2 = rays[3 * idx + 2];
        if (all_zero(d1)) return;   // dead path: explicit no-op (the reference reaches the same state through 0 * x)
        ray = ray_make(xyz(d0), xyz(d1)); color = xyz(d2); thr = f3(d0.w, d1.w, d2.w);
    }
    TriHit th = trihit_unpack(cam.ref_hits[2 * idx], cam.ref_hits[2 * idx + 1]);
    if (!trihit_some(th)) {
        color = color + thr * atmosphere_sample(sc, world_sun_dir(sc.world), ray.d);
        rays[3 * idx] = f4zero(); rays[3 * idx + 1] = f4zero(); rays[3 * idx + 2] = f4(color, 0.0f);
        return;
    }
    GpuMaterial m = sc.materials[th.material_id];
    if (depth > 0u) m.roughness = rmax(m.roughness, 0.75f * 0.75f);
    Hit hit;
    hit.point = th.point + th.normal * 0.01f; hit.origin = ray.o; hit.dir = ray.d;
    hit.g.base_color = mat_base_color(sc, m, th.uv); hit.g.normal = th.normal; hit.g.metallic = m.metallic; hit.g.emissive = mat_emissive(sc, m, th.uv);
    hit.g.roughness = m.roughness; hit.g.reflectance = m.reflectance; hit.g.depth = 0.0f;
    color = color + thr * hit.g.emissive;
    if (sc.world.light_count > 0u) {
        u32 lid = rng_u32(rng) % sc.world.light_count;
        float lpdf = 1.0f / (float)sc.world.light_count;
        GpuLight light = light_load(sc, lid);
        bool occ = trace_any(light_ray_wnoise(light, rng, hit.point), sc, stk);
        if (!occ) color = color + thr * lightrad_sum(light_radiance(light, hit)) / lpdf;
    }
    BrdfS rs = brdf_layered_sample(hit.g, rng, -hit.dir);
    if (rs.pdf == 0.0f) { rays[3 * idx] = f4zero(); rays[3 * idx + 1] = f4zero(); return; }
    thr = thr * dot(rs.dir, hit.g.normal);
    thr = thr * (rs.radiance / rs.pdf);
    rays[3 * idx] = f4(hit.point, thr.x);
    rays[3 * idx + 1] = f4(rs.dir, thr.y);
    rays[3 * idx + 2] = f4(color, thr.z);
}

// K3 bvh_heatmap::main (bvh_heatmap.rs:4-77)
template <bool BATCHED>
__global__ void __launch_bounds__(ST_BLOCK) k_bvh_heatmap(VPARAMS) {
    VIEW;
    ST_TRACE_STACK();
    Px p = pixel_full(cam);
    if (!p.in) return;
    u32 used = 0u;
    trace_closest<true>(cam_ray(cam.curr, p.x, p.y), sc, stk, &used);
    float progress = (float)used / 8192.0f;
    const float3 cols[4] = {f3(0.f, 0.f, 1.f), f3(0.f, 1.f, 0.f), f3(1.f, 0.f, 0.f), f3(0.f, 0.f, 0.f)};
    float3 c = cols[3];
    if (progress <= 0.0f) c = cols[0];
    else {
        float step = 1.0f / (4.0f - 1.0f);
        bool done = false;
        for (int k = 0; k < 3 && !done; k++) {
            float mn = step * (float)k, mx = step * ((float)k + 1.0f);
            if (progress >= mn && progress <= mx) { float rhs = (progress - mn) / step; float lhs = 1.0f - rhs; c = lhs * cols[k] + rhs * cols[k + 1]; done = true; }
        }
    }
    cam.ref_colors[pix(cam, p.x, p.y)] = f4(c, 1.0f);
}

// ---------------------------------------------------------------------------------------------
// Ray-stream kernels (the K1/K8/K16 shape without the screen): 8 floats per ray
// (origin.xyz, len, dir.xyz, pad) in, packed hits / occlusion flags out.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(ST_BLOCK) k_trace_stream_closest(const __grid_constant__ SceneDev sc, const float4* __restrict__ rays, long n, float4* __restrict__ out) {
    ST_TRACE_STACK();
    long i = (long)blockIdx.x * ST_BLOCK + threadIdx.x;
    if (i >= n) return;
    float4 a = rays[2 * i], b = rays[2 * i + 1];
    u32 used = 0u;
    TriHit h = trace_closest<true>(ray_make(xyz(a), xyz(b)), sc, stk, &used);
    float4 h0, h1; trihit_pack(h, &h0, &h1);
    out[3 * i] = h0; out[3 * i + 1] = h1; out[3 * i + 2] = f4(h.t, bitsf(h.triangle_id), bitsf(h.material_id), (float)used);
}
__global__ void __launch_bounds__(ST_BLOCK) k_trace_stream_any(const __grid_constant__ SceneDev sc, const float4* __restrict__ rays, long n, u32* __restrict__ out) {
    ST_TRACE_STACK();
    long i = (long)blockIdx.x * ST_BLOCK + threadIdx.x;
    if (i >= n) return;
    float4 a = rays[2 * i], b = rays[2 * i + 1];
    out[i] = trace_any(ray_make(xyz(a), xyz(b), a.w), sc, stk) ? 1u : 0u;
}
// elementary-function test hook
__global__ void k_math(int op, const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ out, long n) {
    long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float r = 0.f;
    switch (op) {
        case 0: r = sin_det(a[i]); break; case 1: r = cos_det(a[i]); break; case 2: r = acos_det(a[i]); break;
        case 3: r = atan2_det(a[i], b[i]); break; case 4: r = exp_det(a[i]); break; case 5: r = pow_det(a[i], b[i]); break;
        case 6: r = acos_approx_glam(a[i]); break;
    }
    out[i] = r;
}

// derived tables: packed gamma colour per material, byte -> linear table for GBufferEntry::unpack
__global__ void k_material_derive(const GpuMaterial* __restrict__ mats, u32 n, u32* __restrict__ packed) {
    u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) packed[i] = gbuf_pack_color(mats[i].base_color);
}
__global__ void k_srgb_lut(float* __restrict__ lut) {   // sRGB electro-optical transfer function per byte
    u32 i = threadIdx.x;
    float c = (float)i / 255.0f;
    lut[i] = (c <= 0.04045f) ? c / 12.92f : pow_det((c + 0.055f) / 1.055f, 2.4f);
}
__global__ void k_unpack_lut(float* __restrict__ lut) {
    u32 i = threadIdx.x;   // 256 threads
    lut[i] = pow_det((float)i / 255.0f, 2.2f);
    lut[256u + i] = pow_det((float)i / 63.0f, 2.2f);
}

// ---------------------------------------------------------------------------------------------
// Atmosphere LUT generation (strolle-shaders/src/atmosphere/*.rs; Hillaire 2020).  Runs once /
// on sun change (90 k texels) — outside the per-frame hot path, kept on the GPU so that the
// product needs no CPU fallback for it.  Rgba16Float storage == f32 rounded to binary16.
// ---------------------------------------------------------------------------------------------
ST_DEV float round_f16(float f) { return __half2float(__float2half_rn(f)); }
ST_DEV void atm_scattering(float3 pos, float3* rayleigh, float* mie, float3* ext) {   // atmosphere/utils.rs:3-27
    float alt_km = (len(pos) - ST_ATM_GROUND) * 1000.0f;
    float rd = exp_det(-alt_km / 8.0f);
    float md = exp_det(-alt_km / 1.2f);
    float3 rs = f3(5.802f, 13.558f, 33.1f) * rd;
    float ms = 3.996f * md;
    float ma = 4.4f * md;
    float3 oz = f3(0.650f, 1.881f, 0.085f) * rmax(1.0f - fabs_(alt_km - 25.0f) / 15.0f, 0.0f);
    *rayleigh = rs; *mie = ms;
    *ext = ((rs + f3s(ms)) + f3s(ma)) + oz;   // RAYLEIGH_ABSORPTION_BASE == 0.0 contributes nothing (quirk C-18)
}
ST_DEV float atm_mie_phase(float c) {
    const float G = 0.8f; const float SCALE = 3.0f / (8.0f * kPi);
    float num = (1.0f - G * G) * (1.0f + c * c);
    float den = (2.0f + G * G) * pow_det(1.0f + G * G - 2.0f * G * c, 1.5f);
    return SCALE * num / den;
}
ST_DEV float atm_rayleigh_phase(float c) { const float K = 3.0f / (16.0f * kPi); return K * (1.0f + c * c); }
ST_DEV float3 exp3(float3 v) { return f3(exp_det(v.x), exp_det(v.y), exp_det(v.z)); }
ST_DEV float3 atm_transmittance(float3 pos, float3 sun_dir) {   // generate_transmittance_lut.rs:29-59
    if (ray_sphere(ray_make(pos, sun_dir), ST_ATM_GROUND) > 0.0f) return f3s(0.f);
    float adist = ray_sphere(ray_make(pos, sun_dir), ST_ATM_TOP);
    float t = 0.0f; float3 tr = f3s(1.0f);
    for (float i = 0.0f; i < 40.0f; i += 1.0f) {
        float nt = ((i + 0.3f) / 40.0f) * adist;
        float dt = nt - t; t = nt;
        float3 rs, ext; float ms; atm_scattering(pos + t * sun_dir, &rs, &ms, &ext);
        tr = tr * exp3(-dt * ext);
    }
    return tr;
}
__global__ void k_atm_transmittance(float4* __restrict__ out) {   // 256x64
    int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= 256 || y >= 64) return;
    float2 uv = f2((float)x, (float)y) / f2(256.0f, 64.0f);
    float sct = 2.0f * uv.x - 1.0f;
    float sth = acos_det(rclamp(sct, -1.0f, 1.0f));
    float height = lerpc(ST_ATM_GROUND, ST_ATM_TOP, uv.y);
    float3 v = atm_transmittance(f3(0.0f, height, 0.0f), norm(f3(0.0f, sct, -sin_det(sth))));
    out[y * 256 + x] = f4(round_f16(v.x), round_f16(v.y), round_f16(v.z), 1.0f);
}
__global__ void k_atm_sun_color(float4* __restrict__ out, GpuWorld world) {   // strolle/src/lights.rs:84-99
    float3 sd = world_sun_dir(world);
    float3 c = atm_transmittance(atm_view_pos(), sd);
    c = c * 20.0f * 5.0f;
    float3 pos = sd * 1000.0f;
    out[0] = f4(pos, 25.0f); out[1] = f4(c, finf());
}
__global__ void k_atm_scattering(const float4* __restrict__ tl, float4* __restrict__ out) {   // 32x32, generate_scattering_lut.rs
    int x = threadIdx.x, y = blockIdx.x;
    float2 uv = f2((float)x, (float)y) / f2(32.0f, 32.0f);
    float sct = 2.0f * uv.x - 1.0f;
    float sth = acos_det(rclamp(sct, -1.0f, 1.0f));
    float height = lerpc(ST_ATM_GROUND, ST_ATM_TOP, rmax(uv.y, 0.01f));
    float3 pos = f3(0.0f, height, 0.0f);
    float3 sun_dir = norm(f3(0.0f, sct, -sin_det(sth)));
    float3 lum_total = f3s(0.f), fms = f3s(0.f);
    const int S = 8;
    float inv_samples = 1.0f / (float)(S * S);
    for (int i = 0; i < S; i++) for (int j = 0; j < S; j++) {
        float theta = kPi * ((float)i + 0.5f) / (float)S;
        float phi = acos_det(rclamp(1.0f - 2.0f * ((float)j + 0.5f) / (float)S, -1.0f, 1.0f));
        float sph, cph, sth2, cth2; sincos_det(phi, &sph, &cph); sincos_det(theta, &sth2, &cth2);
        float3 rd = f3(sph * sth2, cph, sph * cth2);
        float adist = ray_sphere(ray_make(pos, rd), ST_ATM_TOP);
        float gdist = ray_sphere(ray_make(pos, rd), ST_ATM_GROUND);
        float t_max = (gdist > 0.0f) ? gdist : adist;
        float ct = dot(rd, sun_dir);
        float mp = atm_mie_phase(ct), rp = atm_rayleigh_phase(-ct);
        float3 lum = f3s(0.f), lf = f3s(0.f), tr = f3s(1.0f);
        float t = 0.0f;
        for (float s = 0.0f; s < 20.0f; s += 1.0f) {
            float nt = ((s + 0.3f) / 20.0f) * t_max;
            float dt = nt - t; t = nt;
            float3 np = pos + t * rd;
            float3 rs, ext; float ms; atm_scattering(np, &rs, &ms, &ext);
            float3 st_ = exp3(-dt * ext);
            float3 snp = rs + f3s(ms);
            float3 sf = (snp - snp * st_) / ext;
            lf = lf + tr * sf;
            float3 sun_t = atm_lut(tl, 256, 64, np, sun_dir);
            float3 ri = rs * rp;
            float mi = ms * mp;
            float3 ins = (ri + f3s(mi)) * sun_t;
            float3 si = (ins - ins * st_) / ext;
            lum = lum + si * tr;
            tr = tr * st_;
        }
        if (gdist > 0.0f) {
            float3 hp = pos + gdist * rd;
            if (dot(pos, sun_dir) > 0.0f) {
                hp = norm(hp) * ST_ATM_GROUND;
                lum = lum + tr * f3s(0.25f) * atm_lut(tl, 256, 64, hp, sun_dir);
            }
        }
        fms = fms + lf * inv_samples;
        lum_total = lum_total + lum * inv_samples;
    }
    float3 o = lum_total / (f3s(1.0f) - fms);
    out[y * 32 + x] = f4(round_f16(o.x), round_f16(o.y), round_f16(o.z), 1.0f);
}
__global__ void k_atm_sky(const float4* __restrict__ tl, const float4* __restrict__ sl, float sun_altitude, float4* __restrict__ out) {   // 256x256, generate_sky_lut.rs
    int x = threadIdx.x, y = blockIdx.x;
    float2 uv = f2((float)x, (float)y) / f2(256.0f, 256.0f);
    float azimuth = (uv.x - 0.5f) * 2.0f * kPi;
    float v;
    if (uv.y < 0.5f) { float c = 1.0f - 2.0f * uv.y; v = -c * c; }
    else { float c = uv.y * 2.0f - 1.0f; v = c * c; }
    float3 vp = atm_view_pos();
    float height = len(vp);
    float horizon;
    { float t = sq(height) - sq(ST_ATM_GROUND); t = sqrtf(t) / height; horizon = acos_det(rclamp(t, -1.0f, 1.0f)) - 0.5f * kPi; }
    float altitude = v * 0.5f * kPi - horizon;
    float sa, ca, sz, cz; sincos_det(altitude, &sa, &ca); sincos_det(azimuth, &sz, &cz);
    float3 rd = f3(ca * sz, sa, -ca * cz);
    float sal = fmodf(sun_altitude, 2.0f * kPi);
    float ss, cs_; sincos_det(sal, &ss, &cs_);
    float3 sun_dir = (sal < 0.5f * kPi) ? f3(0.0f, ss, -cs_) : f3(0.0f, ss, cs_);
    float adist = ray_sphere(ray_make(vp, rd), ST_ATM_TOP);
    float gdist = ray_sphere(ray_make(vp, rd), ST_ATM_GROUND);
    float t_max = (gdist < 0.0f) ? adist : gdist;
    float ct = dot(rd, sun_dir);
    float mp = atm_mie_phase(ct), rp = atm_rayleigh_phase(-ct);
    float3 lum = f3s(0.f), tr = f3s(1.0f);
    float t = 0.0f;
    for (float i = 0.0f; i < 32.0f; i += 1.0f) {
        float nt = ((i + 0.3f) / 32.0f) * t_max;
        float dt = nt - t; t = nt;
        float3 np = vp + t * rd;
        float3 rs, ext; float ms; atm_scattering(np, &rs, &ms, &ext);
        float3 st_ = exp3(-dt * ext);
        float3 sun_t = atm_lut(tl, 256, 64, np, sun_dir);
        float3 psi = atm_lut(sl, 32, 32, np, sun_dir);
        float3 ri = rs * (rp * sun_t + psi);
        float3 mi = ms * (mp * sun_t + psi);
        float3 ins = ri + mi;
        float3 si = (ins - ins * st_) / ext;
        lum = lum + si * tr;
        tr = tr * st_;
    }
    out[y * 256 + x] = f4(round_f16(lum.x), round_f16(lum.y), round_f16(lum.z), 1.0f);
}

#endif   // ST_EXACT_ONLY

// ---------------------------------------------------------------------------------------------
// Host-side launchers
// ---------------------------------------------------------------------------------------------
static dim3 grid_full(const CameraDev& cam) { return dim3((cam.w + TILE_W - 1) / TILE_W, (cam.y1 - cam.y0 + TILE_H - 1) / TILE_H); }
static dim3 grid_half(const CameraDev& cam) { int hw = 8 * (((cam.w + 7) / 8) / 2); return dim3((hw + TILE_W - 1) / TILE_W, (cam.y1 - cam.y0 + TILE_H - 1) / TILE_H); }
// One launch over the views of `v` (blockIdx.z = view): the single-camera instantiation `one` for one view, the batched `many` otherwise.
template <class K1, class K2, class... A>
static void vlaunch(K1 one, K2 many, dim3 g, const ViewSet& v, cudaStream_t st, const A&... args) {
    if (g.x == 0 || g.y == 0) return;
    g.z = (unsigned)v.size();
    if (v.size() == 1) { ViewBatch<false> b; b.v[0] = v[0]; one<<<g, ST_BLOCK, 0, st>>>(b, args...); return; }
    ViewBatch<true> b;
    std::copy(v.begin(), v.end(), b.v);
    many<<<g, ST_BLOCK, 0, st>>>(b, args...);
}
#define FULL_LAUNCH(kernel, v, st, ...) vlaunch(kernel<false>, kernel<true>, grid_full(v[0].cam), v, st, __VA_ARGS__)
#define HALF_LAUNCH(kernel, v, st, ...) vlaunch(kernel<false>, kernel<true>, grid_half(v[0].cam), v, st, __VA_ARGS__)

void launch_di_sampling(const ViewSet& v, const SceneDev& s, int cur, u32 seed, u32 frame, cudaStream_t st) { FULL_LAUNCH(k_di_sampling, v, st, s, cur, seed, frame); }
void launch_di_temporal(const ViewSet& v, const SceneDev& s, int cur, u32 seed, cudaStream_t st) { FULL_LAUNCH(k_di_temporal, v, st, s, cur, seed); }
void launch_di_spatial_pick(const ViewSet& v, const SceneDev& s, int cur, u32 seed, u32 frame, cudaStream_t st) { HALF_LAUNCH(k_di_spatial_pick, v, st, s, cur, seed, frame); }
void launch_spatial_trace(const ViewSet& v, const SceneDev& s, const float4* d0, const float4* d1, float4* d2, cudaStream_t st) { FULL_LAUNCH(k_spatial_trace, v, st, s, d0, d1, d2); }
void launch_di_spatial_sample(const ViewSet& v, const SceneDev& s, u32 seed, u32 frame, cudaStream_t st) { HALF_LAUNCH(k_di_spatial_sample, v, st, s, seed, frame); }
void launch_di_resolving(const ViewSet& v, const SceneDev& s, int cur, cudaStream_t st) { FULL_LAUNCH(k_di_resolving, v, st, s, cur); }
void launch_gi_reprojection(const ViewSet& v, const SceneDev& s, int cur, cudaStream_t st) { FULL_LAUNCH(k_gi_reprojection, v, st, s, cur); }
void launch_gi_sampling_a(const ViewSet& v, const SceneDev& s, int cur, u32 seed, u32 frame, cudaStream_t st) { HALF_LAUNCH(k_gi_sampling_a, v, st, s, cur, seed, frame); }
void launch_gi_sampling_b(const ViewSet& v, const SceneDev& s, int cur, u32 seed, u32 frame, cudaStream_t st) { HALF_LAUNCH(k_gi_sampling_b, v, st, s, cur, seed, frame); }
void launch_gi_temporal(const ViewSet& v, const SceneDev& s, int cur, u32 seed, u32 frame, int inline_reprojection, cudaStream_t st) { FULL_LAUNCH(k_gi_temporal, v, st, s, cur, seed, frame, inline_reprojection); }
void launch_gi_spatial_pick(const ViewSet& v, const SceneDev& s, int cur, u32 seed, u32 frame, cudaStream_t st) { HALF_LAUNCH(k_gi_spatial_pick, v, st, s, cur, seed, frame); }
void launch_gi_spatial_sample(const ViewSet& v, const SceneDev& s, u32 seed, u32 frame, cudaStream_t st) { HALF_LAUNCH(k_gi_spatial_sample, v, st, s, seed, frame); }
void launch_gi_preview(const ViewSet& v, const SceneDev& s, int cur, u32 seed, u32 nth, const float4* in, float4* out, int mirror_reach, cudaStream_t st) { FULL_LAUNCH(k_gi_preview, v, st, s, cur, seed, nth, in, out, mirror_reach); }
void launch_gi_resolving(const ViewSet& v, const SceneDev& s, int cur, const float4* in, cudaStream_t st) { FULL_LAUNCH(k_gi_resolving, v, st, s, cur, in); }
void launch_di_sample_temporal(const ViewSet& v, const SceneDev& s, int cur, u32 seed_sampling, u32 seed_temporal, u32 frame, cudaStream_t st) { FULL_LAUNCH(k_di_sample_temporal, v, st, s, cur, seed_sampling, seed_temporal, frame); }
void launch_di_spatial_fused(const ViewSet& v, const SceneDev& s, int cur, u32 seed_pick, u32 seed_sample, u32 frame, cudaStream_t st) { HALF_LAUNCH(k_di_spatial_fused, v, st, s, cur, seed_pick, seed_sample, frame); }
void launch_gi_sampling_fused(const ViewSet& v, const SceneDev& s, int cur, u32 seed_a, u32 seed_b, u32 frame, cudaStream_t st) { HALF_LAUNCH(k_gi_sampling_fused, v, st, s, cur, seed_a, seed_b, frame); }
void launch_gi_spatial_fused(const ViewSet& v, const SceneDev& s, int cur, u32 seed_pick, u32 seed_sample, u32 frame, cudaStream_t st) { HALF_LAUNCH(k_gi_spatial_fused, v, st, s, cur, seed_pick, seed_sample, frame); }
void launch_gi_preview_resolve(const ViewSet& v, const SceneDev& s, int cur, u32 seed, const float4* in, const float4* source, cudaStream_t st) { FULL_LAUNCH(k_gi_preview_resolve, v, st, s, cur, seed, in, source); }
#if ST_EXACT_ONLY
void launch_prim_gbuffer(const ViewSet& v, const SceneDev& s, int cur, int with_reprojection, cudaStream_t st) { FULL_LAUNCH(k_prim_gbuffer, v, st, s, cur, with_reprojection); }
void launch_frame_reprojection(const ViewSet& v, const SceneDev& s, int cur, cudaStream_t st) { FULL_LAUNCH(k_frame_reprojection, v, st, s, cur); }
void launch_denoise_reproject(const ViewSet& v, const SceneDev& s, int cur, const float4* pc, const float4* pm, const float4* smp, float4* col, float4* mom, cudaStream_t st) { FULL_LAUNCH(k_denoise_reproject, v, st, s, cur, pc, pm, smp, col, mom); }
void launch_denoise_reproject_pair(const ViewSet& v, const SceneDev& s, int cur, cudaStream_t st) {
    const CameraDev& c = v[0].cam;
    ReprojectSignal di{c.di_diff_prev_colors, c.di_diff_moments[cur ^ 1], c.di_diff_samples, c.di_diff_curr_colors, c.di_diff_moments[cur]};
    ReprojectSignal gi{c.gi_diff_prev_colors, c.gi_diff_moments[cur ^ 1], c.gi_diff_samples, c.gi_diff_curr_colors, c.gi_diff_moments[cur]};
    FULL_LAUNCH(k_denoise_reproject_pair, v, st, s, cur, di, gi);
}
void launch_denoise_variance(const ViewSet& v, const SceneDev& s, int cur, bool fast, cudaStream_t st) {
    const dim3 g = grid_full(v[0].cam);
    if (fast) vlaunch(k_denoise_variance<false, true>, k_denoise_variance<true, true>, g, v, st, s, cur);
    else vlaunch(k_denoise_variance<false, false>, k_denoise_variance<true, false>, g, v, st, s, cur);
}
void launch_denoise_wavelet(const ViewSet& v, const SceneDev& s, int cur, u32 frame, u32 stride, float strength, const float4* di_in, float4* di_out, const float4* gi_in, float4* gi_out,
                            const float4* pair_in, float4* pair_out, bool fast, cudaStream_t st) {
#define ST_WG(F_, P_) vlaunch(k_denoise_wavelet<false, F_, P_>, k_denoise_wavelet<true, F_, P_>, grid_full(v[0].cam), v, st, s, cur, frame, stride, strength, di_in, di_out, gi_in, gi_out, pair_in, pair_out)
    if (pair_in) { if (fast) ST_WG(true, true); else ST_WG(false, true); }
    else { if (fast) ST_WG(true, false); else ST_WG(false, false); }
#undef ST_WG
}
// K21, tile-staged: the 6x5 window of frame_denoising::estimate_variance (quirk C-3: row -2 spans x in [-2,2], rows -1..2 span
// x in [-3,2]) is only walked by pixels whose history is shorter than 4 frames, but a warp pays for it as soon as one of its
// pixels does; with the (TW+6) x (TH+4) neighbourhood in shared memory (three TMA tensor copies, zero fill outside the frame)
// those 29 taps are LDS.128 at fixed offsets instead of 87 gathered global loads.  Same taps, order and arithmetic as
// k_denoise_variance.
template <int TW, int TH> struct VarianceTile {
    static constexpr int HX = 3, HY = 2, BW = TW + 2 * HX, BH = TH + 2 * HY;
    static constexpr u32 BOX_BYTES = (u32)(BW * BH * 16);
    static constexpr u32 PLANE = (BOX_BYTES + 127u) & ~127u;
    static constexpr u32 SMEM = 3u * PLANE + 128u;
};
template <bool FAST, int TW, int TH>
__global__ void __launch_bounds__(TW * TH) k_denoise_variance_tiled(KPARAMS, int cur, const __grid_constant__ CUtensorMap tm_nd, const __grid_constant__ CUtensorMap tm_di,
                                                                    const __grid_constant__ CUtensorMap tm_gi, u32* __restrict__ errors) {
    typedef VarianceTile<TW, TH> T;
    extern __shared__ unsigned char s_raw[];
    __shared__ __align__(8) unsigned long long s_bar;
    const int tx = (int)threadIdx.x % TW, ty = (int)threadIdx.x / TW;
    const int x0 = (int)blockIdx.x * TW, y0 = cam.y0 + (int)blockIdx.y * TH;
    const u32 bar = smem_addr(&s_bar);
    const u32 raw = smem_addr(s_raw);
    const u32 base = (raw + 127u) & ~127u;
    if (threadIdx.x == 0) { mbar_init(bar, 1u); mbar_fence_init(); }
    __syncthreads();
    if (threadIdx.x == 0) {
        mbar_expect_tx(bar, 3u * T::BOX_BYTES);
        tma_load_2d(base, &tm_nd, (x0 - T::HX) * 2, y0 - T::HY, bar);
        tma_load_2d(base + T::PLANE, &tm_di, (x0 - T::HX) * 2, y0 - T::HY, bar);
        tma_load_2d(base + 2u * T::PLANE, &tm_gi, (x0 - T::HX) * 2, y0 - T::HY, bar);
    }
    const u32 px = (u32)(x0 + tx), py = (u32)(y0 + ty);
    const bool in = px < (u32)cam.w && py < (u32)cam.y1;
    const size_t i = in ? pix(cam, px, py) : 0;
    float4 mdi = f4zero(), mgi = f4zero();
    if (in) { mdi = cam.di_diff_moments[cur][i]; mgi = cam.gi_diff_moments[cur][i]; }   // in flight together with the tile
    {
        bool done = false;
        for (u32 spin = 0; spin < (1u << 20) && !done; spin++) done = mbar_try_wait(bar, 0u);
        if (!done) { if (threadIdx.x == 0) atomicAdd(errors, 1u); return; }
    }
    if (!in) return;
    const float4* __restrict__ t_nd = reinterpret_cast<const float4*>(s_raw + (base - raw));
    const float4* __restrict__ t_di = reinterpret_cast<const float4*>(s_raw + (base - raw) + T::PLANE);
    const float4* __restrict__ t_gi = reinterpret_cast<const float4*>(s_raw + (base - raw) + 2u * T::PLANE);
    const int c = (ty + T::HY) * T::BW + (tx + T::HX);
    float4 cnd = t_nd[c];
    float4 cdi = t_di[c], cgi = t_gi[c];
    if (cnd.w == 0.0f) { cam.di_diff_stash[i] = cdi; cam.gi_diff_stash[i] = cgi; return; }
    float di_var, gi_var;
    if (mdi.x >= 4.0f) { di_var = mdi.z - sq(mdi.y); gi_var = mgi.z - sq(mgi.y); }
    else {
        float3 cn = xyz(cnd);
        float scdl = sv_sqrt<FAST>(sv_luma<FAST>(xyz(cdi))), scgl = sv_sqrt<FAST>(sv_luma<FAST>(xyz(cgi)));
        float3 sdi = f3s(0.f), sgi = f3s(0.f);
#pragma unroll
        for (int oy = -2; oy <= 2; oy++) {
#pragma unroll
            for (int ox = -3; ox <= 2; ox++) {
                if (oy == -2 && ox == -3) continue;   // quirk C-3: the first row starts at -2
                const int k = c + oy * T::BW + ox;
                float4 nds = t_nd[k];
                if (nds.w != 0.0f) {   // zero = sky, or outside the frame (zero-filled by the tensor copy)
                    float common = svgf_depth_weight<FAST>(cnd.w, nds.w, 0.2f);
                    float nw = svgf_normal_weight<FAST>(cn, xyz(nds));
                    float sl = sv_luma<FAST>(xyz(t_di[k]));
                    float w = svgf_luma_weight<FAST>(scdl, sl, 1.0f) * common * nw;
                    sdi = sdi + f3(sl, sl * sl, 1.0f) * f3s(w);
                    float gl = sv_luma<FAST>(xyz(t_gi[k]));
                    float wg = svgf_luma_weight<FAST>(scgl, gl, 1.0f) * common * nw;
                    sgi = sgi + f3(gl, gl * gl, 1.0f) * f3s(wg);
                }
            }
        }
        { float m1 = sdi.x / sdi.z, m2 = sdi.y / sdi.z; di_var = fabs_(m2 - m1 * m1) * 4.0f; }
        { float m1 = sgi.x / sgi.z, m2 = sgi.y / sgi.z; gi_var = fabs_(m2 - m1 * m1) * 4.0f; }
    }
    di_var = rmax(di_var, 0.0f); gi_var = rmax(gi_var, 0.0f);
    cam.di_diff_stash[i] = f4(xyz(cdi), di_var);
    cam.gi_diff_stash[i] = f4(xyz(cgi), gi_var);
}

// ---- tile-staged K22: tensor maps + launcher --------------------------------------------------
// A float4 image plane as a 2-D tensor of 8-byte elements (2W x H; the widest element type a tensor map
// takes, so that a (TW+2·HL)-pixel box row stays under the 256-element box limit), row pitch W·16 B, no
// swizzle / interleave, zero fill outside the frame.  Maps are cached per (plane, frame size, box).
typedef CUresult (*TensorMapEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                      const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static TensorMapEncodeFn tensor_map_encoder() {
    static TensorMapEncodeFn fn = [] {
        void* p = nullptr; cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) p = nullptr;
        return (TensorMapEncodeFn)p;
    }();
    return fn;
}
static bool wavelet_tensor_map(const float4* plane, int w, int h, int bw, int bh, CUtensorMap* out) {
    typedef std::tuple<const void*, int, int, int, int> Key;
    static std::map<Key, CUtensorMap> cache; static std::mutex mu;
    std::lock_guard<std::mutex> lock(mu);
    Key key(plane, w, h, bw, bh);
    auto it = cache.find(key);
    if (it != cache.end()) { *out = it->second; return true; }
    TensorMapEncodeFn enc = tensor_map_encoder();
    if (!enc) {   // no driver entry point for tensor maps: the callers fall back to the gather kernels; say so once
        static bool warned = false;
        if (!warned) { warned = true; std::fprintf(stderr, "strolle_b200: cuTensorMapEncodeTiled is not available from this driver; the tile-staged SVGF kernels are off\n"); }
        return false;
    }
    cuuint64_t dims[2] = {(cuuint64_t)w * 2u, (cuuint64_t)h};
    cuuint64_t strides[1] = {(cuuint64_t)w * 16u};
    cuuint32_t box[2] = {(cuuint32_t)bw * 2u, (cuuint32_t)bh};
    cuuint32_t estr[2] = {1u, 1u};
    CUtensorMap tm;
    if (enc(&tm, CU_TENSOR_MAP_DATA_TYPE_UINT64, 2, const_cast<float4*>(plane), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS) return false;
    if (cache.size() > 4096) cache.clear();
    cache[key] = tm; *out = tm;
    return true;
}
template <bool FAST, int S, int J, int TW, int TH>
static bool wavelet_tiled_go(const CameraDev& c, const SceneDev& s, u32 frame, float strength, const float4* di_in, float4* di_out, const float4* gi_in, float4* gi_out,
                             float4* pair_out, u32* errors, cudaStream_t st) {
    typedef WaveletTile<S, J, TW, TH> T;
    if (T::BW * 2 > 256 || T::BH > 256) return false;
    CUtensorMap tn, td, tg;
    if (!wavelet_tensor_map(c.surface_nd, c.w, c.h, T::BW, T::BH, &tn) || !wavelet_tensor_map(di_in, c.w, c.h, T::BW, T::BH, &td) ||
        !wavelet_tensor_map(gi_in, c.w, c.h, T::BW, T::BH, &tg)) return false;
    auto kern = k_denoise_wavelet_tiled<FAST, S, J, TW, TH>;
    static bool attr_set[64] = {};   // per instantiation and device
    int dev = 0; cudaGetDevice(&dev); dev &= 63;
    if (!attr_set[dev]) { if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)T::SMEM) != cudaSuccess) { cudaGetLastError(); return false; } attr_set[dev] = true; }
    dim3 grid((c.w + TW - 1) / TW, (c.y1 - c.y0 + TH - 1) / TH);
    kern<<<grid, TW * TH, T::SMEM, st>>>(c, s, frame, strength, tn, td, tg, di_out, gi_out, pair_out, errors);
    return true;
}
template <bool FAST, int S, int J>
static bool wavelet_tiled_cfg(int cfg, const CameraDev& c, const SceneDev& s, u32 frame, float strength, const float4* di_in, float4* di_out, const float4* gi_in, float4* gi_out,
                              float4* pair_out, u32* errors, cudaStream_t st) {
    switch (cfg) {
    case 0: return wavelet_tiled_go<FAST, S, J, 32, 8>(c, s, frame, strength, di_in, di_out, gi_in, gi_out, pair_out, errors, st);
    case 1: return wavelet_tiled_go<FAST, S, J, 32, 16>(c, s, frame, strength, di_in, di_out, gi_in, gi_out, pair_out, errors, st);
    case 2: return wavelet_tiled_go<FAST, S, J, 64, 4>(c, s, frame, strength, di_in, di_out, gi_in, gi_out, pair_out, errors, st);
    case 3: return wavelet_tiled_go<FAST, S, J, 64, 8>(c, s, frame, strength, di_in, di_out, gi_in, gi_out, pair_out, errors, st);
    default: return false;
    }
}
// Returns false when the tile-staged kernel cannot be used for this launch (the caller then runs the gather kernel):
// the camera's screen is not the buffer size, no tensor-map encoder, or an unknown configuration.
bool launch_denoise_wavelet_tiled(const CameraDev& c, const SceneDev& s, u32 frame, u32 stride, float strength, const float4* di_in, float4* di_out, const float4* gi_in,
                                  float4* gi_out, float4* pair_out, bool fast, int cfg, u32* errors, cudaStream_t st) {
    if (c.curr.screen.x != (float)c.w || c.curr.screen.y != (float)c.h) return false;   // zero fill == Camera::contains only then
#define ST_WT(S_, J_) (fast ? wavelet_tiled_cfg<true, S_, J_>(cfg, c, s, frame, strength, di_in, di_out, gi_in, gi_out, pair_out, errors, st) \
                            : wavelet_tiled_cfg<false, S_, J_>(cfg, c, s, frame, strength, di_in, di_out, gi_in, gi_out, pair_out, errors, st))
    switch (stride) {
    case 1: return ST_WT(1, 0);
    case 2: return ST_WT(2, 0);
    case 4: return ST_WT(4, 0);
    case 8: return ST_WT(8, 1);
    case 16: return ST_WT(16, 3);
    default: return false;
    }
#undef ST_WT
}
template <bool FAST>
static bool variance_tiled_go(const CameraDev& c, const SceneDev& s, int cur, u32* errors, cudaStream_t st) {
    typedef VarianceTile<32, 8> T;
    CUtensorMap tn, td, tg;
    if (!wavelet_tensor_map(c.surface_nd, c.w, c.h, T::BW, T::BH, &tn) || !wavelet_tensor_map(c.di_diff_curr_colors, c.w, c.h, T::BW, T::BH, &td) ||
        !wavelet_tensor_map(c.gi_diff_curr_colors, c.w, c.h, T::BW, T::BH, &tg)) return false;
    auto kern = k_denoise_variance_tiled<FAST, 32, 8>;
    static bool attr_set[64] = {};
    int dev = 0; cudaGetDevice(&dev); dev &= 63;
    if (!attr_set[dev]) { if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)T::SMEM) != cudaSuccess) { cudaGetLastError(); return false; } attr_set[dev] = true; }
    dim3 grid((c.w + 31) / 32, (c.y1 - c.y0 + 7) / 8);
    kern<<<grid, 256, T::SMEM, st>>>(c, s, cur, tn, td, tg, errors);
    return true;
}
bool launch_denoise_variance_tiled(const CameraDev& c, const SceneDev& s, int cur, bool fast, u32* errors, cudaStream_t st) {
    if (c.curr.screen.x != (float)c.w || c.curr.screen.y != (float)c.h) return false;   // zero fill == Camera::contains only then
    return fast ? variance_tiled_go<true>(c, s, cur, errors, st) : variance_tiled_go<false>(c, s, cur, errors, st);
}
void launch_composition(const ViewSet& v, const SceneDev& s, int cur, u32 mode, const float4* di_diff, const float4* gi_diff, cudaStream_t st) { FULL_LAUNCH(k_composition, v, st, s, cur, mode, di_diff, gi_diff); }
void launch_output_store(const ViewSet& v, const SceneDev& s, int format, cudaStream_t st) {
    const dim3 g = grid_full(v[0].cam);
    if (format == OUT_RGBA32F) vlaunch(k_output_store<false, OUT_RGBA32F>, k_output_store<true, OUT_RGBA32F>, g, v, st, s);
    else if (format == OUT_RGBA16F) vlaunch(k_output_store<false, OUT_RGBA16F>, k_output_store<true, OUT_RGBA16F>, g, v, st, s);
    else vlaunch(k_output_store<false, OUT_RGBA8_SRGB>, k_output_store<true, OUT_RGBA8_SRGB>, g, v, st, s);
}
void launch_ref_tracing(const ViewSet& v, const SceneDev& s, u32 depth, cudaStream_t st) { FULL_LAUNCH(k_ref_tracing, v, st, s, depth); }
void launch_ref_shading(const ViewSet& v, const SceneDev& s, u32 seed, u32 depth, cudaStream_t st) { FULL_LAUNCH(k_ref_shading, v, st, s, seed, depth); }
void launch_bvh_heatmap(const ViewSet& v, const SceneDev& s, cudaStream_t st) { FULL_LAUNCH(k_bvh_heatmap, v, st, s); }
void launch_trace_stream_closest(const SceneDev& s, const float4* rays, long n, float4* out, cudaStream_t st) { k_trace_stream_closest<<<(unsigned)((n + ST_BLOCK - 1) / ST_BLOCK), ST_BLOCK, 0, st>>>(s, rays, n, out); }
void launch_trace_stream_any(const SceneDev& s, const float4* rays, long n, u32* out, cudaStream_t st) { k_trace_stream_any<<<(unsigned)((n + ST_BLOCK - 1) / ST_BLOCK), ST_BLOCK, 0, st>>>(s, rays, n, out); }
void launch_math(int op, const float* a, const float* b, float* out, long n, cudaStream_t st) { k_math<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(op, a, b, out, n); }
void launch_material_derive(const GpuMaterial* mats, u32 n, u32* packed, cudaStream_t st) { if (n) k_material_derive<<<(n + 127) / 128, 128, 0, st>>>(mats, n, packed); }
void launch_srgb_lut(float* lut, cudaStream_t st) { k_srgb_lut<<<1, 256, 0, st>>>(lut); }
void launch_unpack_lut(float* lut, cudaStream_t st) { k_unpack_lut<<<1, 256, 0, st>>>(lut); }
// ---- dynamic images: caller surfaces -> atlas rectangles, one launch per tick for every image (st_tick) --------------------------------------
// A block copies rows [r0, r1) of one image: the tile's units (4-byte texels of the ragged head and tail, 16-byte groups in between) are
// spread over the block's threads.  Sources may be peer device memory or mapped host memory; every load is read once.
constexpr u32 kAtlasRefreshThreads = 256;
__global__ void __launch_bounds__(kAtlasRefreshThreads) k_atlas_refresh(const __grid_constant__ AtlasCopyBatch b, uchar4* __restrict__ atlas) {
    int lo = 0, hi = b.n - 1;
    while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (b.c[mid].block0 <= blockIdx.x) lo = mid; else hi = mid - 1; }
    const AtlasCopy& c = b.c[lo];
    const u32 r0 = (blockIdx.x - c.block0) * c.rows_per_block, rows = min(c.h - r0, c.rows_per_block);
    const u32 units = c.head + c.body + c.tail, total = rows * units;
    for (u32 i = threadIdx.x; i < total; i += kAtlasRefreshThreads) {
        const u32 r = r0 + i / units, u = i % units;
        const char* s = c.src + (size_t)r * c.pitch;
        uchar4* d = atlas + (size_t)(c.y + r) * kAtlasSize + c.x;
        if (u >= c.head && u < c.head + c.body) {
            const u32 t = c.head + 4u * (u - c.head);
            *reinterpret_cast<uint4*>(d + t) = __ldcs(reinterpret_cast<const uint4*>(s + 4 * (size_t)t));
        } else {
            const u32 t = u < c.head ? u : u + 3u * c.body;   // tail texel: head + 4 * body + (u - head - body)
            d[t] = __ldcs(reinterpret_cast<const uchar4*>(s + 4 * (size_t)t));
        }
    }
}
int launch_atlas_refresh(std::vector<AtlasCopy>& copies, uchar4* atlas, cudaStream_t st) {
    int launches = 0;
    for (size_t c0 = 0; c0 < copies.size(); c0 += kAtlasCopies) {
        AtlasCopyBatch b; b.n = (int)std::min<size_t>(kAtlasCopies, copies.size() - c0);
        u32 blocks = 0;
        for (int k = 0; k < b.n; k++) {
            AtlasCopy& c = copies[c0 + k];
            // 16-byte groups need the source row and the atlas row to share their address modulo 16 on every row
            const u32 dmis = (4u * c.x) & 15u;
            const bool wide = ((uintptr_t)c.src & 15u) == dmis && c.pitch % 16 == 0;
            c.head = wide ? std::min(c.w, ((16u - dmis) & 15u) / 4u) : c.w;
            c.body = wide ? (c.w - c.head) / 4u : 0u;
            c.tail = c.w - c.head - 4u * c.body;
            const u32 units = c.head + c.body + c.tail;
            c.rows_per_block = std::max(1u, std::min(c.h, kAtlasRefreshThreads / units));   // about one unit per thread
            c.block0 = blocks;
            blocks += (c.h + c.rows_per_block - 1) / c.rows_per_block;
            b.c[k] = c;
        }
        k_atlas_refresh<<<blocks, kAtlasRefreshThreads, 0, st>>>(b, atlas);
        launches++;
    }
    return launches;
}
// ---- strips, fused transport: sequence flags between ranks + the temporal pull -------------------------------------------
// Flags live in each rank's own memory, word [slot * ST_PEER_MAX_RANKS + source rank]; a rank raises its word in a peer's array to
// the frame's sequence number with a system-scope release store after the kernels that produced the rows have completed
// (stream order + fence), and a consumer spins on its local words with acquire loads.  One warp, lane r <-> rank r.
ST_DEV void st_release_sys(u32* p, u32 v) { asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
ST_DEV u32 ld_acquire_sys(const u32* p) { u32 v; asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v; }
__global__ void __launch_bounds__(32) k_strip_signal(const __grid_constant__ StripSync s, int slot, u32 seq, u32 dst_mask, int* reset_need, int h) {
    __threadfence_system();
    int r = (int)threadIdx.x;
    if (r < s.n_ranks && r != s.rank && ((dst_mask >> r) & 1u) && s.peer_flags[r] != nullptr) st_release_sys(s.peer_flags[r] + slot * ST_PEER_MAX_RANKS + s.rank, seq);
    if (reset_need != nullptr && r == 0) { reset_need[0] = h; reset_need[1] = -1; }
}
__global__ void __launch_bounds__(32) k_strip_wait(const __grid_constant__ StripSync s, int slot, u32 seq, u32 src_mask) {
    int r = (int)threadIdx.x;
    if (r < s.n_ranks && r != s.rank && ((src_mask >> r) & 1u)) {
        const u32* f = s.my_flags + slot * ST_PEER_MAX_RANKS + r;
        long long t0 = clock64();
        while ((int)(ld_acquire_sys(f) - seq) < 0) {
            if (clock64() - t0 > 20000000000ll) {   // ~10 s: a peer died; do not hang the GPU.  errors[1] keeps the first wait that gave up
                atomicAdd(s.errors, 1u); atomicCAS(s.errors + 1, 0u, 0x80000000u | ((u32)slot << 16) | ((u32)r << 8) | (seq & 0xffu)); break;
            }
            __nanosleep(64);
        }
    }
    __threadfence_system();
}
// Temporal pull: rows [need_lo, own_y0) and [own_y1, need_hi] of last frame's outputs, read from their owners' arenas over NVLink
// (P2P loads).  The row range was measured on the device by this frame's G-buffer pass, so a static camera pulls nothing and
// any amount of motion is covered exactly.  blockIdx.y = buffer.
__global__ void __launch_bounds__(256) k_strip_pull(const __grid_constant__ StripPull p) {
    const int lo = max(0, min(p.need_rows[0], p.own_y0)), hi = min(p.h - 1, max(p.need_rows[1], p.own_y1 - 1));
    const StripPullItem it = p.items[blockIdx.y];
    // rows this rank already holds because it computes them itself (the extended G-buffer rows of the previous frame)
    const int have_lo = max(0, p.own_y0 - it.local_rows), have_hi = min(p.h, p.own_y1 + it.local_rows);
    const int up0 = lo, up1 = min(p.own_y0, have_lo), dn0 = max(p.own_y1, have_hi), dn1 = hi + 1;
    const int nup = max(0, up1 - up0), ndn = max(0, dn1 - dn0);
    const unsigned long long per_row = (unsigned long long)p.w * (unsigned long long)it.vec4_per_px;
    const unsigned long long total = (unsigned long long)(nup + ndn) * per_row;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (unsigned long long)gridDim.x * blockDim.x) {
        int ri = (int)(i / per_row);
        unsigned long long col = i - (unsigned long long)ri * per_row;
        int row = ri < nup ? up0 + ri : dn0 + (ri - nup);
        int owner = 0;
        while (owner + 1 < p.n_ranks && row >= p.bounds[owner + 1]) owner++;
        size_t off = it.offset + ((size_t)row * per_row + col) * 16;
        *reinterpret_cast<uint4*>(p.arena[p.rank] + off) = *reinterpret_cast<const uint4*>(p.arena[owner] + off);
    }
    // statistics: rows of last frame this strip reached into, beyond its own (whatever part of them a buffer then had to fetch)
    if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) { int reach = max(0, p.own_y0 - lo) + max(0, hi + 1 - p.own_y1); if (reach > 0) atomicAdd(p.pulled_rows, (unsigned long long)reach); }
}
// a signal and a wait that follow each other on the stream, as one launch
__global__ void __launch_bounds__(32) k_strip_signal_wait(const __grid_constant__ StripSync s, int sig_slot, u32 seq, u32 dst_mask, int wait_slot, u32 wait_seq, u32 src_mask) {
    __threadfence_system();
    int r = (int)threadIdx.x;
    if (r < s.n_ranks && r != s.rank && ((dst_mask >> r) & 1u) && s.peer_flags[r] != nullptr) st_release_sys(s.peer_flags[r] + sig_slot * ST_PEER_MAX_RANKS + s.rank, seq);
    if (r < s.n_ranks && r != s.rank && ((src_mask >> r) & 1u)) {
        const u32* f = s.my_flags + wait_slot * ST_PEER_MAX_RANKS + r;
        long long t0 = clock64();
        while ((int)(ld_acquire_sys(f) - wait_seq) < 0) {
            if (clock64() - t0 > 20000000000ll) { atomicAdd(s.errors, 1u); break; }
            __nanosleep(64);
        }
    }
    __threadfence_system();
}
void launch_strip_signal_wait(const StripSync& s, int sig_slot, u32 seq, u32 dst_mask, int wait_slot, u32 wait_seq, u32 src_mask, cudaStream_t st) { k_strip_signal_wait<<<1, 32, 0, st>>>(s, sig_slot, seq, dst_mask, wait_slot, wait_seq, src_mask); }
void launch_strip_signal(const StripSync& s, int slot, u32 seq, u32 dst_mask, int* reset_need, int h, cudaStream_t st) { k_strip_signal<<<1, 32, 0, st>>>(s, slot, seq, dst_mask, reset_need, h); }
void launch_strip_wait(const StripSync& s, int slot, u32 seq, u32 src_mask, cudaStream_t st) { k_strip_wait<<<1, 32, 0, st>>>(s, slot, seq, src_mask); }
void launch_strip_pull(const StripPull& p, cudaStream_t st) { if (p.nitems > 0) k_strip_pull<<<dim3(48, (unsigned)p.nitems), 256, 0, st>>>(p); }

// ---- strips: push boundary rows into the neighbours' buffers, then barrier --------------------------------------
// One launch per exchange point.  blockIdx.y = segment (a run of rows of one buffer for one peer), blockIdx.x strides
// it with 16-byte stores that land in the peer's HBM through NVLink.  The last block to finish (completion counter)
// publishes `seq` in every peer's flag array after a system-scope fence and then spins until every peer has published
// the same `seq` here, so the next kernel on this stream sees all incoming rows.  Every exchange is a barrier over all
// ranks, which also orders a buffer's next overwrite after its last remote read.
__global__ void __launch_bounds__(256) k_peer_exchange(const __grid_constant__ PeerExchange x) {
    if (x.nseg > 0) {
        const PeerSegment& sg = x.seg[blockIdx.y];
        const uint4* __restrict__ src = sg.src; uint4* __restrict__ dst = sg.dst;
        for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < sg.n; i += (unsigned long long)gridDim.x * blockDim.x) dst[i] = src[i];
    }
    if (!x.signal) return;
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x != 0) return;
    unsigned total = gridDim.x * gridDim.y;
    if (atomicAdd(x.counter, 1u) != total - 1u) return;
    *x.counter = 0u;
    __threadfence_system();
    for (int r = 0; r < x.n_ranks; r++) if (r != x.rank) *(volatile u32*)x.peer_flags[r] = x.seq;
    long long t0 = clock64();
    for (int r = 0; r < x.n_ranks; r++) {
        if (r == x.rank) continue;
        const volatile u32* f = x.my_flags + r;
        while ((int)(*f - x.seq) < 0) {
            if (clock64() - t0 > 20000000000ll) { atomicAdd(x.errors, 1u); break; }   // ~10 s: a peer died; do not hang the GPU
            __nanosleep(100);
        }
    }
    __threadfence_system();
}
void launch_peer_exchange(const PeerExchange& x, cudaStream_t st) {
    unsigned ny = x.nseg > 0 ? (unsigned)x.nseg : 1u;
    unsigned nx = x.nseg > 0 ? std::max(4u, std::min(64u, 1184u / ny)) : 1u;
    k_peer_exchange<<<dim3(nx, ny), 256, 0, st>>>(x);
}
void launch_atm_transmittance(float4* out, cudaStream_t st) { k_atm_transmittance<<<dim3(2, 64), 128, 0, st>>>(out); }
void launch_atm_scattering(const float4* tl, float4* out, cudaStream_t st) { k_atm_scattering<<<32, 32, 0, st>>>(tl, out); }
void launch_atm_sky(const float4* tl, const float4* sl, float sun_altitude, float4* out, cudaStream_t st) { k_atm_sky<<<256, 256, 0, st>>>(tl, sl, sun_altitude, out); }
void launch_atm_sun_color(float4* out2, const GpuWorld& world, cudaStream_t st) { k_atm_sun_color<<<1, 1, 0, st>>>(out2, world); }

#endif   // ST_EXACT_ONLY

// Load every kernel of this translation unit's module now.  CUDA loads kernels lazily, at their first launch, and that load can
// synchronise the whole context; the strip transport lets one stream spin on a flag that a kernel launched later (by the same host
// thread, for another member of a device group) raises, so a load at that moment would stall the thread until the wait gives up.
// The module is found through one of its kernels; every function it holds is then loaded (cuFuncLoad, CUDA >= 12.4).
int preload_kernels() {
    static int states[64];   // per flavour (this function is compiled into st:: and stf::) and per device: every context holds its own copy of the module
    static bool init = false;
    if (!init) { for (int& v : states) v = -1; init = true; }
    int dev = 0; cudaGetDevice(&dev);
    int& state = states[dev & 63];
    if (state >= 0) return state;
    auto entry = [](const char* name) -> void* {
        void* p = nullptr; cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint(name, &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) return nullptr;
        return p;
    };
    typedef CUresult (*GetModule)(CUmodule*, CUfunction);
    typedef CUresult (*GetCount)(unsigned int*, CUmodule);
    typedef CUresult (*Enumerate)(CUfunction*, unsigned int, CUmodule);
    typedef CUresult (*Load)(CUfunction);
    GetModule get_module = (GetModule)entry("cuFuncGetModule"); GetCount get_count = (GetCount)entry("cuModuleGetFunctionCount");
    Enumerate enumerate = (Enumerate)entry("cuModuleEnumerateFunctions"); Load load = (Load)entry("cuFuncLoad");
    cudaGetLastError();
    if (!get_module || !get_count || !enumerate || !load) return state = 1;
    cudaFunction_t anchor = nullptr;
    if (cudaGetFuncBySymbol(&anchor, (const void*)k_di_sample_temporal<false>) != cudaSuccess) { cudaGetLastError(); return state = 2; }
    CUmodule mod = nullptr; unsigned int n = 0;
    if (get_module(&mod, (CUfunction)anchor) != CUDA_SUCCESS || get_count(&n, mod) != CUDA_SUCCESS || n == 0u) return state = 3;
    std::vector<CUfunction> fns(n);
    if (enumerate(fns.data(), n, mod) != CUDA_SUCCESS) return state = 4;
    for (CUfunction f : fns) if (load(f) != CUDA_SUCCESS) return state = 5;
    return state = 0;
}
}  // namespace ST_NS
