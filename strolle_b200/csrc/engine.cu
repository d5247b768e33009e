// strolle_b200 — host engine behind the C ABI (include/strolle_b200.h).
//
// Mirrors strolle::Engine (strolle/src/lib.rs:104-395): scene stores, world-space triangle
// baking, binned-SAH BVH build + DFS serialisation, the light slot protocol, per-camera
// buffers and the per-frame pass schedule of CameraController::render — with CUDA device
// allocations, one stream and cudaMemcpyAsync uploads in place of wgpu buffers, bind groups
// and queue.write_buffer.  Host float arithmetic is compiled with -ffp-contract=off.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <deque>
#include <functional>
#include <limits>
#include <memory>
#include <string>
#include <unordered_map>
#include <vector>

#include <nccl.h>

#include "../../include/strolle_b200.h"
#include "kernels.h"

// NCCL is bound at run time (dlopen), never at link time: the host process normally already holds the NCCL that
// its torch build ships, and a second copy with the same soname must not shadow it.
#include <dlfcn.h>
namespace {
struct NcclApi {
    void* lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    bool load(std::string* err) {
        if (lib) return true;
        void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);
        if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_LOCAL);
        if (!h) { *err = std::string("cannot load libnccl.so.2: ") + dlerror(); return false; }
        auto sym = [&](const char* n) { void* p = dlsym(h, n); if (!p) *err = std::string("libnccl.so.2 lacks ") + n; return p; };
        GetUniqueId = (decltype(GetUniqueId))sym("ncclGetUniqueId"); CommInitRank = (decltype(CommInitRank))sym("ncclCommInitRank");
        CommDestroy = (decltype(CommDestroy))sym("ncclCommDestroy"); GroupStart = (decltype(GroupStart))sym("ncclGroupStart");
        GroupEnd = (decltype(GroupEnd))sym("ncclGroupEnd"); Send = (decltype(Send))sym("ncclSend"); Recv = (decltype(Recv))sym("ncclRecv");
        GetErrorString = (decltype(GetErrorString))sym("ncclGetErrorString");
        if (!GetUniqueId || !CommInitRank || !CommDestroy || !GroupStart || !GroupEnd || !Send || !Recv || !GetErrorString) return false;
        lib = h; return true;
    }
};
NcclApi g_nccl;
}


namespace st {

static thread_local std::string g_err;
static int fail(int code, const std::string& msg) { g_err = msg; return code; }
#define CK(call)                                                                                   \
    do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return fail(ST_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); } while (0)

// ---- small host vector maths (glam evaluation order) ----------------------------------------------
struct H3 { float x, y, z; };
static inline H3 h3(float x, float y, float z) { H3 r = {x, y, z}; return r; }
static inline H3 operator+(H3 a, H3 b) { return h3(a.x + b.x, a.y + b.y, a.z + b.z); }
static inline H3 operator-(H3 a, H3 b) { return h3(a.x - b.x, a.y - b.y, a.z - b.z); }
static inline H3 operator*(H3 a, float s) { return h3(a.x * s, a.y * s, a.z * s); }
static inline H3 operator*(H3 a, H3 b) { return h3(a.x * b.x, a.y * b.y, a.z * b.z); }
static inline H3 operator/(H3 a, float s) { return h3(a.x / s, a.y / s, a.z / s); }
static inline float hdot(H3 a, H3 b) { return (a.x * b.x) + (a.y * b.y) + (a.z * b.z); }
static inline H3 hcross(H3 a, H3 b) { return h3(a.y * b.z - b.y * a.z, a.z * b.x - b.z * a.x, a.x * b.y - b.x * a.y); }
static inline H3 hnorm(H3 a) { return a * (1.0f / std::sqrt(hdot(a, a))); }
static inline float hmin(float a, float b) { return (a != a) ? b : ((b != b) ? a : (a < b ? a : b)); }
static inline float hmax(float a, float b) { return (a != a) ? b : ((b != b) ? a : (a > b ? a : b)); }
static inline uint32_t to_u32(float f) { if (!(f == f) || f <= 0.0f) return 0u; if (f >= 4294967296.0f) return 0xffffffffu; return (uint32_t)f; }
static inline float bits2f(uint32_t u) { float f; std::memcpy(&f, &u, 4); return f; }
static inline uint32_t f2bits(float f) { uint32_t u; std::memcpy(&u, &f, 4); return u; }
static const float FMAX = std::numeric_limits<float>::max();

struct Affine3 { H3 x, y, z, t; };
static inline H3 aff_mat(const Affine3& a, H3 v) { return (a.x * v.x + a.y * v.y) + a.z * v.z; }
static inline H3 aff_point(const Affine3& a, H3 p) { return aff_mat(a, p) + a.t; }
static Affine3 aff_inverse(const Affine3& a) {   // glam Affine3A::inverse
    H3 t0 = hcross(a.y, a.z), t1 = hcross(a.z, a.x), t2 = hcross(a.x, a.y);
    float det = hdot(a.z, t2);
    float inv = 1.0f / det;
    H3 c0 = t0 * inv, c1 = t1 * inv, c2 = t2 * inv;
    Affine3 r;
    r.x = h3(c0.x, c1.x, c2.x); r.y = h3(c0.y, c1.y, c2.y); r.z = h3(c0.z, c1.z, c2.z);
    H3 mt = aff_mat(r, a.t);
    r.t = h3(-mt.x, -mt.y, -mt.z);
    return r;
}

struct Box {   // strolle/src/utils/bounding_box.rs
    H3 lo, hi;
    Box() : lo(h3(FMAX, FMAX, FMAX)), hi(h3(-FMAX, -FMAX, -FMAX)) {}
    void grow(H3 p) { lo = h3(hmin(lo.x, p.x), hmin(lo.y, p.y), hmin(lo.z, p.z)); hi = h3(hmax(hi.x, p.x), hmax(hi.y, p.y), hmax(hi.z, p.z)); }
    void grow(const Box& b) { grow(b.lo); grow(b.hi); }
    // same results as grow() when no operand is NaN (the NaN-ignoring min/max of Rust's f32::min/max reduce to these selects)
    void grow_finite(H3 p) {
        lo.x = (lo.x < p.x) ? lo.x : p.x; lo.y = (lo.y < p.y) ? lo.y : p.y; lo.z = (lo.z < p.z) ? lo.z : p.z;
        hi.x = (hi.x > p.x) ? hi.x : p.x; hi.y = (hi.y > p.y) ? hi.y : p.y; hi.z = (hi.z > p.z) ? hi.z : p.z;
    }
    void grow_finite(const Box& b) { grow_finite(b.lo); grow_finite(b.hi); }
    template <bool FINITE> void add(H3 p) { if (FINITE) grow_finite(p); else grow(p); }
    template <bool FINITE> void add(const Box& b) { if (FINITE) grow_finite(b); else grow(b); }
    bool set() const { return lo.x != FMAX; }
    float half_area() const { H3 e = hi - lo; return e.x * e.y + e.y * e.z + e.z * e.x; }
};

// 4x4 column-major helpers for Camera::serialize (strolle/src/camera.rs:50-66)
struct HM4 { float m[16]; };
static HM4 hm_mul(const HM4& a, const HM4& b) {
    HM4 r;
    for (int c = 0; c < 4; c++) {
        float v0 = b.m[4 * c], v1 = b.m[4 * c + 1], v2 = b.m[4 * c + 2], v3 = b.m[4 * c + 3];
        for (int k = 0; k < 4; k++) {
            float acc = a.m[k] * v0;
            acc = acc + a.m[4 + k] * v1;
            acc = acc + a.m[8 + k] * v2;
            acc = acc + a.m[12 + k] * v3;
            r.m[4 * c + k] = acc;
        }
    }
    return r;
}
static HM4 hm_inverse(const HM4& s) {   // cofactor expansion in glam's Mat4::inverse order
    const float* m = s.m;
    float m00 = m[0], m01 = m[1], m02 = m[2], m03 = m[3], m10 = m[4], m11 = m[5], m12 = m[6], m13 = m[7];
    float m20 = m[8], m21 = m[9], m22 = m[10], m23 = m[11], m30 = m[12], m31 = m[13], m32 = m[14], m33 = m[15];
    float c00 = m22 * m33 - m32 * m23, c02 = m12 * m33 - m32 * m13, c03 = m12 * m23 - m22 * m13;
    float c04 = m21 * m33 - m31 * m23, c06 = m11 * m33 - m31 * m13, c07 = m11 * m23 - m21 * m13;
    float c08 = m21 * m32 - m31 * m22, c10 = m11 * m32 - m31 * m12, c11 = m11 * m22 - m21 * m12;
    float c12 = m20 * m33 - m30 * m23, c14 = m10 * m33 - m30 * m13, c15 = m10 * m23 - m20 * m13;
    float c16 = m20 * m32 - m30 * m22, c18 = m10 * m32 - m30 * m12, c19 = m10 * m22 - m20 * m12;
    float c20 = m20 * m31 - m30 * m21, c22 = m10 * m31 - m30 * m11, c23 = m10 * m21 - m20 * m11;
    float f0[4] = {c00, c00, c02, c03}, f1[4] = {c04, c04, c06, c07}, f2[4] = {c08, c08, c10, c11};
    float f3[4] = {c12, c12, c14, c15}, f4[4] = {c16, c16, c18, c19}, f5[4] = {c20, c20, c22, c23};
    float v0[4] = {m10, m00, m00, m00}, v1[4] = {m11, m01, m01, m01}, v2[4] = {m12, m02, m02, m02}, v3[4] = {m13, m03, m03, m03};
    float sa[4] = {1.f, -1.f, 1.f, -1.f}, sb[4] = {-1.f, 1.f, -1.f, 1.f};
    HM4 r;
    for (int k = 0; k < 4; k++) {
        r.m[k] = ((v1[k] * f0[k] - v2[k] * f1[k]) + v3[k] * f2[k]) * sa[k];
        r.m[4 + k] = ((v0[k] * f0[k] - v2[k] * f3[k]) + v3[k] * f4[k]) * sb[k];
        r.m[8 + k] = ((v0[k] * f1[k] - v1[k] * f3[k]) + v3[k] * f5[k]) * sa[k];
        r.m[12 + k] = ((v0[k] * f2[k] - v1[k] * f4[k]) + v2[k] * f5[k]) * sb[k];
    }
    float d0 = m[0] * r.m[0], d1 = m[1] * r.m[4], d2 = m[2] * r.m[8], d3 = m[3] * r.m[12];
    float det = d0 + d1 + d2 + d3;
    float rcp = 1.0f / det;
    for (int k = 0; k < 16; k++) r.m[k] = r.m[k] * rcp;
    return r;
}
// host powf(x, 2.0) == x*x exactly (Material::serialize, strolle/src/material.rs:39)

// ---- first-fit slot allocator (strolle/src/utils/allocator.rs) ----------------------------------------
struct SlotAllocator {
    struct Slot { size_t b, e; };
    std::vector<Slot> free_;
    bool unsorted = false;
    void give(size_t b, size_t e) { if (!free_.empty() && b <= free_.back().e) unsorted = true; free_.push_back({b, e}); }
    bool take(size_t n, size_t* b, size_t* e) {
        if (unsorted && !free_.empty()) {
            std::stable_sort(free_.begin(), free_.end(), [](const Slot& p, const Slot& q) { return p.b < q.b; });
            for (size_t i = 0; i + 1 < free_.size();) { if (free_[i].e == free_[i + 1].b) { free_[i].e = free_[i + 1].e; free_.erase(free_.begin() + i + 1); } else i++; }
        }
        unsorted = false;
        for (size_t i = 0; i < free_.size(); i++) {
            size_t len = free_[i].e - free_[i].b;
            if (len < n) continue;
            *b = free_[i].b; *e = free_[i].b + n;
            if (len == n) free_.erase(free_.begin() + i); else free_[i].b += n;
            return true;
        }
        return false;
    }
};

// ---- BVH: binned SAH build + DFS flatten (strolle/src/bvh/builder.rs, serializer.rs) ---------------------
struct Prim { uint32_t tri, mat; H3 center; Box box; };
struct BvhOut { std::vector<float4> buf; int depth = 0; };
class BvhBuild {
public:
    static const int kBins = 12;   // builder.rs:15
    struct Node { Box box; uint32_t b, e; int32_t left, right; uint64_t lhash, rhash; };
    std::vector<Node> nodes;
    std::vector<Prim> prims;
    // Last refresh's tree and primitive order (BvhPrimitives::previous, primitives.rs:63-65): the donor of subtrees whose
    // primitive-centre sequence is unchanged (builder.rs:245-275, SURVEY §8f-4).
    std::vector<Node> old_nodes;
    std::vector<Prim> old_prims;
    uint32_t grafted = 0;   // subtrees taken over by the last build
    bool finite = true;

    // `reuse` = the reference's behaviour.  A grafted subtree is the old one verbatim, including every field of its
    // primitives as they were when it was built: the hash covers the centres only (primitive.rs:27-37), so a primitive
    // whose centre is unchanged keeps its old triangle id, material id and bounds in the tree (quirk C-20).
    void build(const std::vector<Prim>& all, bool reuse = true) {
        old_nodes.swap(nodes); old_prims.swap(prims);
        prims.clear();
        finite = true;   // no NaN anywhere in the live primitives: the bounding-box updates may use plain selects
        for (const Prim& p : all) if (p.center.x != FMAX) {   // alive only (primitives.rs:58-61)
            prims.push_back(p);
            const float v[9] = {p.center.x, p.center.y, p.center.z, p.box.lo.x, p.box.lo.y, p.box.lo.z, p.box.hi.x, p.box.hi.y, p.box.hi.z};
            for (float f : v) if (f != f) finite = false;
        }
        nodes.clear(); grafted = 0;
        nodes.push_back(Node{Box(), 0u, (uint32_t)prims.size(), -1, -1, 0, 0});   // root bounds stay unset: SAH cost = +inf (quirk C-8)
        struct Item { int id, donor; };   // donor: node of the old tree at the same position, -1 = none
        std::deque<Item> work; work.push_back(Item{0, (reuse && !old_nodes.empty()) ? 0 : -1});
        while (!work.empty()) {
            Item it = work.front(); work.pop_front();
            int axis; float at, cost;
            if (!(finite ? best_plane<true>(it.id, &axis, &at, &cost) : best_plane<false>(it.id, &axis, &at, &cost))) continue;
            float leaf_cost = (float)(nodes[it.id].e - nodes[it.id].b) * nodes[it.id].box.half_area();
            if (!(cost < leaf_cost)) continue;
            if (finite) partition<true>(it.id, axis, at); else partition<false>(it.id, axis, at);
            const int li = nodes[it.id].left, ri = nodes[it.id].right;
            int ldonor = -1, rdonor = -1; bool lgraft = false, rgraft = false;
            if (it.donor >= 0 && old_nodes[it.donor].left >= 0) {
                const Node& d = old_nodes[it.donor];
                ldonor = d.left; rdonor = d.right;
                lgraft = d.lhash == nodes[it.id].lhash; rgraft = d.rhash == nodes[it.id].rhash;
            }
            if (lgraft) graft(li, ldonor); else work.push_back(Item{li, ldonor});
            if (rgraft) graft(ri, rdonor); else work.push_back(Item{ri, rdonor});
        }
    }
    void flatten(const std::vector<uint8_t>& alpha_blend, BvhOut* out) const { out->buf.clear(); out->depth = 0; emit(0, 1, alpha_blend, out); }

private:
    static float comp(H3 v, int a) { return a == 0 ? v.x : (a == 1 ? v.y : v.z); }
    template <bool FINITE> bool best_plane(int id, int* axis_out, float* at_out, float* cost_out) const {   // builder.rs:70-181
        const Node& nd = nodes[id];
        uint32_t n = nd.e - nd.b;
        if (n <= 1) return false;
        const Prim* p = prims.data() + nd.b;
        Box cb;
        for (uint32_t i = 0; i < n; i++) cb.add<FINITE>(p[i].center);
        H3 ext = cb.hi - cb.lo;
        H3 scale = h3((float)kBins / ext.x, (float)kBins / ext.y, (float)kBins / ext.z);
        Box bb[3][kBins]; uint32_t cnt[3][kBins] = {};
        for (uint32_t i = 0; i < n; i++) {
            H3 f = scale * (p[i].center - cb.lo);
            uint32_t id3[3] = {std::min(to_u32(f.x), (uint32_t)kBins - 1), std::min(to_u32(f.y), (uint32_t)kBins - 1), std::min(to_u32(f.z), (uint32_t)kBins - 1)};
            for (int a = 0; a < 3; a++) { cnt[a][id3[a]] += 1; bb[a][id3[a]].add<FINITE>(p[i].box); }
        }
        float la[3][kBins - 1], ra[3][kBins - 1]; uint32_t lc[3][kBins - 1], rc[3][kBins - 1];
        for (int a = 0; a < 3; a++) {
            Box lb, rb; uint32_t ln = 0, rn = 0;
            for (int i = 0; i < kBins - 1; i++) {
                ln += cnt[a][i]; lc[a][i] = ln;
                if (bb[a][i].set()) lb.add<FINITE>(bb[a][i]);
                la[a][i] = lb.half_area();
                rn += cnt[a][kBins - 1 - i]; rc[a][kBins - 2 - i] = rn;
                if (bb[a][kBins - 1 - i].set()) rb.add<FINITE>(bb[a][kBins - 1 - i]);
                ra[a][kBins - 2 - i] = rb.half_area();
            }
        }
        bool any = false; float best = 0.f;
        H3 step = h3(ext.x / (float)kBins, ext.y / (float)kBins, ext.z / (float)kBins);
        for (int a = 0; a < 3; a++) for (int i = 0; i < kBins - 1; i++) {
            float c = (float)lc[a][i] * la[a][i] + (float)rc[a][i] * ra[a][i];
            if (!any || c <= best) {   // NaN costs stick once taken (quirk C-7)
                any = true; best = c; *axis_out = a; *at_out = comp(cb.lo, a) + comp(step, a) * (float)(i + 1);
            }
        }
        *cost_out = best;
        return any;
    }
    // fxhash 0.2.1 FxHasher (64-bit) over the centre bits of each primitive, in the order the partition meets them
    // (builder.rs:201-228, primitive.rs:27-37); third-party crate, restated from its published definition.
    static void fx(uint64_t* h, uint32_t w) { *h = (((*h << 5) | (*h >> 59)) ^ (uint64_t)w) * 0x517cc1b727220a95ull; }
    static void fx_prim(uint64_t* h, const Prim& p) { fx(h, f2bits(p.center.x)); fx(h, f2bits(p.center.y)); fx(h, f2bits(p.center.z)); }
    template <bool FINITE> void partition(int id, int axis, float at) {   // builder.rs:183-319
        uint32_t b = nodes[id].b, e = nodes[id].e;
        Prim* d = prims.data() + b;
        int l = 0, r = (int)(e - b) - 1;
        Box lb, rb; uint64_t lh = 0, rh = 0;
        while (l <= r) {
            Prim cur = d[l];
            if (comp(cur.center, axis) < at) { l++; lb.add<FINITE>(cur.box); fx_prim(&lh, cur); }
            else { std::swap(d[l], d[r]); r--; rb.add<FINITE>(cur.box); fx_prim(&rh, cur); }
        }
        uint32_t mid = b + (uint32_t)l;
        int li = (int)nodes.size(); nodes.push_back(Node{lb, b, mid, -1, -1, 0, 0});
        int ri = (int)nodes.size(); nodes.push_back(Node{rb, mid, e, -1, -1, 0, 0});
        nodes[id].left = li; nodes[id].right = ri; nodes[id].lhash = lh; nodes[id].rhash = rh;
    }
    // builder.rs:321-359 (copy + offset_primitives): node `id` (a fresh leaf over [b, e)) becomes the old subtree `donor`,
    // shifted to this range, and the range gets the old subtree's primitives in their old order.
    void graft(int id, int donor) {
        const Node& src = old_nodes[donor];
        const uint32_t b = nodes[id].b;
        for (uint32_t i = src.b; i < src.e; i++) prims[b + (i - src.b)] = old_prims[i];
        grafted++;
        struct Pair { int dst, src; };
        std::vector<Pair> todo; todo.push_back(Pair{id, donor});
        const int64_t shift = (int64_t)b - (int64_t)src.b;
        while (!todo.empty()) {
            Pair pr = todo.back(); todo.pop_back();
            const Node o = old_nodes[pr.src];
            Node n = o; n.b = (uint32_t)((int64_t)o.b + shift); n.e = (uint32_t)((int64_t)o.e + shift); n.left = n.right = -1;
            if (o.left >= 0) {
                n.left = (int)nodes.size(); nodes.push_back(Node{}); n.right = (int)nodes.size(); nodes.push_back(Node{});
                todo.push_back(Pair{n.left, o.left}); todo.push_back(Pair{n.right, o.right});
            }
            nodes[pr.dst] = n;
        }
    }
    uint32_t emit(int id, int depth, const std::vector<uint8_t>& alpha, BvhOut* out) const {   // serializer.rs:20-110
        uint32_t at = (uint32_t)out->buf.size();
        if (depth > out->depth) out->depth = depth;
        const Node& nd = nodes[id];
        if (nd.left >= 0) {
            out->buf.resize(out->buf.size() + 4, make_float4(0, 0, 0, 0));
            emit(nd.left, depth + 1, alpha, out);
            uint32_t rp = emit(nd.right, depth + 1, alpha, out);
            const Box& lb = nodes[nd.left].box; const Box& rb = nodes[nd.right].box;
            out->buf[at] = make_float4(lb.lo.x, lb.lo.y, lb.lo.z, bits2f(0u));
            out->buf[at + 1] = make_float4(lb.hi.x, lb.hi.y, lb.hi.z, bits2f(rp));
            out->buf[at + 2] = make_float4(rb.lo.x, rb.lo.y, rb.lo.z, 0.0f);
            out->buf[at + 3] = make_float4(rb.hi.x, rb.hi.y, rb.hi.z, 0.0f);
        } else {
            uint32_t n = nd.e - nd.b;
            for (uint32_t i = 0; i < n; i++) {
                const Prim& p = prims[nd.b + i];
                uint32_t flags = (i + 1 < n ? 1u : 0u) | ((alpha[p.mat] ? 1u : 0u) << 1);
                out->buf.push_back(make_float4(bits2f(flags), bits2f(p.tri), bits2f(p.mat), bits2f(1u)));
            }
        }
        return at;
    }
};

// ---- device buffer helper ------------------------------------------------------------------------------
struct DevMem {
    void* p = nullptr; size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return ST_OK;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = std::max<size_t>(bytes, 256);
        CK(cudaMalloc(&p, want));
        CK(cudaMemset(p, 0, want));
        CK(cudaDeviceSynchronize());   // the fill runs on the legacy stream; engine streams are non-blocking
        cap = want;
        return ST_OK;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

static const char* kPassNames[P_COUNT] = {
    "prim_gbuffer", "di_sampling", "di_temporal_resampling", "di_spatial_resampling_pick", "di_spatial_resampling_trace", "di_spatial_resampling_sample",
    "di_resolving", "gi_reprojection", "gi_sampling_a", "gi_sampling_b", "gi_temporal_resampling", "gi_spatial_resampling_pick",
    "gi_spatial_resampling_trace", "gi_spatial_resampling_sample", "gi_preview_resampling", "gi_resolving", "frame_reprojection",
    "frame_denoising_reproject", "frame_denoising_estimate_variance", "frame_denoising_wavelet", "frame_composition", "ref_tracing",
    "ref_shading", "bvh_heatmap", "atmosphere", "trace_stream", "halo_exchange"};

static uint32_t dispatch_seed(uint32_t base, uint32_t frame, uint32_t k) {
    uint32_t s = base ^ (frame * 64u + k);
    s = s * 747796405u + 2891336453u;
    uint32_t w = ((s >> ((s >> 28) + 4u)) ^ s) * 277803737u;
    return (w >> 22) ^ w;
}

static_assert(OUT_RGBA32F == ST_FORMAT_RGBA32F && OUT_RGBA8_SRGB == ST_FORMAT_RGBA8_SRGB && OUT_RGBA16F == ST_FORMAT_RGBA16F, "kernel output formats follow the C ABI");
// bytes per pixel of an output format; 0 = not a format
static size_t format_bpp(int format) { return format == ST_FORMAT_RGBA32F ? 16 : format == ST_FORMAT_RGBA16F ? 8 : format == ST_FORMAT_RGBA8_SRGB ? 4 : 0; }
// the widest format that is converted through the staging buffer (RGBA32F leaves straight from `output`)
static const size_t kStagingBpp = 8;

struct CameraSlot {
    bool alive = false;
    st_camera desc;
    uint32_t frame = 0;
    CameraDev dev;
    std::vector<std::pair<std::string, float4**>> named;   // buffer name -> pointer slot in `dev`
    std::vector<std::pair<std::string, size_t>> sizes;      // float4 count per named buffer
    DevMem arena;
    DevMem svgf_pairs; float4* pair[2] = {nullptr, nullptr};   // interleaved {DI, GI} records of the wide-stride à-trous iterations (ST_OPT_WAVELET_PAIRED); private scratch, never exchanged
    // converted frames on their way to host memory or to rank 0 of a strip gather: two frame-sized slots of kStagingBpp bytes per pixel,
    // allocated at that size from the start because the buffer is exported to the other ranks (a later growth would leave their mappings stale)
    DevMem staging; int staging_slot = 0;
    // asynchronous read-back: slot k of the staging buffer is converted on the engine stream (ev_ready[k]) and copied to
    // the host on the copy stream (ev_copied[k]); the engine stream only waits for ev_copied[k] before reusing slot k
    cudaEvent_t ev_ready[2] = {nullptr, nullptr}, ev_copied[2] = {nullptr, nullptr};
    // peer-memory link of the strip partition: other ranks' arena / flag / staging allocations mapped through CUDA IPC
    // sync words: [0, 128) fused-transport flags (slot * 16 + source rank), 128.. legacy k_peer_exchange flags, 144 its block counter,
    // 145 its time-outs, 200/201 need_rows {min, max}, 202 fused-transport wait time-outs, 204 (u64) rows pulled
    // copy-engine pushes of the large GI halos (ST_OPT_STRIP_DMA): one side stream per neighbour (0 = up, 1 = down), `pushed` = the last push issued there
    cudaStream_t side[2] = {nullptr, nullptr}; cudaEvent_t ev_produced = nullptr, ev_pushed[2] = {nullptr, nullptr}; bool pushed_pending[2] = {false, false};
    struct PeerLink { bool ready = false; bool ipc = false; std::vector<char*> arena, staging; std::vector<uint32_t*> flags; DevMem sync; uint32_t seq = 0, fseq = 0; } peer;
};

struct Step { int pass; std::function<void(cudaStream_t)> run; int sub = -1; };   // sub: à-trous iteration of a K22 step

}  // namespace st

using namespace st;

struct st_engine {
    int device = 0;
    cudaStream_t stream = nullptr; bool own_stream = true;
    cudaStream_t copy_stream = nullptr;   // device->host copies of finished frames (ST_OPT_ASYNC_OUTPUT), so that they overlap the next frame
    // meshes / materials / instances / triangles -------------------------------------------------
    std::unordered_map<st_handle, std::vector<st_mesh_triangle>> meshes;
    std::vector<st_material> materials; std::vector<st_handle> material_handles; bool materials_dirty = false;
    struct MatTex { st_handle tex[4]; uint32_t mask; };
    std::vector<MatTex> material_textures;
    // images (strolle/src/images.rs): shelf allocator in place of the guillotiere crate; only the rect handed to the
    // materials (Images::lookup) is visible to the kernels
    struct ImageRect { st_handle handle; uint32_t x, y, w, h; };
    std::vector<ImageRect> images; uint32_t shelf_x = 0, shelf_y = 0, shelf_h = 0; bool images_dirty = false;
    // dynamic images (st_insert_dynamic_image): at each tick, before anything else the tick enqueues, every surface is copied into its image's
    // rectangle.  `src` = the address this device reads (device, peer, managed, or the device pointer of page-locked host memory).
    struct DynImage { st_handle handle; const char* src; size_t pitch; };
    std::vector<DynImage> dynamic;
    cudaEvent_t ev_output = nullptr;   // recorded on copy_stream: the refresh waits for queued output copies into host surfaces
    cudaEvent_t ev_queued = nullptr;   // recorded on `stream` by st_multi_tick: the other members' refreshes wait for this member's row stores
    DevMem d_atlas, d_srgb, d_tri_instance, d_instance_xforms;
    bool motion_dirty = true;
    bool moved_last_tick = false;   // an instance was inserted / moved / removed in the tick that prepared the current frame
    struct Inst { st_handle handle, mesh, material; Affine3 xf, xf_inv, prev_xf; bool dirty; };
    std::vector<Inst> instances; bool instances_dirty = false;
    struct Range { st_handle handle; size_t b, e; };
    std::vector<Range> tri_ranges; SlotAllocator tri_alloc;
    std::vector<float4> h_triangles; std::vector<Prim> prims; bool triangles_dirty = false;
    BvhBuild bvh; BvhOut bvh_out; bool bvh_dirty = false;
    std::vector<GpuMaterial> h_materials;
    // lights (strolle/src/lights.rs): slot 0 is the sun ------------------------------------------
    static const st_handle kSun = ~(st_handle)0;
    std::vector<GpuLight> h_lights; std::vector<std::pair<st_handle, uint32_t>> light_slots;
    std::vector<st_handle> lights_created, lights_updated; std::vector<std::pair<st_handle, uint32_t>> lights_remapped; std::vector<uint32_t> lights_killed;
    uint32_t next_light = 1; bool lights_dirty = true;
    float sun_azimuth = 0.0f, sun_altitude = 0.35f; bool sun_dirty = true;
    GpuWorld world;
    uint32_t frame = 1, seed_base = 0xC0FFEEu;
    // device scene ------------------------------------------------------------------------------
    DevMem d_triangles, d_bvh, d_materials, d_matpacked, d_unpacklut, d_lights, d_noise, d_tlut, d_slut, d_skylut, d_scratch, d_raycount;
    bool count_rays = false;
    bool svgf_fast = true;   // ST_OPT_SVGF_FAST_MATH
    bool shading_fast = ST_SHADING_FAST_DEFAULT != 0;   // ST_OPT_SHADING_FAST_MATH
    bool fused_passes = ST_FUSED_PASSES_DEFAULT != 0;   // ST_OPT_FUSED_PASSES
    bool async_output = false;   // ST_OPT_ASYNC_OUTPUT
    bool halo_nccl = false;      // ST_OPT_HALO_NCCL
    int wavelet_paired = ST_WAVELET_PAIRED_DEFAULT;   // ST_OPT_WAVELET_PAIRED
    int strip_dma = ST_STRIP_DMA_DEFAULT;   // ST_OPT_STRIP_DMA: 1 = gi_reservoirs[1] / [2] halo rows by copy engine on side streams instead of in-kernel mirror stores; 2 = also the G-buffer halo rows (instead of recomputing them); 3 = also di_reservoirs[1] and gi_reservoirs[3]; -1 = 1 for two strips, 2 from three on
    bool strip_fused = true;     // ST_OPT_STRIP_FUSED: mirror stores + neighbour flags + recompute instead of stand-alone exchanges
    bool last_frame_fused = false;
    int wavelet_tiled = ST_WAVELET_TILED_DEFAULT;   // ST_OPT_WAVELET_TILED: bit i = à-trous iteration i (stride 2^i) runs the tile-staged (TMA) kernel
    int wavelet_cfg = ST_WAVELET_CFG_DEFAULT;       // ST_OPT_WAVELET_TILE_CFG: 4 bits per iteration, tile shape index (kernels.cu wavelet_tiled_cfg)
    DevMem d_tile_errors; uint64_t wavelet_tiled_launches = 0;
    bool fuse_reproject = ST_FUSE_REPROJECT_DEFAULT != 0;   // ST_OPT_FUSE_REPROJECT
    bool bvh_reuse = true;   // ST_OPT_BVH_REUSE
    bool variance_tiled = ST_VARIANCE_TILED_DEFAULT != 0; uint64_t variance_tiled_launches = 0;   // ST_OPT_VARIANCE_TILED
    bool luts_static_ready = false, sky_ready = false; float sky_for_altitude = 0.0f;
    std::vector<CameraSlot*> cameras;
    // timing ---------------------------------------------------------------------------------------
    bool timing = false;
    float pass_ms[P_COUNT] = {}; uint32_t pass_launches[P_COUNT] = {};
    float wavelet_ms[5] = {}; uint32_t wavelet_launches[5] = {};   // K22 per à-trous iteration (st_wavelet_times)
    struct Timed { int pass; cudaEvent_t a, b; int sub; };
    std::vector<Timed> pending; std::vector<cudaEvent_t> event_pool;
    cudaEvent_t mark_a = nullptr, mark_b = nullptr;
    // row-strip partition (SURVEY §8e): NCCL communicator over the ranks that share the frame
    ncclComm_t comm = nullptr; int rank = 0, n_ranks = 1;
    uint64_t halo_bytes_last_frame = 0;

    SceneDev scene() const {
        SceneDev s;
        s.triangles = (const float4*)d_triangles.p; s.bvh = (const float4*)d_bvh.p; s.bvh_len = (uint32_t)bvh_out.buf.size(); s.materials = (const GpuMaterial*)d_materials.p;
        s.lights = (const GpuLight*)d_lights.p; s.blue_noise = (const uchar4*)d_noise.p;
        s.transmittance_lut = (const float4*)d_tlut.p; s.scattering_lut = (const float4*)d_slut.p; s.sky_lut = (const float4*)d_skylut.p;
        s.world = world;
        s.tri_instance = (const uint32_t*)d_tri_instance.p; s.instance_xforms = (const float4*)d_instance_xforms.p;
        s.atlas = (const uchar4*)d_atlas.p; s.srgb_lut = (const float*)d_srgb.p;
        s.material_packed = (const uint32_t*)d_matpacked.p; s.unpack_lut = (const float*)d_unpacklut.p;
        s.ray_counter = count_rays ? (unsigned long long*)d_raycount.p : nullptr;
        return s;
    }
    uint32_t* light_slot(st_handle h) { for (auto& p : light_slots) if (p.first == h) return &p.second; return nullptr; }
    cudaEvent_t get_event() { if (!event_pool.empty()) { cudaEvent_t e = event_pool.back(); event_pool.pop_back(); return e; } cudaEvent_t e; cudaEventCreate(&e); return e; }
    void run_timed(int pass, const std::function<void(cudaStream_t)>& fn, int sub = -1) {
        if (!timing) { fn(stream); pass_launches[pass]++; return; }
        Timed t; t.pass = pass; t.sub = sub; t.a = get_event(); t.b = get_event();
        cudaEventRecord(t.a, stream); fn(stream); cudaEventRecord(t.b, stream);
        pending.push_back(t); pass_launches[pass]++;
    }
    void collect_timing() {
        for (Timed& t : pending) { cudaEventSynchronize(t.b); float ms = 0; cudaEventElapsedTime(&ms, t.a, t.b); pass_ms[t.pass] += ms; if (t.pass == P_DENOISE_WAVELET && t.sub >= 0 && t.sub < 5) { wavelet_ms[t.sub] += ms; wavelet_launches[t.sub]++; } event_pool.push_back(t.a); event_pool.push_back(t.b); }
        pending.clear();
    }
};

namespace st {

static GpuLight make_sun(float4 d0, float4 d1) {   // strolle-gpu/src/light.rs:49-65
    GpuLight l; std::memset(&l, 0, sizeof l); l.d0 = d0; l.d1 = d1; l.d2 = make_float4(bits2f(1u), 0, 0, 0); return l;
}
static void uniq_add(std::vector<st_handle>& v, st_handle h) { if (std::find(v.begin(), v.end(), h) == v.end()) v.push_back(h); }
static void uniq_del(std::vector<st_handle>& v, st_handle h) { v.erase(std::remove(v.begin(), v.end(), h), v.end()); }

static void light_overwrite(st_engine* e, uint32_t slot, st_handle h, GpuLight nl) {   // Lights::update (lights.rs:168-182)
    const GpuLight& old = e->h_lights[slot];
    nl.prev_d0 = old.d0; nl.prev_d1 = old.d1; nl.prev_d2 = old.d2;
    uniq_add(e->lights_updated, h);
    e->h_lights[slot] = nl; e->lights_dirty = true;
}

static float2 oct_encode_host(H3 n) {   // strolle-gpu/src/normal.rs:9-23 (spot light direction)
    float s = std::fabs(n.x) + std::fabs(n.y) + std::fabs(n.z);
    n = n / s;
    float2 r;
    if (n.z >= 0.0f) r = make_float2(n.x, n.y);
    else r = make_float2(std::copysign(1.0f - std::fabs(n.y), n.x), std::copysign(1.0f - std::fabs(n.x), n.y));
    return make_float2(r.x * 0.5f + 0.5f, r.y * 0.5f + 0.5f);
}

// world-space bake of one mesh triangle (strolle/src/mesh_triangle.rs:47-86) + serialisation
// (strolle/src/triangle.rs:16-38)
static void bake_triangle(const st_mesh_triangle& t, const Affine3& xf, const Affine3& inv, float4* out9, Prim* prim) {
    Affine3 nt;   // transpose of inv's 3x3
    nt.x = h3(inv.x.x, inv.y.x, inv.z.x); nt.y = h3(inv.x.y, inv.y.y, inv.z.y); nt.z = h3(inv.x.z, inv.y.z, inv.z.z); nt.t = h3(0, 0, 0);
    float det = hdot(xf.z, hcross(xf.x, xf.y));
    float sign = (f2bits(det) >> 31) ? -1.0f : 1.0f;
    H3 pos[3];
    for (int k = 0; k < 3; k++) {
        pos[k] = aff_point(xf, h3(t.positions[k][0], t.positions[k][1], t.positions[k][2]));
        H3 n = hnorm(aff_mat(nt, h3(t.normals[k][0], t.normals[k][1], t.normals[k][2])));
        H3 tg = hnorm(aff_mat(xf, h3(t.tangents[k][0], t.tangents[k][1], t.tangents[k][2])));
        out9[3 * k] = make_float4(pos[k].x, pos[k].y, pos[k].z, t.uvs[k][0]);
        out9[3 * k + 1] = make_float4(n.x, n.y, n.z, t.uvs[k][1]);
        out9[3 * k + 2] = make_float4(tg.x, tg.y, tg.z, t.tangents[k][3] * sign);
    }
    prim->center = (((h3(0, 0, 0) + pos[0]) + pos[1]) + pos[2]) / 3.0f;
    prim->box = Box();
    for (int k = 0; k < 3; k++) prim->box.grow(pos[k]);
}

static void release_range(st_engine* e, st_handle inst) {   // Triangles::remove (triangles.rs:157-171)
    for (size_t i = 0; i < e->tri_ranges.size(); i++) if (e->tri_ranges[i].handle == inst) {
        e->tri_alloc.give(e->tri_ranges[i].b, e->tri_ranges[i].e);
        for (size_t t = e->tri_ranges[i].b; t < e->tri_ranges[i].e; t++) e->prims[t].center = h3(FMAX, FMAX, FMAX);
        e->tri_ranges.erase(e->tri_ranges.begin() + i);
        return;
    }
}

// Instances::refresh (instances.rs:69-139) in instance-insertion order
static bool refresh_instances(st_engine* e) {
    if (!e->instances_dirty) return false;
    e->instances_dirty = false;
    for (auto& in : e->instances) {
        if (!in.dirty) continue;
        in.dirty = false;
        auto mesh = e->meshes.find(in.mesh);
        auto mat = std::find(e->material_handles.begin(), e->material_handles.end(), in.material);
        if (mesh == e->meshes.end() || mat == e->material_handles.end()) { in.dirty = true; e->instances_dirty = true; continue; }   // retried next tick
        uint32_t mat_id = (uint32_t)(mat - e->material_handles.begin());
        const std::vector<st_mesh_triangle>& tris = mesh->second;
        st_engine::Range* have = nullptr;
        for (auto& r : e->tri_ranges) if (r.handle == in.handle) have = &r;
        size_t b, en;
        if (have && have->e - have->b == tris.size()) { b = have->b; en = have->e; }
        else {
            if (have) release_range(e, in.handle);
            if (!e->tri_alloc.take(tris.size(), &b, &en)) {
                b = e->h_triangles.size() / 9; en = b + tris.size();
                e->h_triangles.resize(9 * en, make_float4(0, 0, 0, 0));
                e->prims.resize(en);
            }
            e->tri_ranges.push_back({in.handle, b, en});
        }
        for (size_t i = 0; i < tris.size(); i++) {
            Prim& p = e->prims[b + i];
            p.tri = (uint32_t)(b + i); p.mat = mat_id;
            bake_triangle(tris[i], in.xf, in.xf_inv, &e->h_triangles[9 * (b + i)], &p);
        }
        e->triangles_dirty = true;
    }
    return true;
}

static int upload(st_engine* e, DevMem& d, const void* src, size_t bytes) {
    int rc = d.ensure(bytes); if (rc) return rc;
    if (bytes) CK(cudaMemcpyAsync(d.p, src, bytes, cudaMemcpyHostToDevice, e->stream));
    return ST_OK;
}

static int ensure_luts(st_engine* e) {   // AtmospherePass::run (passes/atmosphere.rs:67-111)
    int rc;
    if (!e->luts_static_ready) {
        if ((rc = e->d_tlut.ensure(256 * 64 * 16))) return rc;
        if ((rc = e->d_slut.ensure(32 * 32 * 16))) return rc;
        if ((rc = e->d_skylut.ensure(256 * 256 * 16))) return rc;
        e->run_timed(P_ATMOSPHERE, [&](cudaStream_t s) { launch_atm_transmittance((float4*)e->d_tlut.p, s); launch_atm_scattering((const float4*)e->d_tlut.p, (float4*)e->d_slut.p, s); });
        e->luts_static_ready = true;
    }
    if (!e->sky_ready || e->sky_for_altitude != e->world.sun_altitude) {   // one source of truth: the altitude st_tick published in `world`
        float alt = e->world.sun_altitude;
        e->run_timed(P_ATMOSPHERE, [&](cudaStream_t s) { launch_atm_sky((const float4*)e->d_tlut.p, (const float4*)e->d_slut.p, alt, (float4*)e->d_skylut.p, s); });
        e->sky_ready = true; e->sky_for_altitude = alt;
    }
    return ST_OK;
}

static GpuCamera serialize_camera(const st_camera& c) {   // Camera::serialize (strolle/src/camera.rs:50-66)
    HM4 t, p; std::memcpy(t.m, c.transform, 64); std::memcpy(p.m, c.projection, 64);
    HM4 pv = hm_mul(p, hm_inverse(t)), n2w = hm_mul(t, hm_inverse(p));
    GpuCamera g;
    std::memcpy(g.projection_view, pv.m, 64); std::memcpy(g.ndc_to_world, n2w.m, 64);
    g.origin = make_float4(c.transform[12], c.transform[13], c.transform[14], 0.0f);
    g.screen = make_float4((float)c.width, (float)c.height, 0.0f, 0.0f);
    return g;
}

// CameraBuffers::new (strolle/src/camera_controller/buffers.rs:53-339): one zero-filled arena
static int allocate_camera(st_engine* e, CameraSlot* cs) {
    CameraDev& d = cs->dev;
    size_t n = (size_t)cs->desc.width * cs->desc.height;
    cs->named.clear(); cs->sizes.clear();
    auto reg = [&](const char* name, float4** slot, size_t count) { cs->named.push_back({name, slot}); cs->sizes.push_back({name, count}); };
    reg("prim_gbuffer_d0_a", &d.prim_gbuffer_d0[0], n); reg("prim_gbuffer_d0_b", &d.prim_gbuffer_d0[1], n);
    reg("prim_gbuffer_d1_a", &d.prim_gbuffer_d1[0], n); reg("prim_gbuffer_d1_b", &d.prim_gbuffer_d1[1], n);
    reg("prim_surface_map_a", &d.prim_surface_map[0], n); reg("prim_surface_map_b", &d.prim_surface_map[1], n);
    reg("reprojection_map", &d.reprojection_map, n); reg("velocity_map", &d.velocity_map, n);
    reg("di_reservoirs_0", &d.di_reservoirs[0], 2 * n); reg("di_reservoirs_1", &d.di_reservoirs[1], 2 * n); reg("di_reservoirs_2", &d.di_reservoirs[2], 2 * n);
    reg("di_diff_samples", &d.di_diff_samples, n); reg("di_diff_prev_colors", &d.di_diff_prev_colors, n); reg("di_diff_curr_colors", &d.di_diff_curr_colors, n);
    reg("di_diff_moments_a", &d.di_diff_moments[0], n); reg("di_diff_moments_b", &d.di_diff_moments[1], n); reg("di_diff_stash", &d.di_diff_stash, n);
    reg("di_spec_samples", &d.di_spec_samples, n);
    reg("gi_d0", &d.gi_d0, n); reg("gi_d1", &d.gi_d1, n); reg("gi_d2", &d.gi_d2, n);
    reg("gi_reservoirs_0", &d.gi_reservoirs[0], 4 * n); reg("gi_reservoirs_1", &d.gi_reservoirs[1], 4 * n);
    reg("gi_reservoirs_2", &d.gi_reservoirs[2], 4 * n); reg("gi_reservoirs_3", &d.gi_reservoirs[3], 4 * n);
    reg("gi_diff_samples", &d.gi_diff_samples, n); reg("gi_diff_prev_colors", &d.gi_diff_prev_colors, n); reg("gi_diff_curr_colors", &d.gi_diff_curr_colors, n);
    reg("gi_diff_moments_a", &d.gi_diff_moments[0], n); reg("gi_diff_moments_b", &d.gi_diff_moments[1], n); reg("gi_diff_stash", &d.gi_diff_stash, n);
    reg("gi_spec_samples", &d.gi_spec_samples, n);
    reg("ref_hits", &d.ref_hits, 2 * n); reg("ref_rays", &d.ref_rays, 3 * n); reg("ref_colors", &d.ref_colors, n);
    reg("prim_triangle_ids", &d.prim_triangle_ids, n); reg("surface_nd", &d.surface_nd, n); reg("output", &d.output, n);
    size_t total = 0;
    for (auto& s : cs->sizes) total += (s.second * 16 + 255) / 256 * 256;
    cs->arena.release();
    int rc = cs->arena.ensure(total); if (rc) return rc;
    CK(cudaMemsetAsync(cs->arena.p, 0, total, e->stream));
    const size_t pair_bytes = (2 * n * 16 + 255) / 256 * 256;
    cs->svgf_pairs.release();
    if ((rc = cs->svgf_pairs.ensure(2 * pair_bytes))) return rc;
    CK(cudaMemsetAsync(cs->svgf_pairs.p, 0, 2 * pair_bytes, e->stream));
    cs->pair[0] = (float4*)cs->svgf_pairs.p; cs->pair[1] = (float4*)((char*)cs->svgf_pairs.p + pair_bytes);
    size_t off = 0;
    for (size_t i = 0; i < cs->named.size(); i++) { *cs->named[i].second = (float4*)((char*)cs->arena.p + off); off += (cs->sizes[i].second * 16 + 255) / 256 * 256; }
    d.w = (int)cs->desc.width; d.h = (int)cs->desc.height; d.y0 = 0; d.y1 = d.h;
    d.own_y0 = 0; d.own_y1 = d.h; d.mirror_up = 0; d.mirror_dn = 0; d.need_rows = nullptr; d.gi_mirror_reach = 128; d.di_mirror_reach = 128;
    return ST_OK;
}

// CameraController::render (strolle/src/camera_controller.rs:87-174) as an explicit step list
// Rows a pass computes beyond the owned strip [y0, y1) in a strip-partitioned frame (fused transport): the G-buffer pass recomputes the
// rows its neighbours' spatial taps reach, K21 / K22 recompute the rows the following à-trous iterations read, so that none of
// those buffers has to travel.  All zero = every pass runs on [y0, y1).
struct StripExt { int gbuffer = 0, variance = 0, wavelet[5] = {0, 0, 0, 0, 0}; int preview_mirror[2] = {0, 0}; bool still = false; /* nothing moved: no rows of last frame are pulled */ };
static CameraDev grown(const CameraDev& c, int rows) { CameraDev g = c; g.y0 = std::max(0, c.y0 - rows); g.y1 = std::min(c.h, c.y1 + rows); return g; }
// camera `c` as a view of a launch whose view 0 is `first` (same size: the arenas have the same layout), rows grown by `rows`
static ViewDev view_of(const CameraSlot* c, const CameraSlot* first, int rows) {
    ViewDev v; v.cam = grown(c->dev, rows);
    v.arena_delta = (const char*)c->arena.p - (const char*)first->arena.p; v.pair_delta = (const char*)c->svgf_pairs.p - (const char*)first->svgf_pairs.p;
    v.dst = nullptr; v.pitch = 0;
    return v;
}
typedef std::shared_ptr<const ViewSet> Views;
// `group`: one camera, or up to kBatchViews cameras of one size, mode, denoise and ref_depth rendered after the same tick (they share the
// frame id, hence every pass, seed and buffer parity), each pass one launch over all of them.  Pointer arguments are group[0]'s.
static void build_schedule(st_engine* e, const std::vector<CameraSlot*>& group, std::vector<Step>* steps, const StripExt* ext = nullptr) {
    CameraSlot* cs = group[0];
    const CameraDev cam = cs->dev;   // snapshot (pointers + cameras)
    const StripExt no_ext; const StripExt& x = ext ? *ext : no_ext;
    auto views = [&](int rows) { auto v = std::make_shared<ViewSet>(); for (CameraSlot* c : group) v->push_back(view_of(c, cs, rows)); return Views(v); };
    const Views V = views(0), VG = views(x.gbuffer), VV = views(x.variance);
    const bool one = group.size() == 1;   // the tile-staged K21 / K22 encode one camera's planes; several views run the gather kernels (same bits)
    const int pm0 = x.preview_mirror[0], pm1 = x.preview_mirror[1];
    const SceneDev sc = e->scene();
    const uint32_t f = cs->frame;
    const int cur = (f % 2u) == 1u ? 1 : 0;   // is_alternate (camera_controller.rs:185-187)
    const st_camera& d = cs->desc;
    const bool fs = e->shading_fast;   // ReSTIR kernels from the fast-shading build (ST_OPT_SHADING_FAST_MATH)
    auto seed = [&](uint32_t k) { return dispatch_seed(e->seed_base, f, k); };
    auto add = [&](int pass, std::function<void(cudaStream_t)> fn) { steps->push_back(Step{pass, std::move(fn)}); };
    const float4* di_final = (d.denoise && (d.mode == ST_MODE_IMAGE || d.mode == ST_MODE_DI_DIFFUSE)) ? cam.di_diff_curr_colors : cam.di_diff_samples;
    const float4* gi_final = (d.denoise && (d.mode == ST_MODE_IMAGE || d.mode == ST_MODE_GI_DIFFUSE)) ? cam.gi_diff_curr_colors : cam.gi_diff_samples;
    if (d.mode == ST_MODE_BVH_HEATMAP) {
        add(P_BVH_HEATMAP, [=](cudaStream_t s) { launch_bvh_heatmap(*V, sc, s); });
        add(P_COMPOSITION, [=](cudaStream_t s) { launch_composition(*V, sc, cur, 5u, di_final, gi_final, s); });
        return;
    }
    if (d.mode == ST_MODE_REFERENCE) {
        for (uint32_t depth = 0; depth <= (uint32_t)d.ref_depth; depth++) {
            uint32_t sd = seed(P_REF_SHADING_SEED + depth);
            add(P_REF_TRACING, [=](cudaStream_t s) { launch_ref_tracing(*V, sc, depth, s); });
            add(P_REF_SHADING, [=](cudaStream_t s) { launch_ref_shading(*V, sc, sd, depth, s); });
        }
        add(P_REF_SHADING, [=](cudaStream_t s) { launch_ref_shading(*V, sc, 0u, 255u, s); });
        add(P_COMPOSITION, [=](cudaStream_t s) { launch_composition(*V, sc, cur, 6u, di_final, gi_final, s); });
        return;
    }
    const bool needs_di = d.mode == ST_MODE_IMAGE || d.mode == ST_MODE_DI_DIFFUSE || d.mode == ST_MODE_DI_SPECULAR;
    const bool needs_gi = d.mode == ST_MODE_IMAGE || d.mode == ST_MODE_GI_DIFFUSE || d.mode == ST_MODE_GI_SPECULAR;
    // K4 inside the G-buffer launch: only where nothing has to happen between the two (a strip pulls last frame's rows in between,
    // unless nothing moved: then every reprojected read is the pixel itself)
    const int k4_in_k0 = (e->fused_passes && (ext == nullptr || ext->still) && !e->instances.empty()) ? 1 : 0;
    add(P_PRIM_GBUFFER, [=](cudaStream_t s) { launch_prim_gbuffer(*VG, sc, cur, k4_in_k0, s); });
    // ST_OPT_FUSED_PASSES: passes whose hand-over is private to a pixel (or to a checkerboard pair) run as one launch; the step keeps
    // the pass id of the member that gathers from other pixels, which is what the strip plans key on.
    const bool fp = e->fused_passes;
    if (!e->instances.empty()) {
        if (!k4_in_k0) add(P_FRAME_REPROJECTION, [=](cudaStream_t s) { launch_frame_reprojection(*V, sc, cur, s); });
        if (needs_di) {
            uint32_t s1 = seed(P_DI_SAMPLING), s2 = seed(P_DI_TEMPORAL), s3 = seed(P_DI_SPATIAL_PICK), s5 = seed(P_DI_SPATIAL_SAMPLE);
            if (fp) {
                add(P_DI_TEMPORAL, [=](cudaStream_t s) { (fs ? stf::launch_di_sample_temporal : st::launch_di_sample_temporal)(*V, sc, cur, s1, s2, f, s); });
                add(P_DI_SPATIAL_PICK, [=](cudaStream_t s) { (fs ? stf::launch_di_spatial_fused : st::launch_di_spatial_fused)(*V, sc, cur, s3, s5, f, s); });
            } else {
                add(P_DI_SAMPLING, [=](cudaStream_t s) { (fs ? stf::launch_di_sampling : st::launch_di_sampling)(*V, sc, cur, s1, f, s); });
                add(P_DI_TEMPORAL, [=](cudaStream_t s) { (fs ? stf::launch_di_temporal : st::launch_di_temporal)(*V, sc, cur, s2, s); });
                add(P_DI_SPATIAL_PICK, [=](cudaStream_t s) { (fs ? stf::launch_di_spatial_pick : st::launch_di_spatial_pick)(*V, sc, cur, s3, f, s); });
                add(P_DI_SPATIAL_TRACE, [=](cudaStream_t s) { (fs ? stf::launch_spatial_trace : st::launch_spatial_trace)(*V, sc, cam.di_diff_samples, cam.di_diff_curr_colors, cam.di_diff_stash, s); });
                add(P_DI_SPATIAL_SAMPLE, [=](cudaStream_t s) { (fs ? stf::launch_di_spatial_sample : st::launch_di_spatial_sample)(*V, sc, s5, f, s); });
            }
            add(P_DI_RESOLVING, [=](cudaStream_t s) { (fs ? stf::launch_di_resolving : st::launch_di_resolving)(*V, sc, cur, s); });
        }
        if (needs_gi) {
            uint32_t sa = seed(P_GI_SAMPLING_A), sb = seed(P_GI_SAMPLING_B), st_ = seed(P_GI_TEMPORAL), sp = seed(P_GI_SPATIAL_PICK), ss = seed(P_GI_SPATIAL_SAMPLE), sv = seed(P_GI_PREVIEW);
            uint32_t source;
            const bool tracing = f % 6u < 4u;
            const int inline_rp = (fp && tracing) ? 1 : 0;   // K11 inside K14; validation frames keep K11 (K12 / K13 read its output)
            if (!inline_rp) add(P_GI_REPROJECTION, [=](cudaStream_t s) { (fs ? stf::launch_gi_reprojection : st::launch_gi_reprojection)(*V, sc, cur, s); });
            auto sampling = [&]() {
                if (fp) { add(P_GI_SAMPLING_B, [=](cudaStream_t s) { (fs ? stf::launch_gi_sampling_fused : st::launch_gi_sampling_fused)(*V, sc, cur, sa, sb, f, s); }); return; }
                add(P_GI_SAMPLING_A, [=](cudaStream_t s) { (fs ? stf::launch_gi_sampling_a : st::launch_gi_sampling_a)(*V, sc, cur, sa, f, s); });
                add(P_GI_SAMPLING_B, [=](cudaStream_t s) { (fs ? stf::launch_gi_sampling_b : st::launch_gi_sampling_b)(*V, sc, cur, sb, f, s); });
            };
            if (tracing) {
                if (f % 2u == 0u) sampling();
                add(P_GI_TEMPORAL, [=](cudaStream_t s) { (fs ? stf::launch_gi_temporal : st::launch_gi_temporal)(*V, sc, cur, st_, f, inline_rp, s); });
                if (f % 2u == 1u) {
                    if (fp) add(P_GI_SPATIAL_PICK, [=](cudaStream_t s) { (fs ? stf::launch_gi_spatial_fused : st::launch_gi_spatial_fused)(*V, sc, cur, sp, ss, f, s); });
                    else {
                        add(P_GI_SPATIAL_PICK, [=](cudaStream_t s) { (fs ? stf::launch_gi_spatial_pick : st::launch_gi_spatial_pick)(*V, sc, cur, sp, f, s); });
                        add(P_GI_SPATIAL_TRACE, [=](cudaStream_t s) { (fs ? stf::launch_spatial_trace : st::launch_spatial_trace)(*V, sc, cam.gi_d0, cam.gi_d1, cam.gi_d2, s); });
                        add(P_GI_SPATIAL_SAMPLE, [=](cudaStream_t s) { (fs ? stf::launch_gi_spatial_sample : st::launch_gi_spatial_sample)(*V, sc, ss, f, s); });
                    }
                    source = 1;
                } else source = 0;
            } else {
                sampling();
                add(P_GI_TEMPORAL, [=](cudaStream_t s) { (fs ? stf::launch_gi_temporal : st::launch_gi_temporal)(*V, sc, cur, st_, f, 0, s); });
                source = 0;
            }
            const float4* src0 = source == 0 ? cam.gi_reservoirs[1] : cam.gi_reservoirs[2];
            add(P_GI_PREVIEW, [=](cudaStream_t s) { (fs ? stf::launch_gi_preview : st::launch_gi_preview)(*V, sc, cur, sv, 0u, src0, cam.gi_reservoirs[3], pm0, s); });
            if (fp) add(P_GI_PREVIEW, [=](cudaStream_t s) { (fs ? stf::launch_gi_preview_resolve : st::launch_gi_preview_resolve)(*V, sc, cur, sv, cam.gi_reservoirs[3], src0, s); });
            else {
                add(P_GI_PREVIEW, [=](cudaStream_t s) { (fs ? stf::launch_gi_preview : st::launch_gi_preview)(*V, sc, cur, sv, 1u, cam.gi_reservoirs[3], cam.gi_reservoirs[0], pm1, s); });
                add(P_GI_RESOLVING, [=](cudaStream_t s) { (fs ? stf::launch_gi_resolving : st::launch_gi_resolving)(*V, sc, cur, src0, s); });
            }
        }
    }
    if (d.denoise) {   // FrameDenoisingPass::run (passes/frame_denoising.rs:143-190)
        if (e->fuse_reproject) {   // ST_OPT_FUSE_REPROJECT: both signals in one launch (same arithmetic, shared surface/reprojection reads)
            add(P_DENOISE_REPROJECT, [=](cudaStream_t s) { launch_denoise_reproject_pair(*V, sc, cur, s); });
        } else {
            add(P_DENOISE_REPROJECT, [=](cudaStream_t s) { launch_denoise_reproject(*V, sc, cur, cam.di_diff_prev_colors, cam.di_diff_moments[cur ^ 1], cam.di_diff_samples, cam.di_diff_curr_colors, cam.di_diff_moments[cur], s); });
            add(P_DENOISE_REPROJECT, [=](cudaStream_t s) { launch_denoise_reproject(*V, sc, cur, cam.gi_diff_prev_colors, cam.gi_diff_moments[cur ^ 1], cam.gi_diff_samples, cam.gi_diff_curr_colors, cam.gi_diff_moments[cur], s); });
        }
        const bool fast = e->svgf_fast;
        const bool var_tiled = one && e->variance_tiled; uint32_t* verr = (uint32_t*)e->d_tile_errors.p;
        add(P_DENOISE_VARIANCE, [=](cudaStream_t s) {
            if (var_tiled && launch_denoise_variance_tiled(VV->front().cam, sc, cur, fast, verr, s)) { e->variance_tiled_launches++; return; }
            launch_denoise_variance(*VV, sc, cur, fast, s);
        });
        float4* di_io[5][2] = {{cam.di_diff_stash, cam.di_diff_prev_colors}, {cam.di_diff_prev_colors, cam.di_diff_stash}, {cam.di_diff_stash, cam.di_diff_curr_colors},
                               {cam.di_diff_curr_colors, cam.di_diff_stash}, {cam.di_diff_stash, cam.di_diff_curr_colors}};
        float4* gi_io[5][2] = {{cam.gi_diff_stash, cam.gi_diff_prev_colors}, {cam.gi_diff_prev_colors, cam.gi_diff_stash}, {cam.gi_diff_stash, cam.gi_diff_curr_colors},
                               {cam.gi_diff_curr_colors, cam.gi_diff_stash}, {cam.gi_diff_stash, cam.gi_diff_curr_colors}};
        // ST_OPT_WAVELET_PAIRED: from which iteration on the signals travel as interleaved records (5 = never)
        const bool whole_or_fused = ext != nullptr || (cam.y0 == 0 && cam.y1 == cam.h);
        const int first_paired_read = (fast && whole_or_fused && cs->pair[0]) ? (e->wavelet_paired == 2 ? 3 : e->wavelet_paired == 1 ? 4 : 5) : 5;
        for (uint32_t nth = 0; nth < 5; nth++) {
            float4 *a = di_io[nth][0], *b = di_io[nth][1], *c = gi_io[nth][0], *g = gi_io[nth][1];
            const bool reads_pair = (int)nth >= first_paired_read, writes_pair = (int)nth + 1 >= first_paired_read && nth < 4;
            const float4* pin = reads_pair ? cs->pair[nth & 1] : nullptr; float4* pout = writes_pair ? cs->pair[(nth + 1) & 1] : nullptr;
            const bool tiled = one && !reads_pair && ((e->wavelet_tiled >> nth) & 1) != 0; const int cfg = (e->wavelet_cfg >> (4 * nth)) & 15;
            uint32_t* terr = (uint32_t*)e->d_tile_errors.p;
            const Views VW = views(x.wavelet[nth]);
            add(P_DENOISE_WAVELET, [=](cudaStream_t s) {
                if (tiled && launch_denoise_wavelet_tiled(VW->front().cam, sc, f, 1u << nth, (float)(1 + nth), a, b, c, g, pout, fast, cfg, terr, s)) { e->wavelet_tiled_launches++; return; }
                launch_denoise_wavelet(*VW, sc, cur, f, 1u << nth, (float)(1 + nth), a, b, c, g, pin, pout, fast, s);
            });
            steps->back().sub = (int)nth;
        }
    }
    uint32_t mode = (uint32_t)d.mode;
    add(P_COMPOSITION, [=](cudaStream_t s) { launch_composition(*V, sc, cur, mode, di_final, gi_final, s); });
}


// ---- strip partition: exchange plan (which rows of which buffers a gathering pass needs from other ranks) ----
struct HaloItem { std::string name; int reach; };
struct HaloExchange { int before_step; std::vector<HaloItem> items; };
static const int kSpatialReach = 128;    // ReSTIR spatial taps, di_spatial_resampling.rs:55-56
static const int kPreview2Reach = 64;    // gi_preview_resampling.rs:64-70
static const int kVarianceReach = 3;     // frame_denoising.rs:128-190
static const int kWaveletReach[5] = {1, 2, 4, 9, 19};   // stride + trunc((stride-1)/4) jitter (frame_denoising.rs:269-286)

static void plan_frame(const int* schedule, int n, uint32_t frame, int temporal_reach, std::vector<HaloExchange>* plan) {
    const char* cur = (frame % 2u == 1u) ? "b" : "a";
    const char* prv = (frame % 2u == 1u) ? "a" : "b";
    bool have_gbuffer = false; int nth_preview = 0, nth_wavelet = 0;
    const char* wavelet_inputs[5] = {"stash", "prev_colors", "stash", "curr_colors", "stash"};
    bool has_preview = false, has_gi_spatial = false;
    for (int i = 0; i < n; i++) { if (schedule[i] == P_GI_PREVIEW) has_preview = true; if (schedule[i] == P_GI_SPATIAL_PICK) has_gi_spatial = true; }
    std::string gi_source = has_gi_spatial ? "gi_reservoirs_2" : "gi_reservoirs_1";
    for (int i = 0; i < n; i++) {
        int p = schedule[i];
        HaloExchange ex; ex.before_step = i;
        auto add = [&](const std::string& name, int reach) { ex.items.push_back({name, reach}); };
        if (i == 0 && temporal_reach > 0) {   // last frame's outputs gathered at reprojected positions (K4, K6, K11, K14, K20)
            add(std::string("prim_surface_map_") + prv, temporal_reach); add(std::string("prim_gbuffer_d0_") + prv, temporal_reach); add(std::string("prim_gbuffer_d1_") + prv, temporal_reach);
            add("di_reservoirs_0", temporal_reach); add("gi_reservoirs_0", temporal_reach); add("di_diff_prev_colors", temporal_reach); add("gi_diff_prev_colors", temporal_reach);
            add(std::string("di_diff_moments_") + prv, temporal_reach); add(std::string("gi_diff_moments_") + prv, temporal_reach);
        }
        if (p == P_DI_SPATIAL_PICK || p == P_GI_SPATIAL_PICK) {
            if (!have_gbuffer) { add(std::string("prim_gbuffer_d0_") + cur, kSpatialReach); add(std::string("prim_gbuffer_d1_") + cur, kSpatialReach); add("surface_nd", kSpatialReach); have_gbuffer = true; }
            add(p == P_DI_SPATIAL_PICK ? "di_reservoirs_1" : "gi_reservoirs_1", kSpatialReach);
        } else if (p == P_GI_PREVIEW) {
            if (nth_preview == 0) {
                add(std::string("prim_surface_map_") + cur, kSpatialReach); add(gi_source, kSpatialReach);
                if (!have_gbuffer) { add("surface_nd", kSpatialReach); have_gbuffer = true; }
            } else add("gi_reservoirs_3", kPreview2Reach);
            nth_preview++;
        } else if (p == P_DENOISE_VARIANCE) {
            add("di_diff_curr_colors", kVarianceReach); add("gi_diff_curr_colors", kVarianceReach);
            if (!have_gbuffer) add("surface_nd", kWaveletReach[4]);
        } else if (p == P_DENOISE_WAVELET && nth_wavelet < 5) {
            add(std::string("di_diff_") + wavelet_inputs[nth_wavelet], kWaveletReach[nth_wavelet]); add(std::string("gi_diff_") + wavelet_inputs[nth_wavelet], kWaveletReach[nth_wavelet]);
            nth_wavelet++;
        }
        (void)has_preview;
        if (!ex.items.empty()) plan->push_back(ex);
    }
}
// Row partition.  A strip pays for each neighbour it has — the G-buffer and SVGF rows it recomputes beyond its own, the rows it mirrors and
// pulls — about as much as for kStripSideRows rows of its own (measured at 8 GPUs: inner strips 1.49 ms, the same pixels without
// neighbours 1.24 ms), so the two outer strips, which have one neighbour, get that many rows more than the inner ones.  Equal strips
// below three ranks or when the inner strips would get short.  multigpu.py::strip_bounds is the same arithmetic (tests compare them).
static const int kStripSideRows = 36;
static void strip_bounds(int height, int world, std::vector<std::pair<int, int>>* b) {
    b->clear();
    long long k = kStripSideRows;
    if (world < 3 || ((long long)height + k * (2 * world - 2)) / world - 2 * k < 160) k = 0;
    const long long total = (long long)height + k * (2 * world - 2);
    auto edge = [&](int r) -> int { return r <= 0 ? 0 : r >= world ? height : (int)(total * r / world - k * (2 * r - 1)); };
    for (int r = 0; r < world; r++) b->push_back({edge(r), edge(r + 1)});
}
static float4* camera_buffer(CameraSlot* cs, const std::string& name, size_t* vec4_per_pixel) {
    size_t n = (size_t)cs->desc.width * cs->desc.height;
    for (size_t i = 0; i < cs->named.size(); i++) if (cs->named[i].first == name) { *vec4_per_pixel = cs->sizes[i].second / n; return *cs->named[i].second; }
    return nullptr;
}
// one NCCL group per exchange point: every rank sends the rows it owns that another rank's grown strip needs
static int halo_exchange(st_engine* e, CameraSlot* cs, const HaloExchange& ex) {
    std::vector<std::pair<int, int>> bounds; strip_bounds((int)cs->desc.height, e->n_ranks, &bounds);
    const int H = (int)cs->desc.height; const size_t W = cs->desc.width;
    ncclResult_t nr = g_nccl.GroupStart();
    if (nr != ncclSuccess) return fail(ST_ERR_CUDA, std::string("ncclGroupStart: ") + g_nccl.GetErrorString(nr));
    for (const HaloItem& it : ex.items) {
        size_t k = 0; float4* base = camera_buffer(cs, it.name, &k);
        if (!base) { g_nccl.GroupEnd(); return fail(ST_ERR_NOT_FOUND, "halo plan names unknown buffer " + it.name); }
        for (int dst = 0; dst < e->n_ranks; dst++) {
            int need0 = std::max(0, bounds[dst].first - it.reach), need1 = std::min(H, bounds[dst].second + it.reach);
            for (int src = 0; src < e->n_ranks; src++) {
                if (src == dst || (src != e->rank && dst != e->rank)) continue;
                int a = std::max(need0, bounds[src].first), b = std::min(need1, bounds[src].second);
                if (a >= b) continue;
                float4* ptr = base + (size_t)a * W * k; size_t count = (size_t)(b - a) * W * k * 4;
                if (src == e->rank) nr = g_nccl.Send(ptr, count, ncclFloat, dst, e->comm, e->stream);
                else { nr = g_nccl.Recv(ptr, count, ncclFloat, src, e->comm, e->stream); e->halo_bytes_last_frame += count * 4; }
                if (nr != ncclSuccess) { g_nccl.GroupEnd(); return fail(ST_ERR_CUDA, std::string("nccl p2p: ") + g_nccl.GetErrorString(nr)); }
            }
        }
    }
    nr = g_nccl.GroupEnd();
    if (nr != ncclSuccess) return fail(ST_ERR_CUDA, std::string("ncclGroupEnd: ") + g_nccl.GetErrorString(nr));
    return ST_OK;
}

static const int kLegacyFlagWord = 128, kNeedRowsWord = 200, kStripErrorWord = 202, kPulledRowsWord = 204, kWarmupWord = 512, kSyncBytes = 4096;
// the same exchange over mapped peer memory: one kernel stores my rows into every neighbour and runs the barrier
static void peer_fill(st_engine* e, CameraSlot* cs, PeerExchange* x) {
    uint32_t* sync = (uint32_t*)cs->peer.sync.p + kLegacyFlagWord;   // [0..16) flags, [16] completion counter, [17] time-outs
    x->nseg = 0; x->n_ranks = e->n_ranks; x->rank = e->rank; x->my_flags = sync; x->counter = sync + 16; x->errors = sync + 17; x->signal = 0; x->seq = 0;
    for (int r = 0; r < ST_PEER_MAX_RANKS; r++) x->peer_flags[r] = (r < e->n_ranks && r != e->rank) ? cs->peer.flags[r] + kLegacyFlagWord + e->rank : nullptr;
}
static void peer_flush(st_engine* e, CameraSlot* cs, PeerExchange* x, bool last) {
    if (last) { x->signal = 1; x->seq = ++cs->peer.seq; }
    PeerExchange copy = *x;
    e->run_timed(P_HALO_EXCHANGE, [copy](cudaStream_t s) { launch_peer_exchange(copy, s); });
    x->nseg = 0;
}
static int halo_exchange_peer(st_engine* e, CameraSlot* cs, const HaloExchange* ex) {   // ex == nullptr: barrier only
    PeerExchange x; peer_fill(e, cs, &x);
    if (ex) {
        std::vector<std::pair<int, int>> bounds; strip_bounds((int)cs->desc.height, e->n_ranks, &bounds);
        const int H = (int)cs->desc.height; const size_t W = cs->desc.width;
        const int s0 = bounds[e->rank].first, s1 = bounds[e->rank].second;
        for (const HaloItem& it : ex->items) {
            size_t k = 0; float4* base = camera_buffer(cs, it.name, &k);
            if (!base) return fail(ST_ERR_NOT_FOUND, "halo plan names unknown buffer " + it.name);
            size_t arena_off = (size_t)((char*)base - (char*)cs->arena.p);
            for (int dst = 0; dst < e->n_ranks; dst++) {
                if (dst == e->rank) continue;
                int a = std::max(std::max(0, bounds[dst].first - it.reach), s0), b = std::min(std::min(H, bounds[dst].second + it.reach), s1);
                if (a >= b) continue;
                if (x.nseg == ST_PEER_MAX_SEGMENTS) peer_flush(e, cs, &x, false);
                size_t first = (size_t)a * W * k, count = (size_t)(b - a) * W * k;
                x.seg[x.nseg++] = {(const uint4*)(base + first), (uint4*)(cs->peer.arena[dst] + arena_off) + first, count};
                // incoming rows mirror what I send (same reach both ways): count them as this rank's received bytes
                int ra = std::max(std::max(0, s0 - it.reach), bounds[dst].first), rb = std::min(std::min(H, s1 + it.reach), bounds[dst].second);
                if (ra < rb) e->halo_bytes_last_frame += (uint64_t)(rb - ra) * W * k * 16;
            }
        }
    }
    peer_flush(e, cs, &x, true);
    return ST_OK;
}

// ---- strip partition, fused transport: the order of one frame (pure; exported as text by st_plan_strip_order for CPU tests) ----
struct StripOp {
    enum Kind { STEP, SIGNAL, WAIT, SIGNAL_WAIT, PULL, PUSH } kind = STEP;
    int step = -1;                                   // STEP: index into the frame schedule
    int sig_slot = -1, wait_slot = -1;               // StripSlot
    bool sig_all = false, wait_all = false;          // every rank instead of the two neighbours
    bool wait_prev_frame = false, reset_need = false;
    const char* buffer = nullptr;                    // PUSH: rows of this buffer go to the neighbours by copy engine, then sig_slot is raised there
    int reach = 0;                                   // PUSH: rows next to each strip edge (0 = the spatial reach)
};
static void plan_strip_order(const std::vector<int>& pass, int dma_level, bool still, std::vector<StripOp>* out) {
    const bool dma = dma_level >= 1, dma_gbuffer = dma_level >= 2, dma_all = dma_level >= 3;
    auto step = [&](int i) { StripOp o; o.kind = StripOp::STEP; o.step = i; out->push_back(o); };
    auto signal = [&](int slot, bool all_ranks = false, bool reset_need = false) { StripOp o; o.kind = StripOp::SIGNAL; o.sig_slot = slot; o.sig_all = all_ranks; o.reset_need = reset_need; out->push_back(o); };
    auto wait = [&](int slot, bool all_ranks = false, bool prev = false) { StripOp o; o.kind = StripOp::WAIT; o.wait_slot = slot; o.wait_all = all_ranks; o.wait_prev_frame = prev; out->push_back(o); };
    auto signal_wait = [&](int sslot, int wslot, bool wall = false) { StripOp o; o.kind = StripOp::SIGNAL_WAIT; o.sig_slot = sslot; o.wait_slot = wslot; o.wait_all = wall; out->push_back(o); };
    auto push = [&](const char* buffer, int slot, int reach = 0) { StripOp o; o.kind = StripOp::PUSH; o.buffer = buffer; o.sig_slot = slot; o.reach = reach; out->push_back(o); };
    // split the reference order into the blocks the interleaving moves around
    std::vector<int> pre, di1, di_pick, di_rest, gi1, gi_sp, pv1, gi_tail, post;
    int nth_preview = 0;
    for (int i = 0; i < (int)pass.size(); i++) {
        switch (pass[i]) {
        case P_PRIM_GBUFFER: case P_FRAME_REPROJECTION: case P_BVH_HEATMAP: case P_REF_TRACING: case P_REF_SHADING: pre.push_back(i); break;
        case P_DI_SAMPLING: case P_DI_TEMPORAL: di1.push_back(i); break;
        case P_DI_SPATIAL_PICK: case P_DI_SPATIAL_TRACE: di_pick.push_back(i); break;
        case P_DI_SPATIAL_SAMPLE: case P_DI_RESOLVING: di_rest.push_back(i); break;
        case P_GI_REPROJECTION: case P_GI_SAMPLING_A: case P_GI_SAMPLING_B: case P_GI_TEMPORAL: gi1.push_back(i); break;
        case P_GI_SPATIAL_PICK: case P_GI_SPATIAL_TRACE: case P_GI_SPATIAL_SAMPLE: gi_sp.push_back(i); break;
        case P_GI_PREVIEW: (nth_preview++ == 0 ? pv1 : gi_tail).push_back(i); break;
        case P_GI_RESOLVING: gi_tail.push_back(i); break;
        default: post.push_back(i); break;
        }
    }
    // frame start: the primary pass needs nobody; then wait until every rank has finished the previous frame, pull, tell everybody
    size_t k = 0;
    if (!pre.empty() && pass[pre[0]] == P_PRIM_GBUFFER) { step(pre[0]); k = 1; }
    // (`still`: neither the camera nor an instance moved, so every temporal read is the pixel itself: nothing to pull, nobody to wait
    // for before history is overwritten; PULL_DONE is still raised so that a rank that does pull never waits for one that does not)
    wait(SLOT_FRAME_DONE, true, true);
    if (!still) { StripOp o; o.kind = StripOp::PULL; out->push_back(o); }
    signal(SLOT_PULL_DONE, true, !still);
    // the G-buffer rows the neighbours' spatial taps and SVGF windows reach: pushed by copy engine (instead of each neighbour
    // recomputing them), with everything up to the first gathering pass to hide behind
    bool gbuf_waited = !dma_gbuffer;
    if (dma_gbuffer && !pre.empty() && pass[pre[0]] == P_PRIM_GBUFFER) push("@gbuffer", SLOT_GBUF); else gbuf_waited = true;
    auto need_gbuffer = [&]() { if (!gbuf_waited) { wait(SLOT_GBUF); gbuf_waited = true; } };
    for (; k < pre.size(); k++) step(pre[k]);
    // DI and GI up to their first gathering pass
    for (int i : di1) step(i);
    if (!di1.empty()) { if (dma_all) push("di_reservoirs_1", SLOT_DI1); else signal(SLOT_DI1); }   // level 3: every halo with slack before its reader goes by copy engine
    for (int i : gi1) step(i);
    if (dma) {   // the flags of the GI halos are raised by the side streams, behind their copies
        if (!gi1.empty()) push("gi_reservoirs_1", SLOT_GI1);
        if (!di_pick.empty()) wait(SLOT_DI1);
    } else if (!gi1.empty() && !di_pick.empty()) signal_wait(SLOT_GI1, SLOT_DI1);
    else if (!gi1.empty()) signal(SLOT_GI1);
    else if (!di_pick.empty()) wait(SLOT_DI1);
    if (!di_pick.empty()) need_gbuffer();
    for (int i : di_pick) step(i);
    if (!gi1.empty()) wait(SLOT_GI1);
    if (!gi_sp.empty()) need_gbuffer();
    for (int i : gi_sp) step(i);
    // from here on this rank overwrites buffers others pull from (di[0], gi[0], prev colours)
    if (!gi_sp.empty() && dma) { push("gi_reservoirs_2", SLOT_GI2); if (!still) wait(SLOT_PULL_DONE, true); }
    else if (!gi_sp.empty() && still) signal(SLOT_GI2);
    else if (!gi_sp.empty()) signal_wait(SLOT_GI2, SLOT_PULL_DONE, true);
    else if (!still) wait(SLOT_PULL_DONE, true);
    if (!di_rest.empty()) step(di_rest[0]);
    if (!gi_sp.empty()) wait(SLOT_GI2);
    if (!pv1.empty()) need_gbuffer();
    for (int i : pv1) step(i);
    if (!pv1.empty()) { if (dma_all) push("gi_reservoirs_3", SLOT_GI3, kPreview2Reach); else signal(SLOT_GI3); }
    for (size_t i = 1; i < di_rest.size(); i++) step(di_rest[i]);
    if (!pv1.empty()) wait(SLOT_GI3);
    for (int i : gi_tail) step(i);
    // SVGF: K20 mirrors its rows, then everything downstream is recomputed locally
    bool svgf_waited = false;
    for (int i : post) {
        if (pass[i] == P_DENOISE_VARIANCE && !svgf_waited) { signal_wait(SLOT_SVGF, SLOT_SVGF); svgf_waited = true; need_gbuffer(); }
        step(i);
    }
    need_gbuffer();   // (a mode without any gathering pass: the flag is still consumed, so that sequence numbers stay in step)
    signal(SLOT_FRAME_DONE, true);
}

// ---- strip partition, fused transport ----------------------------------------------------------------------------------------
// One frame of this rank's strip with no stand-alone exchange step (SURVEY §8e, "overlap with interior compute"):
//  * nothing the rank can recompute travels: the G-buffer pass runs on the strip grown by the spatial reach (primary rays are
//    deterministic), K21 / K22 run on rows grown by what the following à-trous iterations read (35 rows recomputed instead of six
//    exchanges);
//  * what must travel is stored straight into the neighbours' buffers by the kernel that produces it (CameraDev::mirror_up/dn:
//    di[1], gi[1], gi[2], gi[3], the K20 colours and moments), and only the two neighbours are involved: a sequence flag per
//    producer (k_strip_signal after the kernel) and a wait in front of the first consumer (k_strip_wait);
//  * the DI and GI chains are independent until K20, so their passes are interleaved: while one chain's rows are in flight the
//    other chain computes (same kernels, same seeds, same results as the reference order);
//  * last frame's outputs that the temporal passes read at reprojected positions are pulled by the reader (k_strip_pull), sized
//    on the device from this frame's velocities: nothing for a static camera, exact for any motion.
// Every remote access of frame f happens after the rank has seen FRAME_DONE(f-1) from every rank, and a rank overwrites buffers
// others may pull only after every rank signalled PULL_DONE(f).
static int render_strips_fused(st_engine* e, CameraSlot* cs, const std::vector<std::pair<int, int>>& bounds) {
    const int R = e->rank, N = e->n_ranks, H = (int)cs->desc.height;
    const uint32_t seq = ++cs->peer.fseq;
    uint32_t* sync = (uint32_t*)cs->peer.sync.p;
    CameraDev& d = cs->dev;
    d.y0 = d.own_y0 = bounds[R].first; d.y1 = d.own_y1 = bounds[R].second;
    d.mirror_up = R > 0 ? (long long)(cs->peer.arena[R - 1] - cs->peer.arena[R]) : 0;
    d.mirror_dn = R + 1 < N ? (long long)(cs->peer.arena[R + 1] - cs->peer.arena[R]) : 0;
    d.need_rows = (int*)(sync + kNeedRowsWord);
    // ST_OPT_STRIP_DMA; -1 = by rank count: with inner strips (two neighbours each) recomputing both neighbours' G-buffer rows costs more than
    // pushing them, with two strips it does not (measured: N=2 1.351 ms at level 1, 1.398 at level 3; N=8 1.685 ms at level 2)
    const int dma_level = e->strip_dma < 0 ? (N >= 3 ? 2 : 1) : e->strip_dma;
    const bool dma = dma_level >= 1, dma_gbuffer = dma_level >= 2, dma_all = dma_level >= 3;
    d.gi_mirror_reach = dma ? 0 : kSpatialReach; d.di_mirror_reach = dma_all ? 0 : kSpatialReach;
    if (dma && !cs->ev_produced) return fail(ST_ERR_INVALID, "strip side streams missing: link the camera first (st_link_local / st_peer_import)");
    // the copy engines of last frame have long finished; this orders this frame's writes of the pushed rows after them formally
    for (int k = 0; k < 2; k++) if (cs->pushed_pending[k]) { CK(cudaStreamWaitEvent(e->stream, cs->ev_pushed[k], 0)); cs->pushed_pending[k] = false; }
    StripExt ext; ext.gbuffer = dma_gbuffer ? 0 : kSpatialReach; ext.variance = 35; const int wext[5] = {34, 32, 28, 19, 0};
    for (int i = 0; i < 5; i++) ext.wavelet[i] = wext[i];
    ext.preview_mirror[0] = dma_all ? 0 : kPreview2Reach; ext.preview_mirror[1] = 0;
    // Nothing moved since the last frame (same camera bytes, no instance touched): velocities are zero, so K4 / K6 / K14 / K20 read last
    // frame at the pixel itself — no rows to pull, K4 can run inside the G-buffer launch.  Every rank sees the same updates, hence decides alike.
    ext.still = cs->frame > 1 && !e->moved_last_tick && std::memcmp(&cs->dev.curr, &cs->dev.prev, sizeof(GpuCamera)) == 0;
    if (ext.still) d.need_rows = nullptr;
    std::vector<Step> steps; build_schedule(e, {cs}, &steps, &ext);

    StripSync ss; ss.my_flags = sync; ss.errors = sync + kStripErrorWord; ss.n_ranks = N; ss.rank = R;
    for (int r = 0; r < ST_PEER_MAX_RANKS; r++) ss.peer_flags[r] = (r < N && r != R) ? cs->peer.flags[r] : nullptr;
    const uint32_t all = (N >= 32 ? 0xffffffffu : ((1u << N) - 1u)) & ~(1u << R);
    const uint32_t nb = ((R > 0 ? (1u << (R - 1)) : 0u) | (R + 1 < N ? (1u << (R + 1)) : 0u));
    auto signal = [&](int slot, uint32_t mask, bool reset_need = false) {
        int* rn = reset_need ? (int*)(sync + kNeedRowsWord) : nullptr;
        e->run_timed(P_HALO_EXCHANGE, [=](cudaStream_t s) { launch_strip_signal(ss, slot, seq, mask, rn, H, s); });
    };
    auto wait = [&](int slot, uint32_t mask, uint32_t value) { e->run_timed(P_HALO_EXCHANGE, [=](cudaStream_t s) { launch_strip_wait(ss, slot, value, mask, s); }); };
    auto signal_wait = [&](int sig_slot, uint32_t sig_mask, int wait_slot, uint32_t wait_mask, uint32_t value) {
        e->run_timed(P_HALO_EXCHANGE, [=](cudaStream_t s) { launch_strip_signal_wait(ss, sig_slot, seq, sig_mask, wait_slot, value, wait_mask, s); });
    };
    auto emit = [&](const Step& st) { e->run_timed(st.pass, st.run, st.sub); };
    // The 128-row halos of gi_reservoirs[1] / [2] are the bulk of what travels (64 B per pixel).  With ST_OPT_STRIP_DMA they are not
    // mirrored by the producing kernel (whose own time they would stretch) but pushed by the copy engines right after it, one side
    // stream per neighbour, while this stream goes on with the other chain's passes; the flag is raised on the side stream behind the copy.
    int push_rc = ST_OK;
    auto push_rows = [&](const std::vector<std::string>& names, int reach, int slot) {
        cudaEventRecord(cs->ev_produced, e->stream);
        for (int k = 0; k < 2; k++) {
            const int nbr = k == 0 ? R - 1 : R + 1;
            if (nbr < 0 || nbr >= N) continue;
            const int r0 = k == 0 ? d.own_y0 : std::max(d.own_y0, d.own_y1 - reach), r1 = k == 0 ? std::min(d.own_y1, d.own_y0 + reach) : d.own_y1;
            cudaStreamWaitEvent(cs->side[k], cs->ev_produced, 0);
            for (const std::string& name : names) {
                size_t kk = 0; float4* base = camera_buffer(cs, name, &kk);
                if (!base) { push_rc = fail(ST_ERR_NOT_FOUND, std::string("unknown buffer ") + name); return; }
                const size_t W = cs->desc.width, row_bytes = W * kk * 16, off = (size_t)((char*)base - (char*)cs->arena.p);
                cudaMemcpyAsync(cs->peer.arena[nbr] + off + (size_t)r0 * row_bytes, (char*)base + (size_t)r0 * row_bytes, (size_t)(r1 - r0) * row_bytes, cudaMemcpyDefault, cs->side[k]);
            }
            launch_strip_signal(ss, slot, seq, 1u << nbr, nullptr, H, cs->side[k]);
            cudaEventRecord(cs->ev_pushed[k], cs->side[k]); cs->pushed_pending[k] = true;
        }
    };

    // the order of passes, flags, pulls and pushes is planned by a pure function (CPU-testable: st_plan_strip_order); execute it
    std::vector<int> ids; for (const Step& st : steps) ids.push_back(st.pass);
    std::vector<StripOp> ops; plan_strip_order(ids, dma_level, ext.still, &ops);
    const char* prv = (cs->frame % 2u == 1u) ? "a" : "b";
    for (const StripOp& op : ops) {
        const uint32_t smask = op.sig_all ? all : nb, wmask = op.wait_all ? all : nb;
        const uint32_t wseq = op.wait_prev_frame ? seq - 1u : seq;
        switch (op.kind) {
        case StripOp::STEP: emit(steps[op.step]); break;
        case StripOp::SIGNAL: signal(op.sig_slot, smask, op.reset_need); break;
        case StripOp::WAIT: wait(op.wait_slot, wmask, wseq); break;
        case StripOp::SIGNAL_WAIT: signal_wait(op.sig_slot, smask, op.wait_slot, wmask, wseq); break;
        case StripOp::PUSH:
            if (!std::strcmp(op.buffer, "@gbuffer")) {   // what the primary pass wrote for this frame and other strips read at their taps
                const std::string c = (cs->frame % 2u == 1u) ? "b" : "a";
                push_rows({"prim_gbuffer_d0_" + c, "prim_gbuffer_d1_" + c, "prim_surface_map_" + c, "surface_nd"}, kSpatialReach, op.sig_slot);
            } else push_rows({op.buffer}, op.reach ? op.reach : kSpatialReach, op.sig_slot);
            break;
        case StripOp::PULL: {
            StripPull pl; std::memset(&pl, 0, sizeof pl);
            for (int r = 0; r < N; r++) { pl.arena[r] = cs->peer.arena[r]; pl.bounds[r] = bounds[r].first; }
            pl.bounds[N] = H; pl.n_ranks = N; pl.rank = R; pl.w = (int)cs->desc.width; pl.h = H; pl.own_y0 = d.own_y0; pl.own_y1 = d.own_y1;
            pl.need_rows = (const int*)(sync + kNeedRowsWord); pl.pulled_rows = (unsigned long long*)(sync + kPulledRowsWord);
            struct { std::string name; int local; } items[] = {
                {std::string("prim_surface_map_") + prv, kSpatialReach}, {std::string("prim_gbuffer_d0_") + prv, kSpatialReach}, {std::string("prim_gbuffer_d1_") + prv, kSpatialReach},
                {"di_reservoirs_0", 0}, {"gi_reservoirs_0", 0}, {"di_diff_prev_colors", 0}, {"gi_diff_prev_colors", 0},
                {std::string("di_diff_moments_") + prv, 0}, {std::string("gi_diff_moments_") + prv, 0}};
            for (auto& it : items) {
                size_t kk = 0; float4* base = camera_buffer(cs, it.name, &kk);
                if (!base) return fail(ST_ERR_NOT_FOUND, "pull list names unknown buffer " + it.name);
                pl.items[pl.nitems++] = StripPullItem{(size_t)((char*)base - (char*)cs->arena.p), (int)kk, it.local};
            }
            e->run_timed(P_HALO_EXCHANGE, [=](cudaStream_t s) { launch_strip_pull(pl, s); });
            break;
        }
        }
    }
    d.y0 = d.own_y0; d.y1 = d.own_y1;
    if (push_rc) return push_rc;
    CK(cudaGetLastError());
    return ST_OK;
}

static CameraSlot* get_camera(st_engine* e, st_camera_handle h) { return (h >= 0 && (size_t)h < e->cameras.size() && e->cameras[h]->alive) ? e->cameras[h] : nullptr; }

}  // namespace st

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

int st_copy_output(st_engine* e, st_camera_handle h, void* host_out, int format);
const char* st_last_error(void) { return g_err.c_str(); }
const char* st_pass_name(int pass) { return (pass >= 0 && pass < P_COUNT) ? kPassNames[pass] : ""; }

int st_engine_create(int device, st_engine** out) {
    if (!out) return fail(ST_ERR_INVALID, "out is null");
    int count = 0;
    cudaError_t ce = cudaGetDeviceCount(&count);
    if (ce != cudaSuccess || count == 0) return fail(ST_ERR_CUDA, "no CUDA device available: this library has no CPU fallback");
    if (device < 0 || device >= count) return fail(ST_ERR_INVALID, "bad device ordinal");
    CK(cudaSetDevice(device));
    st_engine* e = new st_engine();
    e->device = device;
    CK(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
    std::memset(&e->world, 0, sizeof e->world);
    e->h_lights.push_back(make_sun(make_float4(0, 0, 0, 25.0f), make_float4(0, 0, 0, std::numeric_limits<float>::infinity())));   // Lights::new (lights.rs:33-50)
    e->light_slots.push_back({st_engine::kSun, 0u});
    int rc = e->d_noise.ensure(256 * 256 * 4); if (rc) { delete e; return rc; }
    rc = e->d_unpacklut.ensure(512 * 4); if (rc) { delete e; return rc; }
    rc = e->d_tile_errors.ensure(4); if (rc) { delete e; return rc; }
    launch_unpack_lut((float*)e->d_unpacklut.p, e->stream);
    *out = e;
    return ST_OK;
}
void st_engine_destroy(st_engine* e) {
    if (!e) return;
    cudaSetDevice(e->device);
    cudaStreamSynchronize(e->stream);
    if (e->copy_stream) cudaStreamSynchronize(e->copy_stream);
    for (CameraSlot* c : e->cameras) { for (int k = 0; k < 2; k++) { if (c->side[k]) { cudaStreamSynchronize(c->side[k]); cudaStreamDestroy(c->side[k]); } if (c->ev_pushed[k]) cudaEventDestroy(c->ev_pushed[k]); } if (c->ev_produced) cudaEventDestroy(c->ev_produced);
        c->arena.release(); c->svgf_pairs.release(); c->staging.release(); for (int k = 0; k < 2; k++) { if (c->ev_ready[k]) cudaEventDestroy(c->ev_ready[k]); if (c->ev_copied[k]) cudaEventDestroy(c->ev_copied[k]); } delete c; }
    DevMem* all[] = {&e->d_triangles, &e->d_bvh, &e->d_materials, &e->d_lights, &e->d_noise, &e->d_tlut, &e->d_slut, &e->d_skylut, &e->d_scratch, &e->d_raycount, &e->d_matpacked, &e->d_unpacklut, &e->d_atlas, &e->d_srgb, &e->d_tri_instance, &e->d_instance_xforms, &e->d_tile_errors};
    for (DevMem* d : all) d->release();
    for (auto& t : e->pending) { cudaEventDestroy(t.a); cudaEventDestroy(t.b); }
    for (cudaEvent_t ev : e->event_pool) cudaEventDestroy(ev);
    if (e->ev_output) cudaEventDestroy(e->ev_output);
    if (e->ev_queued) cudaEventDestroy(e->ev_queued);
    if (e->comm) g_nccl.CommDestroy(e->comm);
    if (e->own_stream) cudaStreamDestroy(e->stream);
    if (e->copy_stream) cudaStreamDestroy(e->copy_stream);
    delete e;
}

int st_insert_mesh(st_engine* e, st_handle mesh, const st_mesh_triangle* tris, size_t count) {
    if (!e || (!tris && count)) return fail(ST_ERR_INVALID, "null argument");
    e->meshes[mesh].assign(tris, tris + count);
    return ST_OK;
}
int st_remove_mesh(st_engine* e, st_handle mesh) { if (!e) return fail(ST_ERR_INVALID, "null engine"); e->meshes.erase(mesh); return ST_OK; }

int st_insert_material(st_engine* e, st_handle h, const st_material* m) {   // Materials::insert (materials.rs:36-55)
    if (!e || !m) return fail(ST_ERR_INVALID, "null argument");
    auto it = std::find(e->material_handles.begin(), e->material_handles.end(), h);
    if (it != e->material_handles.end()) e->materials[it - e->material_handles.begin()] = *m;
    else { e->material_handles.push_back(h); e->materials.push_back(*m); st_engine::MatTex mt; std::memset(&mt, 0, sizeof mt); e->material_textures.push_back(mt); }
    e->materials_dirty = true;
    return ST_OK;
}
int st_has_material(st_engine* e, st_handle h) { return e && std::find(e->material_handles.begin(), e->material_handles.end(), h) != e->material_handles.end() ? 1 : 0; }
int st_remove_material(st_engine* e, st_handle h) {
    if (!e) return fail(ST_ERR_INVALID, "null engine");
    // Materials::remove only drops the handle: the slot is never reused (allocator.give(id..id) is an
    // empty range, materials.rs:61-69), so ids of the other materials are stable.
    auto it = std::find(e->material_handles.begin(), e->material_handles.end(), h);
    if (it != e->material_handles.end()) *it = ~(st_handle)0 - 1;
    e->materials_dirty = true;
    return ST_OK;
}

}  // extern "C"
namespace st {
// The atlas rectangle of image `h` for a w x hgt image (Images::insert, images.rs:54-104): a handle that has one of that size keeps it, otherwise
// the shelf allocator places a new one.  ST_ERR_LIMIT leaves the handle's rectangle as it was.
static int place_image(st_engine* e, st_handle h, uint32_t w, uint32_t hgt, st_engine::ImageRect** out) {
    int rc;
    if (!e->d_atlas.p) {
        if ((rc = e->d_atlas.ensure((size_t)kAtlasSize * kAtlasSize * 4))) return rc;
        if ((rc = e->d_srgb.ensure(256 * 4))) return rc;
        launch_srgb_lut((float*)e->d_srgb.p, e->stream);
    }
    st_engine::ImageRect* r = nullptr;
    for (auto& k : e->images) if (k.handle == h) r = &k;
    if (!r || r->w != w || r->h != hgt) {
        if (e->shelf_x + w > kAtlasSize) { e->shelf_x = 0; e->shelf_y += e->shelf_h; e->shelf_h = 0; }
        if (w > kAtlasSize || e->shelf_y + hgt > kAtlasSize) return fail(ST_ERR_LIMIT, "no more space in the atlas");   // images.rs:71-79 (warn!)
        st_engine::ImageRect nr = {h, e->shelf_x, e->shelf_y, w, hgt};
        e->shelf_x += w; if (hgt > e->shelf_h) e->shelf_h = hgt;
        if (r) *r = nr; else { e->images.push_back(nr); r = &e->images.back(); }
    }
    *out = r;
    return ST_OK;
}
// Ends the refresh of image `h`; true if it was dynamic.  The caller then synchronises the stream, so that the old surface may be freed.
static bool drop_dynamic(st_engine* e, st_handle h) {
    const size_t before = e->dynamic.size();
    e->dynamic.erase(std::remove_if(e->dynamic.begin(), e->dynamic.end(), [&](const st_engine::DynImage& d) { return d.handle == h; }), e->dynamic.end());
    return e->dynamic.size() != before;
}
// Copies every dynamic image's surface into its atlas rectangle: one launch (per kAtlasCopies images) on the engine stream, after the output
// copies the copy stream has queued (ST_OPT_ASYNC_OUTPUT may still be writing a page-locked source).  Kernel stores into a source were queued
// on the engine stream itself and come first anyway.
static int wait_output_copies(st_engine* e) {
    if (!e->copy_stream) return ST_OK;
    if (!e->ev_output) CK(cudaEventCreateWithFlags(&e->ev_output, cudaEventDisableTiming));
    CK(cudaEventRecord(e->ev_output, e->copy_stream));
    CK(cudaStreamWaitEvent(e->stream, e->ev_output, 0));
    return ST_OK;
}
static int refresh_dynamic_images(st_engine* e) {
    int rc = wait_output_copies(e); if (rc) return rc;
    std::vector<AtlasCopy> copies;
    for (const st_engine::DynImage& d : e->dynamic)
        for (const st_engine::ImageRect& r : e->images) if (r.handle == d.handle) {
            AtlasCopy c{}; c.src = d.src; c.pitch = d.pitch; c.x = r.x; c.y = r.y; c.w = r.w; c.h = r.h;
            copies.push_back(c);
        }
    launch_atlas_refresh(copies, (uchar4*)e->d_atlas.p, e->stream);
    CK(cudaGetLastError());
    return ST_OK;
}
}  // namespace st
extern "C" {

int st_insert_image(st_engine* e, st_handle h, const uint8_t* rgba8, uint32_t w, uint32_t hgt) {   // Images::insert (images.rs:54-104), ImageData::Raw
    if (!e || !rgba8 || w == 0 || hgt == 0) return fail(ST_ERR_INVALID, "null argument");
    CK(cudaSetDevice(e->device));
    st_engine::ImageRect* r = nullptr;
    int rc = place_image(e, h, w, hgt, &r); if (rc) return rc;
    CK(cudaMemcpy2DAsync((char*)e->d_atlas.p + 4 * ((size_t)r->y * kAtlasSize + r->x), (size_t)kAtlasSize * 4, rgba8, (size_t)w * 4, (size_t)w * 4, hgt, cudaMemcpyHostToDevice, e->stream));
    CK(cudaStreamSynchronize(e->stream));   // the caller's pixels may be freed after return (and so may a dynamic surface this replaces)
    drop_dynamic(e, h);
    e->images_dirty = true;
    return ST_OK;
}
int st_remove_image(st_engine* e, st_handle h) {   // Images::remove (images.rs:106-112): the rect is released, materials keep their stale rect until re-serialised
    if (!e) return fail(ST_ERR_INVALID, "null engine");
    e->images.erase(std::remove_if(e->images.begin(), e->images.end(), [&](const st_engine::ImageRect& r) { return r.handle == h; }), e->images.end());
    if (drop_dynamic(e, h)) { CK(cudaSetDevice(e->device)); CK(cudaStreamSynchronize(e->stream)); }   // the surface may be freed after return
    e->images_dirty = true;
    return ST_OK;
}
int st_set_material_textures(st_engine* e, st_handle material, const st_material_textures* t) {
    if (!e || !t) return fail(ST_ERR_INVALID, "null argument");
    auto it = std::find(e->material_handles.begin(), e->material_handles.end(), material);
    if (it == e->material_handles.end()) return fail(ST_ERR_NOT_FOUND, "unknown material");
    st_engine::MatTex& mt = e->material_textures[it - e->material_handles.begin()];
    mt.tex[0] = t->base_color; mt.tex[1] = t->emissive; mt.tex[2] = t->metallic_roughness; mt.tex[3] = t->normal_map; mt.mask = t->mask;
    e->materials_dirty = true;
    return ST_OK;
}
int st_insert_instance(st_engine* e, st_handle h, st_handle mesh, st_handle material, const float a[12]) {   // Instances::insert (instances.rs:29-50)
    if (!e || !a) return fail(ST_ERR_INVALID, "null argument");
    Affine3 xf; xf.x = h3(a[0], a[1], a[2]); xf.y = h3(a[3], a[4], a[5]); xf.z = h3(a[6], a[7], a[8]); xf.t = h3(a[9], a[10], a[11]);
    for (auto& in : e->instances) if (in.handle == h) { in.prev_xf = in.xf; in.mesh = mesh; in.material = material; in.xf = xf; in.xf_inv = aff_inverse(xf); in.dirty = true; e->instances_dirty = true; e->motion_dirty = true; return ST_OK; }
    st_engine::Inst in; in.handle = h; in.mesh = mesh; in.material = material; in.xf = xf; in.xf_inv = aff_inverse(xf); in.prev_xf = xf; in.dirty = true;
    e->instances.push_back(in); e->instances_dirty = true; e->motion_dirty = true;
    return ST_OK;
}
int st_remove_instance(st_engine* e, st_handle h) {   // Engine::remove_instance (lib.rs:226-229)
    if (!e) return fail(ST_ERR_INVALID, "null engine");
    size_t before = e->instances.size();
    e->instances.erase(std::remove_if(e->instances.begin(), e->instances.end(), [&](const st_engine::Inst& i) { return i.handle == h; }), e->instances.end());
    if (e->instances.size() != before) e->instances_dirty = true;
    e->motion_dirty = true;
    release_range(e, h);
    return ST_OK;
}

int st_insert_light(st_engine* e, st_handle h, const st_light* l) {   // Lights::insert (lights.rs:54-82), Light::serialize (light.rs:25-79)
    if (!e || !l) return fail(ST_ERR_INVALID, "null argument");
    if (h == st_engine::kSun) return fail(ST_ERR_INVALID, "handle reserved for the sun");
    GpuLight g; std::memset(&g, 0, sizeof g);
    g.d0 = make_float4(l->position[0], l->position[1], l->position[2], l->radius);
    g.d1 = make_float4(l->color[0], l->color[1], l->color[2], l->range);
    if (l->kind == ST_LIGHT_POINT) g.d2 = make_float4(bits2f(1u), 0, 0, 0);
    else if (l->kind == ST_LIGHT_SPOT) { float2 d = oct_encode_host(h3(l->direction[0], l->direction[1], l->direction[2])); g.d2 = make_float4(bits2f(2u), d.x, d.y, l->angle); }
    else return fail(ST_ERR_INVALID, "unknown light kind");
    if (uint32_t* slot = e->light_slot(h)) { light_overwrite(e, *slot, h, g); return ST_OK; }
    uint32_t id;
    if (e->next_light < e->h_lights.size()) { id = e->next_light; e->h_lights[id] = g; }
    else { id = (uint32_t)e->h_lights.size(); e->h_lights.push_back(g); }
    e->light_slots.push_back({h, id});
    uniq_add(e->lights_created, h);
    e->next_light += 1; e->lights_dirty = true;
    return ST_OK;
}
int st_remove_light(st_engine* e, st_handle h) {   // Lights::remove (lights.rs:101-127)
    if (!e) return fail(ST_ERR_INVALID, "null engine");
    uint32_t* sp = e->light_slot(h);
    if (!sp) return ST_OK;
    uint32_t id = *sp;
    e->light_slots.erase(std::remove_if(e->light_slots.begin(), e->light_slots.end(), [&](const std::pair<st_handle, uint32_t>& p) { return p.first == h; }), e->light_slots.end());
    e->h_lights.erase(e->h_lights.begin() + id);
    GpuLight zero; std::memset(&zero, 0, sizeof zero); e->h_lights.push_back(zero);
    uniq_del(e->lights_created, h); uniq_del(e->lights_updated, h);
    e->lights_remapped.erase(std::remove_if(e->lights_remapped.begin(), e->lights_remapped.end(), [&](const std::pair<st_handle, uint32_t>& p) { return p.first == h; }), e->lights_remapped.end());
    if (std::find(e->lights_killed.begin(), e->lights_killed.end(), id) == e->lights_killed.end()) e->lights_killed.push_back(id);
    e->next_light -= 1;
    for (auto& p : e->light_slots) if (p.second > id) {
        bool seen = false; for (auto& r : e->lights_remapped) if (r.first == p.first) seen = true;
        if (!seen) e->lights_remapped.push_back({p.first, p.second});
        p.second -= 1;
    }
    e->lights_dirty = true;
    return ST_OK;
}
int st_update_sun(st_engine* e, float az, float alt) { if (!e) return fail(ST_ERR_INVALID, "null engine"); e->sun_azimuth = az; e->sun_altitude = alt; e->sun_dirty = true; return ST_OK; }

int st_set_seed_base(st_engine* e, uint32_t base) { if (!e) return fail(ST_ERR_INVALID, "null engine"); e->seed_base = base; return ST_OK; }
int st_set_blue_noise(st_engine* e, const uint8_t* rgba) {
    if (!e || !rgba) return fail(ST_ERR_INVALID, "null argument");
    CK(cudaSetDevice(e->device));
    CK(cudaMemcpyAsync(e->d_noise.p, rgba, 256 * 256 * 4, cudaMemcpyHostToDevice, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    return ST_OK;
}
uint32_t st_frame(st_engine* e) { return e ? e->frame : 0; }
int st_set_frame(st_engine* e, uint32_t frame) { if (!e || frame == 0) return fail(ST_ERR_INVALID, "frame ids start at 1"); e->frame = frame; return ST_OK; }

int st_create_camera(st_engine* e, const st_camera* c, st_camera_handle* out) {   // CameraController::new (camera_controller.rs:24-43)
    if (!e || !c || !out) return fail(ST_ERR_INVALID, "null argument");
    if (c->width == 0 || c->height == 0) return fail(ST_ERR_INVALID, "empty viewport");
    CK(cudaSetDevice(e->device));
    CameraSlot* cs = new CameraSlot();
    cs->alive = true; cs->desc = *c;
    int rc = allocate_camera(e, cs); if (rc) { delete cs; return rc; }
    cs->dev.curr = serialize_camera(*c); cs->dev.prev = cs->dev.curr;
    e->cameras.push_back(cs);
    *out = (st_camera_handle)e->cameras.size() - 1;
    return ST_OK;
}
int st_update_camera(st_engine* e, st_camera_handle h, const st_camera* c) {   // CameraController::update (camera_controller.rs:45-63)
    CameraSlot* cs = e ? get_camera(e, h) : nullptr;
    if (!cs || !c) return fail(ST_ERR_NOT_FOUND, "unknown camera");
    CK(cudaSetDevice(e->device));
    bool invalidated = cs->desc.mode != c->mode || cs->desc.denoise != c->denoise || cs->desc.ref_depth != c->ref_depth || cs->desc.width != c->width || cs->desc.height != c->height;
    cs->desc = *c;
    cs->dev.prev = cs->dev.curr;
    cs->dev.curr = serialize_camera(*c);
    if (invalidated) { GpuCamera a = cs->dev.curr, b = cs->dev.prev; CK(cudaStreamSynchronize(e->stream)); int rc = allocate_camera(e, cs); if (rc) return rc; cs->dev.curr = a; cs->dev.prev = b; }
    return ST_OK;
}
int st_delete_camera(st_engine* e, st_camera_handle h) {
    CameraSlot* cs = e ? get_camera(e, h) : nullptr;
    if (!cs) return fail(ST_ERR_NOT_FOUND, "unknown camera");
    CK(cudaSetDevice(e->device));
    CK(cudaStreamSynchronize(e->stream));
    if (e->copy_stream) CK(cudaStreamSynchronize(e->copy_stream));
    for (int k = 0; k < 2; k++) if (cs->side[k]) CK(cudaStreamSynchronize(cs->side[k]));
    cs->alive = false; cs->arena.release(); cs->svgf_pairs.release(); cs->pair[0] = cs->pair[1] = nullptr; cs->staging.release();
    return ST_OK;
}
int st_camera_set_strip(st_engine* e, st_camera_handle h, int y0, int y1) {
    CameraSlot* cs = e ? get_camera(e, h) : nullptr;
    if (!cs) return fail(ST_ERR_NOT_FOUND, "unknown camera");
    if (y0 < 0 || y1 > (int)cs->desc.height || y0 >= y1) return fail(ST_ERR_INVALID, "bad strip");
    cs->dev.y0 = y0; cs->dev.y1 = y1; cs->dev.own_y0 = y0; cs->dev.own_y1 = y1;
    return ST_OK;
}

int st_tick(st_engine* e) {   // Engine::tick (lib.rs:301-395)
    if (!e) return fail(ST_ERR_INVALID, "null engine");
    CK(cudaSetDevice(e->device));
    int rc; bool too_deep = false;
    if (!e->dynamic.empty() && (rc = refresh_dynamic_images(e))) return rc;   // Images::flush (images.rs:189-214), lib.rs:311
    if (e->materials_dirty || e->images_dirty) {   // Materials::refresh + Material::serialize (materials.rs:79-85, material.rs:29-50)
        e->materials_dirty = false; e->images_dirty = false;
        auto rect = [&](const st_engine::MatTex& mt, int k) {   // Images::lookup (images.rs:114-127)
            if (!((mt.mask >> k) & 1u)) return make_float4(0, 0, 0, 0);
            for (const auto& r : e->images) if (r.handle == mt.tex[k])
                return make_float4((float)r.x / (float)kAtlasSize, (float)r.y / (float)kAtlasSize, (float)r.w / (float)kAtlasSize, (float)r.h / (float)kAtlasSize);
            return make_float4(0, 0, 0, 0);
        };
        e->h_materials.resize(e->materials.size());
        for (size_t i = 0; i < e->materials.size(); i++) {
            const st_material& m = e->materials[i];
            GpuMaterial g; std::memset(&g, 0, sizeof g);
            g.base_color = make_float4(m.base_color[0], m.base_color[1], m.base_color[2], m.base_color[3]);
            g.emissive = make_float4(m.emissive[0], m.emissive[1], m.emissive[2], m.emissive[3]);
            g.roughness = m.perceptual_roughness * m.perceptual_roughness; g.metallic = m.metallic; g.reflectance = m.reflectance; g.ior = m.ior;
            const st_engine::MatTex& mt = e->material_textures[i];
            g.base_color_texture = rect(mt, 0); g.emissive_texture = rect(mt, 1); g.metallic_roughness_texture = rect(mt, 2); g.normal_map_texture = rect(mt, 3);
            e->h_materials[i] = g;
        }
        if ((rc = upload(e, e->d_materials, e->h_materials.data(), e->h_materials.size() * sizeof(GpuMaterial)))) return rc;
        if ((rc = e->d_matpacked.ensure(e->h_materials.size() * 4))) return rc;
        launch_material_derive((const GpuMaterial*)e->d_materials.p, (uint32_t)e->h_materials.size(), (uint32_t*)e->d_matpacked.p, e->stream);
    }
    if (refresh_instances(e)) {   // Bvh::refresh (bvh.rs:48-70)
        e->bvh.build(e->prims, e->bvh_reuse);
        std::vector<uint8_t> alpha(e->materials.size());
        for (size_t i = 0; i < alpha.size(); i++) alpha[i] = e->materials[i].alpha_blend ? 1 : 0;
        e->bvh.flatten(alpha, &e->bvh_out);
        // A tree deeper than the traversal stack cannot be walked (the reference silently corrupts a neighbour's stack,
        // strolle-gpu/src/lib.rs:72-76).  The tick still completes — with an EMPTY tree, so that the device never pairs the
        // new triangles with the old BVH — and reports ST_ERR_LIMIT at its end; nothing is drawn until the scene changes.
        if (e->bvh_out.depth - 1 > 24) { e->bvh_out.buf.clear(); too_deep = true; }
        if ((rc = upload(e, e->d_bvh, e->bvh_out.buf.data(), e->bvh_out.buf.size() * 16))) return rc;
    }
    e->moved_last_tick = e->motion_dirty;
    if (e->motion_dirty) {   // per-instance curr_xform_inv / prev_transform for the velocity map (passes/prim_raster.rs:198-223)
        e->motion_dirty = false;
        std::vector<uint32_t> tri_inst(e->h_triangles.size() / 9, 0u);
        std::vector<float4> xf(6 * std::max<size_t>(e->instances.size(), 1), make_float4(0, 0, 0, 0));
        for (size_t k = 0; k < e->instances.size(); k++) {
            const st_engine::Inst& in = e->instances[k];
            const Affine3* a[2] = {&in.xf_inv, &in.prev_xf};
            for (int j = 0; j < 2; j++) {
                xf[6 * k + 3 * j + 0] = make_float4(a[j]->x.x, a[j]->x.y, a[j]->x.z, a[j]->t.x);
                xf[6 * k + 3 * j + 1] = make_float4(a[j]->y.x, a[j]->y.y, a[j]->y.z, a[j]->t.y);
                xf[6 * k + 3 * j + 2] = make_float4(a[j]->z.x, a[j]->z.y, a[j]->z.z, a[j]->t.z);
            }
            for (const auto& r : e->tri_ranges) if (r.handle == in.handle) for (size_t t = r.b; t < r.e; t++) tri_inst[t] = (uint32_t)k;
        }
        if ((rc = upload(e, e->d_tri_instance, tri_inst.data(), tri_inst.size() * 4))) return rc;
        if ((rc = upload(e, e->d_instance_xforms, xf.data(), xf.size() * 16))) return rc;
        CK(cudaStreamSynchronize(e->stream));   // host staging vectors go out of scope
    }
    if (e->triangles_dirty) { e->triangles_dirty = false; if ((rc = upload(e, e->d_triangles, e->h_triangles.data(), e->h_triangles.size() * 16))) return rc; }
    e->world.light_count = e->next_light; e->world.sun_azimuth = e->sun_azimuth; e->world.sun_altitude = e->sun_altitude;
    if (e->sun_dirty) {   // Lights::update_sun (lights.rs:84-99); the transmittance integral runs on the device
        e->sun_dirty = false;
        if ((rc = e->d_scratch.ensure(64))) return rc;
        launch_atm_sun_color((float4*)e->d_scratch.p, e->world, e->stream);
        float4 sun[2];
        CK(cudaMemcpyAsync(sun, e->d_scratch.p, 32, cudaMemcpyDeviceToHost, e->stream));
        CK(cudaStreamSynchronize(e->stream));
        light_overwrite(e, 0, st_engine::kSun, make_sun(sun[0], sun[1]));
    }
    if (e->lights_dirty) {   // Lights::flush (lights.rs:133-162)
        for (uint32_t id : e->lights_killed) e->h_lights[id].d3.x = bits2f(0xcafebabeu);
        for (auto& r : e->lights_remapped) e->h_lights[r.second].d3.x = bits2f(*e->light_slot(r.first) + 1u);
        if ((rc = upload(e, e->d_lights, e->h_lights.data(), e->h_lights.size() * sizeof(GpuLight)))) return rc;
        CK(cudaStreamSynchronize(e->stream));   // the host mirror is edited right below
        bool again = !e->lights_created.empty() || !e->lights_updated.empty() || !e->lights_killed.empty() || !e->lights_remapped.empty();
        for (st_handle h : e->lights_created) { GpuLight& l = e->h_lights[*e->light_slot(h)]; l.prev_d0 = l.d0; l.prev_d1 = l.d1; l.prev_d2 = l.d2; }
        for (st_handle h : e->lights_updated) { GpuLight& l = e->h_lights[*e->light_slot(h)]; l.prev_d0 = l.d0; l.prev_d1 = l.d1; l.prev_d2 = l.d2; }
        for (uint32_t id : e->lights_killed) e->h_lights[id].d3.x = 0.0f;
        for (auto& r : e->lights_remapped) e->h_lights[r.second].d3.x = 0.0f;
        e->lights_created.clear(); e->lights_updated.clear(); e->lights_remapped.clear(); e->lights_killed.clear();
        e->lights_dirty = again;   // commit()/clear_slot() re-dirty the mirror: uploaded on the next tick (mapped_storage_buffer.rs:167-168)
    }
    for (CameraSlot* c : e->cameras) if (c->alive) c->frame = e->frame;   // CameraController::flush (camera_controller.rs:81-85)
    e->frame += 1;
    if (too_deep) return fail(ST_ERR_LIMIT, "BVH deeper than the 24-entry traversal stack (strolle-gpu/src/lib.rs:72-76): the scene is not drawn until it changes");
    return ST_OK;
}

int st_frame_schedule(st_engine* e, st_camera_handle h, int* pass_ids, int cap, int* count) {
    CameraSlot* cs = e ? get_camera(e, h) : nullptr;
    if (!cs || !count) return fail(ST_ERR_NOT_FOUND, "unknown camera");
    std::vector<Step> steps; build_schedule(e, {cs}, &steps);
    *count = (int)steps.size();
    for (int i = 0; i < cap && i < *count; i++) pass_ids[i] = steps[i].pass;
    return ST_OK;
}
int st_render_range(st_engine* e, st_camera_handle h, int first, int last) {
    CameraSlot* cs = e ? get_camera(e, h) : nullptr;
    if (!cs) return fail(ST_ERR_NOT_FOUND, "unknown camera");
    if (cs->frame == 0) return fail(ST_ERR_INVALID, "st_tick must precede st_render_camera");
    CK(cudaSetDevice(e->device));
    int rc = ensure_luts(e); if (rc) return rc;
    std::vector<Step> steps; build_schedule(e, {cs}, &steps);
    if (last < 0 || last >= (int)steps.size()) last = (int)steps.size() - 1;
    for (int i = std::max(first, 0); i <= last; i++) e->run_timed(steps[i].pass, steps[i].run, steps[i].sub);
    CK(cudaGetLastError());
    return ST_OK;
}
int st_render_camera(st_engine* e, st_camera_handle h, void* host_out, int format) {
    int rc = st_render_range(e, h, 0, -1); if (rc) return rc;
    if (host_out) return st_copy_output(e, h, host_out, format);
    return ST_OK;
}
// Where a frame goes: `dst` = the address of camera pixel (0, 0) inside the caller's surface, rows `pitch` bytes apart.  `device`:
// memory a kernel on the engine's device stores into (device memory of that device or of a peer, managed memory); otherwise host memory.
// `kind`: what cudaPointerGetAttributes found (cudaMemoryTypeUnregistered = pageable host memory); `mapped`: the address a kernel on the
// engine's device uses for it (null for pageable memory).
struct OutputTarget { char* dst; size_t pitch; int format; bool device; int kind = cudaMemoryTypeUnregistered; const char* mapped = nullptr; };
// The full-frame host buffer of st_render_camera / st_copy_output: tightly packed rows.
static OutputTarget host_frame(const CameraSlot* cs, void* host_out, int format) { return {(char*)host_out, (size_t)cs->desc.width * format_bpp(format), format, false}; }
// Checks a caller's surface for a `width`-pixel frame and finds what memory it is (cudaPointerGetAttributes).  Device memory of another
// device is made reachable with peer access when the two devices allow it (as st_link_local does); otherwise the surface is refused.
static int resolve_target(st_engine* e, uint32_t width, void* dst, size_t pitch, int format, OutputTarget* t) {
    const size_t bpp = format_bpp(format);
    if (!dst) return fail(ST_ERR_INVALID, "null surface");
    if (!bpp) return fail(ST_ERR_INVALID, "unsupported output format");
    if (pitch == 0) pitch = (size_t)width * bpp;
    if (pitch < (size_t)width * bpp) return fail(ST_ERR_INVALID, "row pitch " + std::to_string(pitch) + " is smaller than a row of the frame (" + std::to_string((size_t)width * bpp) + " bytes)");
    if ((uintptr_t)dst % bpp || pitch % bpp) return fail(ST_ERR_INVALID, "surface address and row pitch must be multiples of the format's " + std::to_string(bpp) + " bytes per pixel");
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, dst) != cudaSuccess) { cudaGetLastError(); a.type = cudaMemoryTypeUnregistered; }
    *t = {(char*)dst, pitch, format, a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged};
    t->kind = a.type;
    t->mapped = a.type == cudaMemoryTypeHost ? (const char*)a.devicePointer : a.type == cudaMemoryTypeUnregistered ? nullptr : (const char*)dst;
    if (a.type == cudaMemoryTypeDevice && a.device != e->device) {
        int can = 0; CK(cudaDeviceCanAccessPeer(&can, e->device, a.device));
        if (!can) return fail(ST_ERR_INVALID, "the surface is memory of device " + std::to_string(a.device) + ", which device " + std::to_string(e->device) + " cannot reach");
        CK(cudaSetDevice(e->device));
        cudaError_t ce = cudaDeviceEnablePeerAccess(a.device, 0);
        if (ce != cudaSuccess && ce != cudaErrorPeerAccessAlreadyEnabled) return fail(ST_ERR_CUDA, std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(ce));
        cudaGetLastError();
    }
    return ST_OK;
}
// rows of `row_bytes` bytes from device to host memory; one linear copy when both sides are tightly packed
static int copy_rows_to_host(char* dst, size_t dpitch, const char* src, size_t spitch, size_t row_bytes, size_t rows, cudaStream_t s) {
    if (dpitch == row_bytes && spitch == row_bytes) CK(cudaMemcpyAsync(dst, src, rows * row_bytes, cudaMemcpyDeviceToHost, s));
    else CK(cudaMemcpy2DAsync(dst, dpitch, src, spitch, row_bytes, rows, cudaMemcpyDeviceToHost, s));
    return ST_OK;
}
// The one place a frame leaves the engine: rows [y0, y1) of the composed frame, in t.format, land at t.dst + y * t.pitch and nothing
// else of the surface is written.  A device target is stored by the store kernel directly; a host target receives one copy, from
// `output` itself (RGBA32F) or from a staging slot the store kernel filled tightly packed.
static int copy_rows_out(st_engine* e, CameraSlot* cs, const OutputTarget& t, int y0, int y1) {
    const size_t W = cs->desc.width, n = W * cs->desc.height, bpp = format_bpp(t.format);
    if (!bpp) return fail(ST_ERR_INVALID, "unsupported output format");
    const size_t rows = (size_t)(y1 - y0), row_bytes = W * bpp;
    SceneDev sc = e->scene(); ViewSet v(1, view_of(cs, cs, 0)); v[0].cam.y0 = y0; v[0].cam.y1 = y1;
    const int format = t.format;
    if (t.device) {
        v[0].dst = t.dst; v[0].pitch = t.pitch;
        e->run_timed(P_COMPOSITION, [&](cudaStream_t s) { launch_output_store(v, sc, format, s); });
        CK(cudaGetLastError());
        return ST_OK;
    }
    char* host = t.dst + (size_t)y0 * t.pitch;
    if (format == ST_FORMAT_RGBA32F) return copy_rows_to_host(host, t.pitch, (const char*)(cs->dev.output + (size_t)y0 * W), row_bytes, row_bytes, rows, e->stream);
    int rc = cs->staging.ensure(2 * n * kStagingBpp); if (rc) return rc;
    cs->staging_slot ^= 1;
    const int k = cs->staging_slot;
    char* slot = (char*)cs->staging.p + (k ? n * kStagingBpp : 0);
    if (e->async_output) {   // conversion on the engine stream, copy on the copy stream: the next frame's passes do not queue behind the copy
        if (!e->copy_stream) CK(cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking));
        if (!cs->ev_ready[k]) { CK(cudaEventCreateWithFlags(&cs->ev_ready[k], cudaEventDisableTiming)); CK(cudaEventCreateWithFlags(&cs->ev_copied[k], cudaEventDisableTiming)); }
        else CK(cudaStreamWaitEvent(e->stream, cs->ev_copied[k], 0));   // slot k's previous copy must have left the staging buffer
    }
    v[0].dst = slot; v[0].pitch = row_bytes;
    e->run_timed(P_COMPOSITION, [&](cudaStream_t s) { launch_output_store(v, sc, format, s); });
    if (e->async_output) {
        CK(cudaEventRecord(cs->ev_ready[k], e->stream));
        CK(cudaStreamWaitEvent(e->copy_stream, cs->ev_ready[k], 0));
        if ((rc = copy_rows_to_host(host, t.pitch, slot + (size_t)y0 * row_bytes, row_bytes, row_bytes, rows, e->copy_stream))) return rc;
        CK(cudaEventRecord(cs->ev_copied[k], e->copy_stream));
        return ST_OK;
    }
    return copy_rows_to_host(host, t.pitch, slot + (size_t)y0 * row_bytes, row_bytes, row_bytes, rows, e->stream);
}
int st_copy_output(st_engine* e, st_camera_handle h, void* host_out, int format) {
    CameraSlot* cs = e ? get_camera(e, h) : nullptr;
    if (!cs || !host_out) return fail(ST_ERR_NOT_FOUND, "unknown camera");
    CK(cudaSetDevice(e->device));
    int rc = copy_rows_out(e, cs, host_frame(cs, host_out, format), 0, (int)cs->desc.height); if (rc) return rc;
    if (!e->async_output) CK(cudaStreamSynchronize(e->stream));
    return ST_OK;
}
int st_render_camera_to(st_engine* e, st_camera_handle h, void* dst, size_t pitch, int format) {
    CameraSlot* cs = e ? get_camera(e, h) : nullptr;
    if (!cs) return fail(ST_ERR_NOT_FOUND, "unknown camera");
    CK(cudaSetDevice(e->device));
    OutputTarget t; int rc = resolve_target(e, cs->desc.width, dst, pitch, format, &t); if (rc) return rc;   // before any pass runs: a refused call changes nothing
    if ((rc = st_render_range(e, h, 0, -1))) return rc;
    if ((rc = copy_rows_out(e, cs, t, 0, (int)cs->desc.height))) return rc;
    if (!t.device && !e->async_output) CK(cudaStreamSynchronize(e->stream));
    return ST_OK;
}
// Several cameras of one frame.  Every camera rendered after the same tick has the same frame id, so cameras of one size and mode run
// the same passes with the same seeds; such a group runs as one launch per pass, blockIdx.z selecting the camera.  Three steps, which
// st_multi_render_cameras runs on every member of a group (each step on all members before the next): check, enqueue, copy out.
struct CameraBatch { std::vector<CameraSlot*> cs; std::vector<OutputTarget> t; };
// Everything is checked before any pass runs, so that a refused call changes nothing.
static int batch_check(st_engine* e, const st_camera_handle* cameras, int n, void* const* dsts, const size_t* pitch_bytes, int format, CameraBatch* b) {
    CK(cudaSetDevice(e->device));
    b->cs.assign(n, nullptr); b->t.assign(n, OutputTarget{});
    for (int i = 0; i < n; i++) {
        if (!(b->cs[i] = get_camera(e, cameras[i]))) return fail(ST_ERR_NOT_FOUND, "unknown camera " + std::to_string(cameras[i]));
        if (std::find(cameras, cameras + i, cameras[i]) != cameras + i) return fail(ST_ERR_INVALID, "camera " + std::to_string(cameras[i]) + " is listed twice");
        const CameraSlot* c = b->cs[i];
        if (c->dev.y0 != 0 || c->dev.y1 != (int)c->desc.height || c->peer.ready)
            return fail(ST_ERR_INVALID, "camera " + std::to_string(cameras[i]) + " renders a row strip; st_render_cameras takes whole-frame cameras only");
        if (c->frame == 0) return fail(ST_ERR_INVALID, "st_tick must precede st_render_camera");
        b->t[i].dst = nullptr;
        if (dsts && dsts[i]) { int rc = resolve_target(e, c->desc.width, dsts[i], pitch_bytes ? pitch_bytes[i] : 0, format, &b->t[i]); if (rc) return rc; }
    }
    return ST_OK;
}
// The passes and the device-surface stores, grouped by (width, height, mode, denoise, ref_depth) in the order of their first camera, list
// order within a group, a group larger than one launch holds split into chunks.  Nothing here waits on the host.
static int batch_enqueue(st_engine* e, const CameraBatch& b, int format) {
    const std::vector<CameraSlot*>& cs = b.cs;
    const int n = (int)cs.size();
    CK(cudaSetDevice(e->device));
    std::vector<std::vector<int>> groups;
    for (int i = 0; i < n; i++) {
        const st_camera& d = cs[i]->desc;
        auto same = [&](const std::vector<int>& g) {
            const st_camera& a = cs[g[0]]->desc;
            return a.width == d.width && a.height == d.height && a.mode == d.mode && a.denoise == d.denoise && a.ref_depth == d.ref_depth;
        };
        auto it = std::find_if(groups.begin(), groups.end(), same);
        if (it == groups.end()) groups.push_back({i}); else it->push_back(i);
    }
    for (const std::vector<int>& g : groups) {
        for (size_t c0 = 0; c0 < g.size(); c0 += kBatchViews) {
            const std::vector<int> idx(g.begin() + c0, g.begin() + std::min(g.size(), c0 + kBatchViews));
            std::vector<CameraSlot*> chunk;
            for (int i : idx) chunk.push_back(cs[i]);
            std::vector<Step> steps; build_schedule(e, chunk, &steps);
            for (const Step& s : steps) e->run_timed(s.pass, s.run, s.sub);
            ViewSet store;   // the device surfaces of the chunk: one store launch
            for (int i : idx) if (b.t[i].dst && b.t[i].device) { store.push_back(view_of(cs[i], chunk[0], 0)); store.back().dst = b.t[i].dst; store.back().pitch = b.t[i].pitch; }
            if (!store.empty()) { const SceneDev sc = e->scene(); e->run_timed(P_COMPOSITION, [&](cudaStream_t s) { launch_output_store(store, sc, format, s); }); }
        }
    }
    CK(cudaGetLastError());
    return ST_OK;
}
// One copy per host surface (behind the passes on the engine's stream); *host_out = there was one.
static int batch_copy_out(st_engine* e, const CameraBatch& b, bool* host_out) {
    CK(cudaSetDevice(e->device));
    *host_out = false;
    for (size_t i = 0; i < b.cs.size(); i++) if (b.t[i].dst && !b.t[i].device) {
        *host_out = true;
        int rc = copy_rows_out(e, b.cs[i], b.t[i], 0, (int)b.cs[i]->desc.height); if (rc) return rc;
    }
    CK(cudaGetLastError());
    return ST_OK;
}
int st_render_cameras(st_engine* e, const st_camera_handle* cameras, int n, void* const* dsts, const size_t* pitch_bytes, int format) {
    if (!e) return fail(ST_ERR_INVALID, "null engine");
    if (n <= 0 || !cameras) return fail(ST_ERR_INVALID, "no cameras to render");
    CameraBatch b;
    int rc = batch_check(e, cameras, n, dsts, pitch_bytes, format, &b); if (rc) return rc;
    if ((rc = ensure_luts(e))) return rc;
    if ((rc = batch_enqueue(e, b, format))) return rc;
    bool host_out = false;
    if ((rc = batch_copy_out(e, b, &host_out))) return rc;
    if (host_out && !e->async_output) CK(cudaStreamSynchronize(e->stream));
    return ST_OK;
}
int st_synchronize(st_engine* e) {
    if (!e) return fail(ST_ERR_INVALID, "null engine");
    CK(cudaSetDevice(e->device)); CK(cudaStreamSynchronize(e->stream));
    if (e->copy_stream) CK(cudaStreamSynchronize(e->copy_stream));
    for (CameraSlot* c : e->cameras) for (int k = 0; k < 2; k++) if (c->side[k]) CK(cudaStreamSynchronize(c->side[k]));   // copy-engine pushes of strip halos
    return ST_OK;
}

// ---- dynamic images (ImageData::Texture { is_dynamic: true }, strolle/src/images.rs:97-102, 189-214) ----------------------------------
// A w x hgt RGBA8 surface this engine's device can read: resolve_target's checks for an Rgba8UnormSrgb frame of width w, and no pageable memory.
static int dynamic_source(st_engine* e, const void* src, size_t pitch, uint32_t w, uint32_t hgt, OutputTarget* t) {
    if (w == 0 || hgt == 0) return fail(ST_ERR_INVALID, "empty image");
    int rc = resolve_target(e, w, const_cast<void*>(src), pitch, ST_FORMAT_RGBA8_SRGB, t); if (rc) return rc;
    if (t->kind == cudaMemoryTypeUnregistered || !t->mapped)
        return fail(ST_ERR_INVALID, "a dynamic image's surface must be device, managed or page-locked host memory (st_insert_image takes pageable pixels)");
    return ST_OK;
}
static int insert_dynamic(st_engine* e, st_handle h, const OutputTarget& t, uint32_t w, uint32_t hgt) {
    CK(cudaSetDevice(e->device));
    st_engine::ImageRect* r = nullptr;
    int rc = place_image(e, h, w, hgt, &r); if (rc) return rc;
    const bool replaced = drop_dynamic(e, h);
    e->dynamic.push_back({h, t.mapped, t.pitch ? t.pitch : (size_t)w * 4});
    e->images_dirty = true;
    if (replaced) CK(cudaStreamSynchronize(e->stream));   // the previous surface may be freed after return
    return ST_OK;
}
int st_insert_dynamic_image(st_engine* e, st_handle image, const void* src, size_t pitch_bytes, uint32_t width, uint32_t height) {
    if (!e) return fail(ST_ERR_INVALID, "null engine");
    CK(cudaSetDevice(e->device));
    OutputTarget t; int rc = dynamic_source(e, src, pitch_bytes, width, height, &t); if (rc) return rc;
    return insert_dynamic(e, image, t, width, height);
}
int st_read_image(st_engine* e, st_handle image, uint8_t* dst, size_t cap_bytes, size_t* bytes) {
    if (!e || !bytes) return fail(ST_ERR_INVALID, "null argument");
    const st_engine::ImageRect* r = nullptr;
    for (const auto& k : e->images) if (k.handle == image) r = &k;
    if (!r) return fail(ST_ERR_NOT_FOUND, "unknown image");
    *bytes = (size_t)r->w * r->h * 4;
    if (!dst) return ST_OK;
    if (cap_bytes < *bytes) return fail(ST_ERR_LIMIT, "buffer too small");
    CK(cudaSetDevice(e->device));
    CK(cudaStreamSynchronize(e->stream));
    CK(cudaMemcpy2D(dst, (size_t)r->w * 4, (const char*)e->d_atlas.p + 4 * ((size_t)r->y * kAtlasSize + r->x), (size_t)kAtlasSize * 4, (size_t)r->w * 4, r->h, cudaMemcpyDeviceToHost));
    return ST_OK;
}

int st_read_buffer(st_engine* e, st_camera_handle h, const char* name, float* dst, size_t cap, size_t* count) {
    CameraSlot* cs = e ? get_camera(e, h) : nullptr;
    if (!cs || !name || !count) return fail(ST_ERR_NOT_FOUND, "unknown camera");
    CK(cudaSetDevice(e->device));
    if (!std::strcmp(name, "curr_camera") || !std::strcmp(name, "prev_camera")) {
        const GpuCamera& c = !std::strcmp(name, "curr_camera") ? cs->dev.curr : cs->dev.prev;
        *count = 40; if (dst) std::memcpy(dst, &c, 4 * std::min<size_t>(cap, 40)); return ST_OK;
    }
    for (size_t i = 0; i < cs->named.size(); i++) if (cs->named[i].first == name) {
        *count = cs->sizes[i].second * 4;
        if (dst) { CK(cudaStreamSynchronize(e->stream)); CK(cudaMemcpy(dst, *cs->named[i].second, 4 * std::min(cap, *count), cudaMemcpyDeviceToHost)); }
        return ST_OK;
    }
    return fail(ST_ERR_NOT_FOUND, std::string("unknown buffer ") + name);
}
int st_buffer_device_ptr(st_engine* e, st_camera_handle h, const char* name, void** ptr, size_t* bytes) {
    CameraSlot* cs = e ? get_camera(e, h) : nullptr;
    if (!cs || !name || !ptr || !bytes) return fail(ST_ERR_NOT_FOUND, "unknown camera");
    for (size_t i = 0; i < cs->named.size(); i++) if (cs->named[i].first == name) { *ptr = *cs->named[i].second; *bytes = cs->sizes[i].second * 16; return ST_OK; }
    return fail(ST_ERR_NOT_FOUND, std::string("unknown buffer ") + name);
}
int st_read_scene(st_engine* e, const char* name, float* dst, size_t cap, size_t* count) {
    if (!e || !name || !count) return fail(ST_ERR_INVALID, "null argument");
    CK(cudaSetDevice(e->device));
    std::string s(name);
    const void* dev = nullptr; size_t n = 0;
    if (s == "world") { *count = 4; if (dst) std::memcpy(dst, &e->world, 4 * std::min<size_t>(cap, 4)); return ST_OK; }
    if (s == "triangles") { dev = e->d_triangles.p; n = e->h_triangles.size() * 4; }
    else if (s == "bvh") { dev = e->d_bvh.p; n = e->bvh_out.buf.size() * 4; }
    else if (s == "materials") { dev = e->d_materials.p; n = e->h_materials.size() * 28; }
    else if (s == "lights") { dev = e->d_lights.p; n = e->h_lights.size() * 28; }
    else if (s == "transmittance_lut" || s == "scattering_lut" || s == "sky_lut") {
        int rc = ensure_luts(e); if (rc) return rc;
        if (s == "transmittance_lut") { dev = e->d_tlut.p; n = 256 * 64 * 4; } else if (s == "scattering_lut") { dev = e->d_slut.p; n = 32 * 32 * 4; } else { dev = e->d_skylut.p; n = 256 * 256 * 4; }
    } else return fail(ST_ERR_NOT_FOUND, "unknown scene buffer " + s);
    *count = n;
    if (dst && n) { CK(cudaStreamSynchronize(e->stream)); CK(cudaMemcpy(dst, dev, 4 * std::min(cap, n), cudaMemcpyDeviceToHost)); }
    return ST_OK;
}
int st_bvh_depth(st_engine* e, int* depth) { if (!e || !depth) return fail(ST_ERR_INVALID, "null argument"); *depth = e->bvh_out.depth; return ST_OK; }

static int trace_stream(st_engine* e, const float* rays, size_t n, void* out, bool closest, float* device_ms) {
    if (!e || !rays || !out) return fail(ST_ERR_INVALID, "null argument");
    if (e->frame <= 1) return fail(ST_ERR_INVALID, "no scene uploaded: call st_tick first");
    CK(cudaSetDevice(e->device));
    size_t out_bytes = closest ? n * 48 : n * 4;
    DevMem d_in, d_out; int rc;
    if ((rc = d_in.ensure(n * 32)) || (rc = d_out.ensure(out_bytes))) { d_in.release(); d_out.release(); return rc; }
    cudaEvent_t a = e->get_event(), b = e->get_event();
    cudaMemcpyAsync(d_in.p, rays, n * 32, cudaMemcpyHostToDevice, e->stream);
    SceneDev sc = e->scene();
    cudaEventRecord(a, e->stream);
    if (closest) launch_trace_stream_closest(sc, (const float4*)d_in.p, (long)n, (float4*)d_out.p, e->stream);
    else launch_trace_stream_any(sc, (const float4*)d_in.p, (long)n, (uint32_t*)d_out.p, e->stream);
    cudaEventRecord(b, e->stream);
    cudaMemcpyAsync(out, d_out.p, out_bytes, cudaMemcpyDeviceToHost, e->stream);
    cudaError_t ce = cudaStreamSynchronize(e->stream);
    float ms = 0; cudaEventElapsedTime(&ms, a, b);
    if (device_ms) *device_ms = ms;
    e->pass_launches[P_TRACE_STREAM]++; e->pass_ms[P_TRACE_STREAM] += ms;
    e->event_pool.push_back(a); e->event_pool.push_back(b);
    d_in.release(); d_out.release();
    if (ce != cudaSuccess) return fail(ST_ERR_CUDA, cudaGetErrorString(ce));
    return ST_OK;
}
int st_trace_closest(st_engine* e, const float* rays, size_t n, float* out, float* ms) { return trace_stream(e, rays, n, out, true, ms); }
int st_trace_any(st_engine* e, const float* rays, size_t n, uint32_t* out, float* ms) { return trace_stream(e, rays, n, out, false, ms); }

int st_device_math(st_engine* e, int op, const float* a, const float* b, float* out, size_t n) {
    if (!e || !a || !out) return fail(ST_ERR_INVALID, "null argument");
    CK(cudaSetDevice(e->device));
    DevMem da, db, dc; int rc;
    if ((rc = da.ensure(n * 4)) || (rc = db.ensure(n * 4)) || (rc = dc.ensure(n * 4))) return rc;
    CK(cudaMemcpyAsync(da.p, a, n * 4, cudaMemcpyHostToDevice, e->stream));
    if (b) CK(cudaMemcpyAsync(db.p, b, n * 4, cudaMemcpyHostToDevice, e->stream));
    launch_math(op, (const float*)da.p, (const float*)db.p, (float*)dc.p, (long)n, e->stream);
    CK(cudaMemcpyAsync(out, dc.p, n * 4, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    da.release(); db.release(); dc.release();
    return ST_OK;
}

int st_set_option(st_engine* e, int option, int value) {
    if (!e) return fail(ST_ERR_INVALID, "null engine");
    if (option == ST_OPT_SVGF_FAST_MATH) { e->svgf_fast = value != 0; return ST_OK; }
    if (option == ST_OPT_SHADING_FAST_MATH) { e->shading_fast = value != 0; return ST_OK; }
    if (option == ST_OPT_ASYNC_OUTPUT) { e->async_output = value != 0; return ST_OK; }
    if (option == ST_OPT_HALO_NCCL) { e->halo_nccl = value != 0; return ST_OK; }
    if (option == ST_OPT_STRIP_FUSED) { e->strip_fused = value != 0; return ST_OK; }
    if (option == ST_OPT_STRIP_DMA) { if (value < -1 || value > 3) return fail(ST_ERR_INVALID, "ST_OPT_STRIP_DMA: -1 .. 3"); e->strip_dma = value; return ST_OK; }
    if (option == ST_OPT_WAVELET_PAIRED) { if (value < 0 || value > 2) return fail(ST_ERR_INVALID, "ST_OPT_WAVELET_PAIRED: 0, 1 or 2"); e->wavelet_paired = value; return ST_OK; }
    if (option == ST_OPT_FUSED_PASSES) { e->fused_passes = value != 0; return ST_OK; }
    if (option == ST_OPT_WAVELET_TILED) { e->wavelet_tiled = value & 31; return ST_OK; }
    if (option == ST_OPT_VARIANCE_TILED) { e->variance_tiled = value != 0; return ST_OK; }
    if (option == ST_OPT_BVH_REUSE) { e->bvh_reuse = value != 0; return ST_OK; }
    if (option == ST_OPT_FUSE_REPROJECT) { e->fuse_reproject = value != 0; return ST_OK; }
    if (option == ST_OPT_WAVELET_TILE_CFG) { e->wavelet_cfg = value & 0xfffff; return ST_OK; }
    return fail(ST_ERR_INVALID, "unknown option");
}
// ---- host-side BVH builder without a device (test / tool hook; strolle/src/bvh/builder.rs, serializer.rs) ----
struct st_bvh_builder { BvhBuild b; BvhOut flat; };
int st_bvh_builder_create(st_bvh_builder** out) { if (!out) return fail(ST_ERR_INVALID, "out is null"); *out = new st_bvh_builder(); return ST_OK; }
void st_bvh_builder_destroy(st_bvh_builder* b) { delete b; }
int st_bvh_builder_read(st_bvh_builder* b, float* out, size_t cap_floats) {   // the stream of the last build
    if (!b || !out) return fail(ST_ERR_INVALID, "null argument");
    if (cap_floats < b->flat.buf.size() * 4) return fail(ST_ERR_LIMIT, "output buffer too small");
    std::memcpy(out, b->flat.buf.data(), b->flat.buf.size() * 16);
    return ST_OK;
}
int st_bvh_builder_build(st_bvh_builder* b, const float* prims11, size_t n, int reuse, float* out, size_t cap_floats, size_t* n_floats, uint32_t* grafted, int* depth) {
    if (!b || (!prims11 && n) || !n_floats) return fail(ST_ERR_INVALID, "null argument");
    std::vector<Prim> all(n);
    uint32_t max_mat = 0;
    for (size_t i = 0; i < n; i++) {
        const float* f = prims11 + 11 * i;
        Prim& p = all[i];
        p.tri = f2bits(f[0]); p.mat = f2bits(f[1]); p.center = h3(f[2], f[3], f[4]);
        p.box.lo = h3(f[5], f[6], f[7]); p.box.hi = h3(f[8], f[9], f[10]);
        max_mat = std::max(max_mat, p.mat);
    }
    b->b.build(all, reuse != 0);
    // a grafted subtree may still name a material of an earlier call (quirk C-20): size the flag table for those too
    for (const Prim& p : b->b.prims) max_mat = std::max(max_mat, p.mat);
    std::vector<uint8_t> alpha((size_t)max_mat + 1, 0);
    b->b.flatten(alpha, &b->flat);
    *n_floats = b->flat.buf.size() * 4;
    if (grafted) *grafted = b->b.grafted;
    if (depth) *depth = b->flat.depth;
    if (out) return st_bvh_builder_read(b, out, cap_floats);
    return ST_OK;
}

int st_get_stat(st_engine* e, int stat, uint64_t* value) {
    if (!e || !value) return fail(ST_ERR_INVALID, "null argument");
    if (stat == ST_STAT_WAVELET_TILED_LAUNCHES) { *value = e->wavelet_tiled_launches; return ST_OK; }
    if (stat == ST_STAT_VARIANCE_TILED_LAUNCHES) { *value = e->variance_tiled_launches; return ST_OK; }
    if (stat == ST_STAT_BVH_GRAFTED_SUBTREES) { *value = e->bvh.grafted; return ST_OK; }
    if (stat == ST_STAT_STRIP_PULLED_ROWS) {   // rows of last frame's buffers this rank fetched from their owners so far (fused strip transport, all cameras)
        CK(cudaSetDevice(e->device)); CK(cudaStreamSynchronize(e->stream));
        uint64_t total = 0;
        for (CameraSlot* c : e->cameras) if (c->alive && c->peer.sync.p) { uint64_t v = 0; CK(cudaMemcpy(&v, (uint32_t*)c->peer.sync.p + kPulledRowsWord, 8, cudaMemcpyDeviceToHost)); total += v; }
        *value = total; return ST_OK;
    }
    if (stat == ST_STAT_STRIP_FIRST_TIMEOUT) {   // 0, or 0x80000000 | slot << 16 | awaited rank << 8 | low byte of the sequence value: the first flag wait that gave up
        CK(cudaSetDevice(e->device)); CK(cudaStreamSynchronize(e->stream));
        *value = 0;
        for (CameraSlot* c : e->cameras) if (c->alive && c->peer.sync.p && !*value) { uint32_t v = 0; CK(cudaMemcpy(&v, (uint32_t*)c->peer.sync.p + kStripErrorWord + 1, 4, cudaMemcpyDeviceToHost)); *value = v; }
        return ST_OK;
    }
    if (stat == ST_STAT_LAST_FRAME_FUSED_STRIPS) { *value = e->last_frame_fused ? 1 : 0; return ST_OK; }
    if (stat == ST_STAT_WAVELET_TILED_ERRORS) {
        CK(cudaSetDevice(e->device));
        CK(cudaStreamSynchronize(e->stream));
        uint32_t v = 0; CK(cudaMemcpy(&v, e->d_tile_errors.p, 4, cudaMemcpyDeviceToHost));
        *value = v; return ST_OK;
    }
    return fail(ST_ERR_INVALID, "unknown statistic");
}
int st_set_stream(st_engine* e, void* cuda_stream, int external) {
    if (!e) return fail(ST_ERR_INVALID, "null engine");
    CK(cudaSetDevice(e->device));
    CK(cudaStreamSynchronize(e->stream));
    if (e->own_stream) { cudaStreamDestroy(e->stream); e->own_stream = false; }
    if (external) e->stream = (cudaStream_t)cuda_stream;   // NULL is the legacy default stream
    else { CK(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking)); e->own_stream = true; }
    return ST_OK;
}
int st_count_rays(st_engine* e, int enabled) {
    if (!e) return fail(ST_ERR_INVALID, "null engine");
    CK(cudaSetDevice(e->device));
    int rc = e->d_raycount.ensure(8); if (rc) return rc;
    e->count_rays = enabled != 0;
    return ST_OK;
}
int st_ray_count(st_engine* e, uint64_t* rays, int reset) {
    if (!e || !rays) return fail(ST_ERR_INVALID, "null argument");
    CK(cudaSetDevice(e->device));
    *rays = 0;
    if (!e->d_raycount.p) return ST_OK;
    CK(cudaStreamSynchronize(e->stream));
    CK(cudaMemcpy(rays, e->d_raycount.p, 8, cudaMemcpyDeviceToHost));
    if (reset) CK(cudaMemset(e->d_raycount.p, 0, 8));
    CK(cudaDeviceSynchronize());
    return ST_OK;
}
int st_nccl_unique_id(uint8_t* out128) {
    if (!out128) return fail(ST_ERR_INVALID, "null argument");
    { std::string err; if (!g_nccl.load(&err)) return fail(ST_ERR_CUDA, err); }
    ncclUniqueId id; ncclResult_t r = g_nccl.GetUniqueId(&id);
    if (r != ncclSuccess) return fail(ST_ERR_CUDA, std::string("ncclGetUniqueId: ") + g_nccl.GetErrorString(r));
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId size");
    std::memcpy(out128, &id, 128);
    return ST_OK;
}
int st_nccl_init(st_engine* e, const uint8_t* id128, int rank, int world) {
    if (!e || !id128 || world < 1 || rank < 0 || rank >= world) return fail(ST_ERR_INVALID, "bad argument");
    { std::string err; if (!g_nccl.load(&err)) return fail(ST_ERR_CUDA, err); }
    CK(cudaSetDevice(e->device));
    ncclUniqueId id; std::memcpy(&id, id128, 128);
    if (e->comm) { g_nccl.CommDestroy(e->comm); e->comm = nullptr; }
    ncclResult_t r = g_nccl.CommInitRank(&e->comm, world, id, rank);
    if (r != ncclSuccess) return fail(ST_ERR_CUDA, std::string("ncclCommInitRank: ") + g_nccl.GetErrorString(r));
    e->rank = rank; e->n_ranks = world;
    return ST_OK;
}
int st_peer_export(st_engine* e, st_camera_handle h, uint8_t* out192) {
    CameraSlot* cs = e ? get_camera(e, h) : nullptr;
    if (!cs || !out192) return fail(ST_ERR_NOT_FOUND, "unknown camera");
    CK(cudaSetDevice(e->device));
    size_t n = (size_t)cs->desc.width * cs->desc.height;
    int rc = cs->staging.ensure(2 * n * kStagingBpp); if (rc) return rc;
    if ((rc = cs->peer.sync.ensure(kSyncBytes))) return rc;
    { const int need0[2] = {(int)cs->desc.height, -1}; CK(cudaMemcpy((uint32_t*)cs->peer.sync.p + kNeedRowsWord, need0, 8, cudaMemcpyHostToDevice)); }
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "ipc handle size");
    cudaIpcMemHandle_t hs[3];
    CK(cudaIpcGetMemHandle(&hs[0], cs->arena.p)); CK(cudaIpcGetMemHandle(&hs[1], cs->peer.sync.p)); CK(cudaIpcGetMemHandle(&hs[2], cs->staging.p));
    std::memcpy(out192, hs, ST_PEER_HANDLE_BYTES);
    return ST_OK;
}
// Side streams and events of the copy-engine halo pushes, created when the camera is linked (peer pointers known) — and the copy path
// to each neighbour is exercised once here: the first such copy may load a driver-internal module, which synchronises the device, and
// inside a frame that would stall this thread while another rank's stream spins on a flag only this thread's later launches can raise.
static int strip_streams_prepare(st_engine* e, CameraSlot* cs) {
    CK(cudaSetDevice(e->device));
    {   // no kernel may be loaded lazily once streams wait on each other's flags (see preload_kernels)
        const int a = st::preload_kernels(), b = stf::preload_kernels();
        static bool warned = false;
        if ((a || b) && !warned) { warned = true; std::fprintf(stderr, "strolle_b200: this driver cannot enumerate the library's kernels (%d/%d); set CUDA_MODULE_LOADING=EAGER when several strips share one host thread\n", a, b); }
    }
    if (!cs->ev_produced) {
        CK(cudaEventCreateWithFlags(&cs->ev_produced, cudaEventDisableTiming));
        for (int k = 0; k < 2; k++) { CK(cudaStreamCreateWithFlags(&cs->side[k], cudaStreamNonBlocking)); CK(cudaEventCreateWithFlags(&cs->ev_pushed[k], cudaEventDisableTiming)); }
    }
    const uint32_t* mine = (const uint32_t*)cs->peer.sync.p;
    for (int k = 0; k < 2; k++) {
        const int nbr = k == 0 ? e->rank - 1 : e->rank + 1;
        if (nbr < 0 || nbr >= e->n_ranks || !cs->peer.flags[nbr]) continue;
        CK(cudaMemcpyAsync(cs->peer.flags[nbr] + kWarmupWord + 8 * k, mine + kWarmupWord + 16, 16, cudaMemcpyDefault, cs->side[k]));
        CK(cudaEventRecord(cs->ev_pushed[k], cs->side[k]));
        CK(cudaStreamSynchronize(cs->side[k]));
    }
    CK(cudaEventRecord(cs->ev_produced, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    return ST_OK;
}
int st_peer_import(st_engine* e, st_camera_handle h, const uint8_t* all, int rank, int world) {
    CameraSlot* cs = e ? get_camera(e, h) : nullptr;
    if (!cs || !all) return fail(ST_ERR_NOT_FOUND, "unknown camera");
    if (world < 1 || world > ST_PEER_MAX_RANKS || rank < 0 || rank >= world) return fail(ST_ERR_LIMIT, "peer transport supports up to 16 ranks");
    if (!cs->peer.sync.p || !cs->staging.p) return fail(ST_ERR_INVALID, "st_peer_export first");
    CK(cudaSetDevice(e->device));
    cs->peer.arena.assign(world, nullptr); cs->peer.staging.assign(world, nullptr); cs->peer.flags.assign(world, nullptr);
    for (int r = 0; r < world; r++) {
        if (r == rank) { cs->peer.arena[r] = (char*)cs->arena.p; cs->peer.flags[r] = (uint32_t*)cs->peer.sync.p; cs->peer.staging[r] = (char*)cs->staging.p; continue; }
        cudaIpcMemHandle_t hs[3]; std::memcpy(hs, all + (size_t)r * ST_PEER_HANDLE_BYTES, ST_PEER_HANDLE_BYTES);
        void* p = nullptr;
        CK(cudaIpcOpenMemHandle(&p, hs[0], cudaIpcMemLazyEnablePeerAccess)); cs->peer.arena[r] = (char*)p;
        CK(cudaIpcOpenMemHandle(&p, hs[1], cudaIpcMemLazyEnablePeerAccess)); cs->peer.flags[r] = (uint32_t*)p;
        CK(cudaIpcOpenMemHandle(&p, hs[2], cudaIpcMemLazyEnablePeerAccess)); cs->peer.staging[r] = (char*)p;
    }
    e->rank = rank; e->n_ranks = world; cs->peer.seq = 0; cs->peer.fseq = 0; cs->peer.ready = true; cs->peer.ipc = true;
    return strip_streams_prepare(e, cs);
}
int st_peer_errors(st_engine* e, st_camera_handle h, uint32_t* count) {
    CameraSlot* cs = e ? get_camera(e, h) : nullptr;
    if (!cs || !count) return fail(ST_ERR_NOT_FOUND, "unknown camera");
    *count = 0;
    if (!cs->peer.sync.p) return ST_OK;
    CK(cudaSetDevice(e->device)); CK(cudaStreamSynchronize(e->stream));
    uint32_t both[2] = {0, 0};
    CK(cudaMemcpy(&both[0], (uint32_t*)cs->peer.sync.p + kLegacyFlagWord + 17, 4, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(&both[1], (uint32_t*)cs->peer.sync.p + kStripErrorWord, 4, cudaMemcpyDeviceToHost));
    *count = both[0] + both[1];
    return ST_OK;
}
int st_plan_frame(const int* schedule, int n, uint32_t frame, int temporal_reach, char* out, size_t cap) {
    if (!schedule || !out || cap == 0) return fail(ST_ERR_INVALID, "null argument");
    std::vector<HaloExchange> plan; plan_frame(schedule, n, frame, temporal_reach, &plan);
    std::string text;
    for (const HaloExchange& ex : plan) for (const HaloItem& it : ex.items) text += std::to_string(ex.before_step) + ":" + it.name + ":" + std::to_string(it.reach) + ";";
    if (text.size() + 1 > cap) return fail(ST_ERR_LIMIT, "plan text buffer too small");
    std::memcpy(out, text.c_str(), text.size() + 1);
    return ST_OK;
}
// enqueues this rank's strip of the frame (no output handling)
static int enqueue_strip_frame(st_engine* e, CameraSlot* cs, int temporal_reach) {
    const bool peer = e->n_ranks > 1 && cs->peer.ready && !e->halo_nccl;
    if (e->n_ranks > 1 && !peer && !e->comm) return fail(ST_ERR_INVALID, "st_nccl_init, st_peer_import or st_link_local first");
    if (cs->frame == 0) return fail(ST_ERR_INVALID, "st_tick must precede rendering");
    int rc = ensure_luts(e); if (rc) return rc;
    std::vector<std::pair<int, int>> bounds; strip_bounds((int)cs->desc.height, e->n_ranks, &bounds);
    cs->dev.y0 = cs->dev.own_y0 = bounds[e->rank].first; cs->dev.y1 = cs->dev.own_y1 = bounds[e->rank].second;
    int min_rows = (int)cs->desc.height;
    for (auto& bd : bounds) min_rows = std::min(min_rows, bd.second - bd.first);
    // the fused transport sends to the two neighbours only: every strip must cover the largest reach
    const bool fused = peer && e->strip_fused && min_rows >= kSpatialReach;
    e->last_frame_fused = fused;
    e->halo_bytes_last_frame = 0;
    if (fused) {
        if ((rc = render_strips_fused(e, cs, bounds))) return rc;
        // rows mirrored into this rank by its neighbours (the K6 / K14 / K17 / K18 / K20 stores); the temporal pull is counted on the device
        const uint64_t W = cs->desc.width; const int nbs = (e->rank > 0 ? 1 : 0) + (e->rank + 1 < e->n_ranks ? 1 : 0);
        std::vector<Step> steps; build_schedule(e, {cs}, &steps);
        bool di = false, gi = false, sp = false, dn = cs->desc.denoise != 0;
        for (const Step& st : steps) { di |= st.pass == P_DI_TEMPORAL; gi |= st.pass == P_GI_TEMPORAL; sp |= st.pass == P_GI_SPATIAL_PICK; }
        uint64_t per_nb = 0;
        if (di) per_nb += (uint64_t)kSpatialReach * 32;
        if (gi) per_nb += (uint64_t)kSpatialReach * 64 * (sp ? 2 : 1) + (uint64_t)kPreview2Reach * 64;
        if (dn) per_nb += 38ull * 64;
        e->halo_bytes_last_frame = per_nb * W * nbs;
    } else {
        cs->dev.mirror_up = cs->dev.mirror_dn = 0; cs->dev.need_rows = nullptr;
        std::vector<Step> steps; build_schedule(e, {cs}, &steps);
        std::vector<int> ids; for (const Step& st : steps) ids.push_back(st.pass);
        std::vector<HaloExchange> plan;
        // The exchange-point transports ship a FIXED number of last frame's rows.  That is only enough while nothing moves: with a moving
        // camera or instance the reprojected reads can land anywhere, so the whole of last frame's buffers is exchanged then (correct for
        // any motion, and slow: the fused transport sizes this on the device instead).
        const bool moving = e->moved_last_tick || std::memcmp(&cs->dev.curr, &cs->dev.prev, sizeof(GpuCamera)) != 0;
        if (e->n_ranks > 1) plan_frame(ids.data(), (int)ids.size(), cs->frame, moving ? (int)cs->desc.height : temporal_reach, &plan);
        size_t next = 0;
        if (peer && (rc = halo_exchange_peer(e, cs, nullptr))) return rc;   // frame barrier: nobody still reads last frame's rows
        for (int i = 0; i < (int)steps.size(); i++) {
            if (next < plan.size() && plan[next].before_step == i) { if ((rc = peer ? halo_exchange_peer(e, cs, &plan[next]) : halo_exchange(e, cs, plan[next]))) return rc; next++; }
            e->run_timed(steps[i].pass, steps[i].run, steps[i].sub);
        }
    }
    CK(cudaGetLastError());
    return ST_OK;
}
// `gather`: 0 = render only; 1 = assemble the composed frame on rank 0 (strips travel in `format`; rank 0 copies it to `host_out`);
// 2 = every rank converts its OWN rows and copies them into rows [y0, y1) of `host_out`, a full-frame host buffer that the ranks
// share (one buffer in a single-process host, a shared-memory segment between processes): no funnel through rank 0.
int st_strip_bounds(int height, int world, int* rows_out) {
    if (!rows_out || height < 1 || world < 1 || world > height) return fail(ST_ERR_INVALID, "st_strip_bounds: 1 <= world <= height");
    std::vector<std::pair<int, int>> b; strip_bounds(height, world, &b);
    for (int r = 0; r < world; r++) { rows_out[2 * r] = b[r].first; rows_out[2 * r + 1] = b[r].second; }
    return ST_OK;
}
int st_plan_strip_order(const int* schedule, int n, int dma, char* out, size_t cap) {
    if (!schedule || !out || cap == 0) return fail(ST_ERR_INVALID, "null argument");
    static const char* kSlot[SLOT_COUNT] = {"FRAME_DONE", "PULL_DONE", "DI1", "GI1", "GI2", "GI3", "SVGF", "GBUF"};
    std::vector<int> ids(schedule, schedule + n);
    std::vector<StripOp> ops; plan_strip_order(ids, dma & 3, (dma & 4) != 0, &ops);
    std::string text;
    for (const StripOp& op : ops) {
        switch (op.kind) {
        case StripOp::STEP: text += "step:" + std::to_string(op.step); break;
        case StripOp::SIGNAL: text += std::string("signal:") + kSlot[op.sig_slot] + (op.sig_all ? ":all" : ":nb"); break;
        case StripOp::WAIT: text += std::string("wait:") + kSlot[op.wait_slot] + (op.wait_all ? ":all" : ":nb") + (op.wait_prev_frame ? ":prev" : ""); break;
        case StripOp::SIGNAL_WAIT: text += std::string("signal:") + kSlot[op.sig_slot] + ":nb;wait:" + kSlot[op.wait_slot] + (op.wait_all ? ":all" : ":nb"); break;
        case StripOp::PULL: text += "pull"; break;
        case StripOp::PUSH: text += std::string("push:") + op.buffer + ":" + kSlot[op.sig_slot]; break;
        }
        text += ";";
    }
    if (text.size() + 1 > cap) return fail(ST_ERR_LIMIT, "plan text buffer too small");
    std::memcpy(out, text.c_str(), text.size() + 1);
    return ST_OK;
}
int st_render_strips(st_engine* e, st_camera_handle h, void* host_out, int format, int temporal_reach, int gather) {
    CameraSlot* cs = e ? get_camera(e, h) : nullptr;
    if (!cs) return fail(ST_ERR_NOT_FOUND, "unknown camera");
    CK(cudaSetDevice(e->device));
    int rc = enqueue_strip_frame(e, cs, temporal_reach); if (rc) return rc;
    if (!gather) return ST_OK;
    const bool peer = e->n_ranks > 1 && cs->peer.ready && !e->halo_nccl;
    std::vector<std::pair<int, int>> bounds; strip_bounds((int)cs->desc.height, e->n_ranks, &bounds);
    if (gather == 2) {
        if (!host_out) return fail(ST_ERR_INVALID, "gather 2 needs the shared host frame");
        if ((rc = copy_rows_out(e, cs, host_frame(cs, host_out, format), bounds[e->rank].first, bounds[e->rank].second))) return rc;
        if (!e->async_output) CK(cudaStreamSynchronize(e->stream));
        return ST_OK;
    }
    // assemble the composed frame on rank 0 (strips travel in the requested output format)
    // RGBA32F strips travel straight from `output` as floats, the converted formats from a staging slot as bytes
    const size_t W = cs->desc.width, n = W * cs->desc.height, px_bytes = format_bpp(format);
    if (!px_bytes) return fail(ST_ERR_INVALID, "unsupported output format");
    char* base; ncclDataType_t dt; size_t per_px;
    if (format == ST_FORMAT_RGBA32F) { base = (char*)cs->dev.output; dt = ncclFloat; per_px = 4; }
    else {
        if ((rc = cs->staging.ensure(2 * n * kStagingBpp))) return rc;
        cs->staging_slot ^= 1;
        SceneDev sc = e->scene(); char* slot = (char*)cs->staging.p + (cs->staging_slot ? n * kStagingBpp : 0);
        ViewSet v(1, view_of(cs, cs, 0)); v[0].dst = slot; v[0].pitch = W * px_bytes;
        e->run_timed(P_COMPOSITION, [&](cudaStream_t s) { launch_output_store(v, sc, format, s); });
        base = slot; dt = ncclUint8; per_px = px_bytes;
    }
    if (peer) {
        PeerExchange x; peer_fill(e, cs, &x);
        if (e->rank != 0) {
            size_t first = (size_t)bounds[e->rank].first * W * px_bytes, bytes = (size_t)(bounds[e->rank].second - bounds[e->rank].first) * W * px_bytes;
            if (first % 16 || bytes % 16) return fail(ST_ERR_INVALID, "the strip gather needs strips that start and end on 16-byte boundaries");
            char* remote = format == ST_FORMAT_RGBA32F ? cs->peer.arena[0] + (size_t)(base - (char*)cs->arena.p) : cs->peer.staging[0] + (size_t)(base - (char*)cs->staging.p);
            x.seg[x.nseg++] = {(const uint4*)(base + first), (uint4*)(remote + first), bytes / 16};
        }
        peer_flush(e, cs, &x, true);
    } else if (e->n_ranks > 1) {
        g_nccl.GroupStart();
        for (int src = 1; src < e->n_ranks; src++) {
            char* ptr = base + (size_t)bounds[src].first * W * px_bytes; size_t count = (size_t)(bounds[src].second - bounds[src].first) * W * per_px;
            if (e->rank == src) g_nccl.Send(ptr, count, dt, 0, e->comm, e->stream);
            else if (e->rank == 0) g_nccl.Recv(ptr, count, dt, src, e->comm, e->stream);
        }
        ncclResult_t r = g_nccl.GroupEnd();
        if (r != ncclSuccess) return fail(ST_ERR_CUDA, std::string("output gather: ") + g_nccl.GetErrorString(r));
    }
    if (host_out && e->rank == 0) {
        CK(cudaMemcpyAsync(host_out, base, n * px_bytes, cudaMemcpyDeviceToHost, e->stream));
        if (!e->async_output) CK(cudaStreamSynchronize(e->stream));
    }
    return ST_OK;
}
// Links engines that live in THIS process into a strip group (rank = index): enables peer access between their devices and hands every
// engine the others' buffers directly (the multi-process route is st_peer_export / st_peer_import over CUDA IPC).  Two ranks may share
// a device, which is how a single-GPU box exercises the whole protocol.
static int link_prepare(st_engine* e, CameraSlot* cs) {
    CK(cudaSetDevice(e->device));
    size_t n = (size_t)cs->desc.width * cs->desc.height;
    int rc = cs->staging.ensure(2 * n * kStagingBpp); if (rc) return rc;
    if ((rc = cs->peer.sync.ensure(kSyncBytes))) return rc;
    const int need0[2] = {(int)cs->desc.height, -1};
    CK(cudaMemcpy((uint32_t*)cs->peer.sync.p + kNeedRowsWord, need0, 8, cudaMemcpyHostToDevice));
    return ST_OK;
}
int st_link_local(st_engine* const* engines, const st_camera_handle* cameras, int n) {
    if (!engines || !cameras || n < 1 || n > ST_PEER_MAX_RANKS) return fail(ST_ERR_LIMIT, "1..16 engines");
    std::vector<CameraSlot*> cams(n);
    for (int r = 0; r < n; r++) {
        cams[r] = engines[r] ? get_camera(engines[r], cameras[r]) : nullptr;
        if (!cams[r]) return fail(ST_ERR_NOT_FOUND, "unknown camera");
        if (cams[r]->desc.width != cams[0]->desc.width || cams[r]->desc.height != cams[0]->desc.height) return fail(ST_ERR_INVALID, "linked cameras must have one size");
        int rc = link_prepare(engines[r], cams[r]); if (rc) return rc;
    }
    for (int a = 0; a < n; a++) for (int b = 0; b < n; b++) {
        if (engines[a]->device == engines[b]->device) continue;
        int can = 0; CK(cudaDeviceCanAccessPeer(&can, engines[a]->device, engines[b]->device));
        if (!can) return fail(ST_ERR_CUDA, "devices cannot access each other's memory");
        CK(cudaSetDevice(engines[a]->device));
        cudaError_t ce = cudaDeviceEnablePeerAccess(engines[b]->device, 0);
        if (ce != cudaSuccess && ce != cudaErrorPeerAccessAlreadyEnabled) return fail(ST_ERR_CUDA, std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(ce));
        cudaGetLastError();
    }
    for (int r = 0; r < n; r++) {
        CameraSlot* cs = cams[r];
        cs->peer.arena.assign(n, nullptr); cs->peer.staging.assign(n, nullptr); cs->peer.flags.assign(n, nullptr);
        for (int q = 0; q < n; q++) { cs->peer.arena[q] = (char*)cams[q]->arena.p; cs->peer.flags[q] = (uint32_t*)cams[q]->peer.sync.p; cs->peer.staging[q] = (char*)cams[q]->staging.p; }
        engines[r]->rank = r; engines[r]->n_ranks = n; cs->peer.seq = 0; cs->peer.fseq = 0; cs->peer.ready = true; cs->peer.ipc = false;
    }
    for (int r = 0; r < n; r++) { int rc = strip_streams_prepare(engines[r], cams[r]); if (rc) return rc; }
    return ST_OK;
}
int st_halo_bytes(st_engine* e, uint64_t* bytes) { if (!e || !bytes) return fail(ST_ERR_INVALID, "null argument"); *bytes = e->halo_bytes_last_frame; return ST_OK; }
int st_mark_begin(st_engine* e) {
    if (!e) return fail(ST_ERR_INVALID, "null engine");
    CK(cudaSetDevice(e->device));
    if (!e->mark_a) { CK(cudaEventCreate(&e->mark_a)); CK(cudaEventCreate(&e->mark_b)); }
    CK(cudaEventRecord(e->mark_a, e->stream));
    return ST_OK;
}
int st_mark_end(st_engine* e, float* ms) {
    if (!e || !ms || !e->mark_a) return fail(ST_ERR_INVALID, "st_mark_begin first");
    CK(cudaSetDevice(e->device));
    CK(cudaEventRecord(e->mark_b, e->stream));
    CK(cudaEventSynchronize(e->mark_b));
    CK(cudaEventElapsedTime(ms, e->mark_a, e->mark_b));
    return ST_OK;
}
int st_enable_timing(st_engine* e, int enabled) { if (!e) return fail(ST_ERR_INVALID, "null engine"); e->timing = enabled != 0; return ST_OK; }
int st_pass_times(st_engine* e, float* ms, uint32_t* launches, int reset) {
    if (!e) return fail(ST_ERR_INVALID, "null engine");
    CK(cudaSetDevice(e->device));
    e->collect_timing();
    for (int i = 0; i < P_COUNT; i++) { if (ms) ms[i] = e->pass_ms[i]; if (launches) launches[i] = e->pass_launches[i]; }
    if (reset) { std::memset(e->pass_ms, 0, sizeof e->pass_ms); std::memset(e->pass_launches, 0, sizeof e->pass_launches); }
    return ST_OK;
}

/* K22 per à-trous iteration (stride 2^i): device time and launch count since the last reset (timing enabled). */
int st_wavelet_times(st_engine* e, float* ms5, uint32_t* launches5, int reset) {
    if (!e) return fail(ST_ERR_INVALID, "null engine");
    CK(cudaSetDevice(e->device));
    e->collect_timing();
    for (int i = 0; i < 5; i++) { if (ms5) ms5[i] = e->wavelet_ms[i]; if (launches5) launches5[i] = e->wavelet_launches[i]; }
    if (reset) { std::memset(e->wavelet_ms, 0, sizeof e->wavelet_ms); std::memset(e->wavelet_launches, 0, sizeof e->wavelet_launches); }
    return ST_OK;
}

// =================================================================================================
// st_multi: ONE host process driving several devices (SURVEY §8b: "st_engine_create(device_ordinals[], n)").
// A thin group over n engines: scene verbs are replayed on every member (the scene is replicated, SURVEY §8e), a camera is created on
// every member and linked (st_link_local), st_multi_render_camera enqueues every rank's strip of the frame (fused transport) and then
// lets every rank copy its own rows into the caller's frame.  What a single-process host (the Bevy plugin) binds instead of st_engine.
// =================================================================================================
// cams[c][rank]: camera c's handle on member `rank` (-1 where it has none).  home[c]: ST_PLACE_STRIPS for a strip camera (one on every member,
// linked), or the one member a placed camera lives on (st_multi_create_camera_on).
struct st_multi { std::vector<st_engine*> e; std::vector<std::vector<st_camera_handle>> cams; std::vector<int> home; };
#define ST_MULTI_ALL(call) do { if (!m) return fail(ST_ERR_INVALID, "null group"); for (st_engine* e : m->e) { int rc_ = (call); if (rc_) return rc_; } return ST_OK; } while (0)
int st_multi_create(const int* devices, int n, st_multi** out) {
    if (!devices || !out || n < 1 || n > ST_PEER_MAX_RANKS) return fail(ST_ERR_LIMIT, "1..16 devices");
    st_multi* m = new st_multi();
    for (int i = 0; i < n; i++) { st_engine* e = nullptr; int rc = st_engine_create(devices[i], &e); if (rc) { for (st_engine* x : m->e) st_engine_destroy(x); delete m; return rc; } m->e.push_back(e); }
    *out = m;
    return ST_OK;
}
void st_multi_destroy(st_multi* m) { if (!m) return; for (st_engine* e : m->e) { cudaSetDevice(e->device); cudaStreamSynchronize(e->stream); } for (st_engine* e : m->e) st_engine_destroy(e); delete m; }
int st_multi_size(st_multi* m) { return m ? (int)m->e.size() : 0; }
st_engine* st_multi_engine(st_multi* m, int rank) { return (m && rank >= 0 && rank < (int)m->e.size()) ? m->e[rank] : nullptr; }
int st_multi_insert_mesh(st_multi* m, st_handle mesh, const st_mesh_triangle* t, size_t count) { ST_MULTI_ALL(st_insert_mesh(e, mesh, t, count)); }
int st_multi_remove_mesh(st_multi* m, st_handle mesh) { ST_MULTI_ALL(st_remove_mesh(e, mesh)); }
int st_multi_insert_material(st_multi* m, st_handle h, const st_material* mat) { ST_MULTI_ALL(st_insert_material(e, h, mat)); }
int st_multi_has_material(st_multi* m, st_handle h) { return (m && !m->e.empty()) ? st_has_material(m->e[0], h) : 0; }
int st_multi_remove_material(st_multi* m, st_handle h) { ST_MULTI_ALL(st_remove_material(e, h)); }
int st_multi_insert_image(st_multi* m, st_handle h, const uint8_t* rgba8, uint32_t w, uint32_t hgt) { ST_MULTI_ALL(st_insert_image(e, h, rgba8, w, hgt)); }
int st_multi_remove_image(st_multi* m, st_handle h) { ST_MULTI_ALL(st_remove_image(e, h)); }
int st_multi_set_material_textures(st_multi* m, st_handle h, const st_material_textures* t) { ST_MULTI_ALL(st_set_material_textures(e, h, t)); }
int st_multi_insert_instance(st_multi* m, st_handle h, st_handle mesh, st_handle material, const float a[12]) { ST_MULTI_ALL(st_insert_instance(e, h, mesh, material, a)); }
int st_multi_remove_instance(st_multi* m, st_handle h) { ST_MULTI_ALL(st_remove_instance(e, h)); }
int st_multi_insert_light(st_multi* m, st_handle h, const st_light* l) { ST_MULTI_ALL(st_insert_light(e, h, l)); }
int st_multi_remove_light(st_multi* m, st_handle h) { ST_MULTI_ALL(st_remove_light(e, h)); }
int st_multi_update_sun(st_multi* m, float az, float alt) { ST_MULTI_ALL(st_update_sun(e, az, alt)); }
int st_multi_set_option(st_multi* m, int option, int value) { ST_MULTI_ALL(st_set_option(e, option, value)); }
int st_multi_set_seed_base(st_multi* m, uint32_t base) { ST_MULTI_ALL(st_set_seed_base(e, base)); }
int st_multi_set_blue_noise(st_multi* m, const uint8_t* rgba) { ST_MULTI_ALL(st_set_blue_noise(e, rgba)); }
int st_multi_insert_dynamic_image(st_multi* m, st_handle h, const void* src, size_t pitch, uint32_t w, uint32_t hgt) {
    if (!m) return fail(ST_ERR_INVALID, "null group");
    std::vector<OutputTarget> t(m->e.size());
    for (size_t i = 0; i < m->e.size(); i++) {   // every member must reach the surface before any of them registers it
        CK(cudaSetDevice(m->e[i]->device));
        int rc = dynamic_source(m->e[i], src, pitch, w, hgt, &t[i]); if (rc) return rc;
    }
    for (size_t i = 0; i < m->e.size(); i++) { int rc = insert_dynamic(m->e[i], h, t[i], w, hgt); if (rc) return rc; }
    return ST_OK;
}
int st_multi_tick(st_multi* m) {
    if (!m) return fail(ST_ERR_INVALID, "null group");
    // Every member stores its own rows of a group camera's frame, so a surface one member refreshes from may hold rows the others wrote: each
    // member's refresh first waits for everything the other members have queued (their output copies included).
    bool dynamic = false;
    for (st_engine* e : m->e) dynamic |= !e->dynamic.empty();
    if (dynamic && m->e.size() > 1) {
        for (st_engine* e : m->e) {
            CK(cudaSetDevice(e->device));
            if (!e->ev_queued) CK(cudaEventCreateWithFlags(&e->ev_queued, cudaEventDisableTiming));
            int rc = wait_output_copies(e); if (rc) return rc;
            CK(cudaEventRecord(e->ev_queued, e->stream));
        }
        for (st_engine* e : m->e) {
            CK(cudaSetDevice(e->device));
            for (st_engine* o : m->e) if (o != e) CK(cudaStreamWaitEvent(e->stream, o->ev_queued, 0));
        }
    }
    ST_MULTI_ALL(st_tick(e));
}
int st_multi_synchronize(st_multi* m) { ST_MULTI_ALL(st_synchronize(e)); }
int st_multi_create_camera(st_multi* m, const st_camera* c, st_camera_handle* out) {
    if (!m || !c || !out) return fail(ST_ERR_INVALID, "null argument");
    std::vector<st_camera_handle> hs(m->e.size());
    for (size_t i = 0; i < m->e.size(); i++) { int rc = st_create_camera(m->e[i], c, &hs[i]); if (rc) return rc; }
    if (m->e.size() > 1) { int rc = st_link_local(m->e.data(), hs.data(), (int)m->e.size()); if (rc) return rc; }
    m->cams.push_back(hs); m->home.push_back(ST_PLACE_STRIPS);
    *out = (st_camera_handle)m->cams.size() - 1;
    return ST_OK;
}
// camera `h` of the group, placed on one member: *rank = that member, *cs = its slot there.  ST_ERR_NOT_FOUND for an unknown or deleted
// camera; nullptr in *cs and ST_OK for a strip camera.
static int placed_camera(st_multi* m, st_camera_handle h, int* rank, CameraSlot** cs) {
    if (!m || h < 0 || (size_t)h >= m->cams.size()) return fail(ST_ERR_NOT_FOUND, "unknown camera " + std::to_string(h));
    *rank = m->home[h]; *cs = nullptr;
    const int r = *rank >= 0 ? *rank : 0;
    CameraSlot* c = get_camera(m->e[r], m->cams[h][r]);
    if (!c) return fail(ST_ERR_NOT_FOUND, "camera " + std::to_string(h) + " was deleted");
    if (*rank >= 0) *cs = c;
    return ST_OK;
}
int st_multi_create_camera_on(st_multi* m, const st_camera* c, int rank, st_camera_handle* out) {
    if (!m || !c || !out) return fail(ST_ERR_INVALID, "null argument");
    const int n = (int)m->e.size();
    if (rank == ST_PLACE_AUTO) {   // the member with the fewest pixels of placed cameras, the lowest rank on a tie
        std::vector<uint64_t> pixels(n, 0);
        for (size_t k = 0; k < m->cams.size(); k++) {
            const int r = m->home[k];
            const CameraSlot* cs = r >= 0 ? get_camera(m->e[r], m->cams[k][r]) : nullptr;
            if (cs) pixels[r] += (uint64_t)cs->desc.width * cs->desc.height;
        }
        rank = (int)(std::min_element(pixels.begin(), pixels.end()) - pixels.begin());
    }
    if (rank < 0 || rank >= n) return fail(ST_ERR_INVALID, "rank " + std::to_string(rank) + " is not a member of this group of " + std::to_string(n));
    st_camera_handle mh = -1;
    int rc = st_create_camera(m->e[rank], c, &mh); if (rc) return rc;
    std::vector<st_camera_handle> hs(n, -1); hs[rank] = mh;
    m->cams.push_back(hs); m->home.push_back(rank);
    *out = (st_camera_handle)m->cams.size() - 1;
    return ST_OK;
}
int st_multi_camera_rank(st_multi* m, st_camera_handle h, int* rank) {
    if (!rank) return fail(ST_ERR_INVALID, "null argument");
    CameraSlot* cs = nullptr; int r = 0;
    int rc = placed_camera(m, h, &r, &cs); if (rc) return rc;
    *rank = r;
    return ST_OK;
}
// The camera's complete state travels: the arena (every named buffer, history included), the paired à-trous scratch, the camera uniforms
// of this and the last frame, and the frame it was ticked for.  The arenas of one size have one layout, so one copy each suffices.
int st_multi_move_camera(st_multi* m, st_camera_handle h, int rank) {
    CameraSlot* cs = nullptr; int from = 0;
    int rc = placed_camera(m, h, &from, &cs); if (rc) return rc;
    if (!cs) return fail(ST_ERR_INVALID, "camera " + std::to_string(h) + " is a strip camera; only placed cameras move");
    if (rank < 0 || rank >= (int)m->e.size()) return fail(ST_ERR_INVALID, "rank " + std::to_string(rank) + " is not a member of this group of " + std::to_string(m->e.size()));
    if (rank == from) return ST_OK;
    st_engine *src = m->e[from], *dst = m->e[rank];
    if ((rc = st_synchronize(src))) return rc;   // the source's queued passes and output copies are done with the arena
    CK(cudaSetDevice(dst->device));
    CameraSlot* ns = new CameraSlot();
    ns->alive = true; ns->desc = cs->desc;
    auto undo = [&](int code) { ns->arena.release(); ns->svgf_pairs.release(); delete ns; return code; };
    if ((rc = allocate_camera(dst, ns))) return undo(rc);
    if (ns->arena.cap != cs->arena.cap || ns->svgf_pairs.cap != cs->svgf_pairs.cap) return undo(fail(ST_ERR_INVALID, "arena layouts differ"));
    // behind allocate_camera's fills on the target's stream; a peer copy when the devices differ
    cudaError_t ce = cudaMemcpyPeerAsync(ns->arena.p, dst->device, cs->arena.p, src->device, cs->arena.cap, dst->stream);
    if (ce == cudaSuccess && cs->svgf_pairs.p) ce = cudaMemcpyPeerAsync(ns->svgf_pairs.p, dst->device, cs->svgf_pairs.p, src->device, cs->svgf_pairs.cap, dst->stream);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(dst->stream);
    if (ce != cudaSuccess) { cudaGetLastError(); return undo(fail(ST_ERR_CUDA, std::string("camera move: ") + cudaGetErrorString(ce))); }
    ns->dev.curr = cs->dev.curr; ns->dev.prev = cs->dev.prev; ns->frame = cs->frame;
    dst->cameras.push_back(ns);
    const st_camera_handle old = m->cams[h][from];
    m->cams[h][from] = -1; m->cams[h][rank] = (st_camera_handle)dst->cameras.size() - 1; m->home[h] = rank;
    return st_delete_camera(src, old);
}
int st_multi_update_camera(st_multi* m, st_camera_handle h, const st_camera* c) {
    if (!m || h < 0 || (size_t)h >= m->cams.size() || !c) return fail(ST_ERR_NOT_FOUND, "unknown camera");
    if (m->home[h] >= 0) return st_update_camera(m->e[m->home[h]], m->cams[h][m->home[h]], c);   // a resize re-creates the buffers there only
    bool relink = false;
    for (size_t i = 0; i < m->e.size(); i++) {
        CameraSlot* cs = get_camera(m->e[i], m->cams[h][i]);
        if (!cs) return fail(ST_ERR_NOT_FOUND, "unknown camera");
        relink |= cs->desc.mode != c->mode || cs->desc.denoise != c->denoise || cs->desc.ref_depth != c->ref_depth || cs->desc.width != c->width || cs->desc.height != c->height;
    }
    if (relink) for (st_engine* e : m->e) { cudaSetDevice(e->device); cudaStreamSynchronize(e->stream); }   // buffers are re-created: nobody may still be writing into them
    for (size_t i = 0; i < m->e.size(); i++) { int rc = st_update_camera(m->e[i], m->cams[h][i], c); if (rc) return rc; }
    if (relink && m->e.size() > 1) return st_link_local(m->e.data(), m->cams[h].data(), (int)m->e.size());
    return ST_OK;
}
int st_multi_delete_camera(st_multi* m, st_camera_handle h) {
    if (!m || h < 0 || (size_t)h >= m->cams.size()) return fail(ST_ERR_NOT_FOUND, "unknown camera");
    if (m->home[h] >= 0) return st_delete_camera(m->e[m->home[h]], m->cams[h][m->home[h]]);
    for (st_engine* e : m->e) { cudaSetDevice(e->device); cudaStreamSynchronize(e->stream); }
    for (size_t i = 0; i < m->e.size(); i++) { int rc = st_delete_camera(m->e[i], m->cams[h][i]); if (rc) return rc; }
    return ST_OK;
}
st_camera_handle st_multi_member_camera(st_multi* m, st_camera_handle h, int rank) { return (m && h >= 0 && (size_t)h < m->cams.size() && rank >= 0 && (size_t)rank < m->e.size()) ? m->cams[h][rank] : -1; }
// Engine::render_camera for the group.  All ranks' frames are enqueued before any output is issued and nothing in between
// synchronises: the ranks wait for each other on the device (sequence flags), never on the host.  Then every rank stores its own rows
// [y0, y1) into its target (targets[rank]: the same surface, reached from that rank's device); targets == nullptr = enqueue only.
static int multi_render(st_multi* m, st_camera_handle h, const OutputTarget* targets) {
    const size_t n = m->e.size();
    std::vector<CameraSlot*> cs(n);
    for (size_t i = 0; i < n; i++) {   // first-use allocations and LUT generation synchronise their device: do them before anything can wait on a peer
        cs[i] = get_camera(m->e[i], m->cams[h][i]);
        if (!cs[i]) return fail(ST_ERR_NOT_FOUND, "unknown camera");
        CK(cudaSetDevice(m->e[i]->device));
        int rc = ensure_luts(m->e[i]); if (rc) return rc;
    }
    for (size_t i = 0; i < n; i++) { CK(cudaSetDevice(m->e[i]->device)); int rc = enqueue_strip_frame(m->e[i], cs[i], 16); if (rc) return rc; }
    if (!targets) return ST_OK;
    std::vector<std::pair<int, int>> bounds; strip_bounds((int)cs[0]->desc.height, (int)n, &bounds);
    for (size_t i = 0; i < n; i++) { CK(cudaSetDevice(m->e[i]->device)); int rc = copy_rows_out(m->e[i], cs[i], targets[i], bounds[i].first, bounds[i].second); if (rc) return rc; }
    for (size_t i = 0; i < n; i++) if (!targets[i].device && !m->e[i]->async_output) { CK(cudaSetDevice(m->e[i]->device)); CK(cudaStreamSynchronize(m->e[i]->stream)); }
    return ST_OK;
}
int st_multi_render_camera(st_multi* m, st_camera_handle h, void* host_out, int format) {
    if (!m || h < 0 || (size_t)h >= m->cams.size()) return fail(ST_ERR_NOT_FOUND, "unknown camera");
    if (m->e.size() == 1) return st_render_camera(m->e[0], m->cams[h][0], host_out, format);
    if (m->home[h] >= 0) return st_render_camera(m->e[m->home[h]], m->cams[h][m->home[h]], host_out, format);   // a whole frame on its member
    std::vector<OutputTarget> t;
    for (size_t i = 0; host_out && i < m->e.size(); i++) {
        CameraSlot* cs = get_camera(m->e[i], m->cams[h][i]);
        if (!cs) return fail(ST_ERR_NOT_FOUND, "unknown camera");
        t.push_back(host_frame(cs, host_out, format));
    }
    return multi_render(m, h, host_out ? t.data() : nullptr);
}
int st_multi_render_camera_to(st_multi* m, st_camera_handle h, void* dst, size_t pitch, int format) {
    if (!m || h < 0 || (size_t)h >= m->cams.size()) return fail(ST_ERR_NOT_FOUND, "unknown camera");
    if (m->e.size() == 1) return st_render_camera_to(m->e[0], m->cams[h][0], dst, pitch, format);
    if (m->home[h] >= 0) return st_render_camera_to(m->e[m->home[h]], m->cams[h][m->home[h]], dst, pitch, format);
    std::vector<OutputTarget> t(m->e.size());
    for (size_t i = 0; i < m->e.size(); i++) {   // every member must reach the surface before any of them renders
        CameraSlot* cs = get_camera(m->e[i], m->cams[h][i]);
        if (!cs) return fail(ST_ERR_NOT_FOUND, "unknown camera");
        CK(cudaSetDevice(m->e[i]->device));
        int rc = resolve_target(m->e[i], cs->desc.width, dst, pitch, format, &t[i]); if (rc) return rc;
    }
    return multi_render(m, h, t.data());
}
// per-camera buffer of the whole frame, assembled from the members' strips (test hook, cf. st_read_buffer)
int st_multi_read_buffer(st_multi* m, st_camera_handle h, const char* name, float* dst, size_t cap, size_t* count) {
    if (!m || h < 0 || (size_t)h >= m->cams.size() || !name || !count) return fail(ST_ERR_NOT_FOUND, "unknown camera");
    if (m->home[h] >= 0) return st_read_buffer(m->e[m->home[h]], m->cams[h][m->home[h]], name, dst, cap, count);
    const size_t n = m->e.size();
    int rc = st_read_buffer(m->e[0], m->cams[h][0], name, nullptr, 0, count); if (rc) return rc;
    if (!dst) return ST_OK;
    if (cap < *count) return fail(ST_ERR_LIMIT, "buffer too small");
    CameraSlot* c0 = get_camera(m->e[0], m->cams[h][0]);
    std::vector<std::pair<int, int>> bounds; strip_bounds((int)c0->desc.height, (int)n, &bounds);
    const size_t per_row = *count / c0->desc.height;
    for (size_t i = 0; i < n; i++) {
        void* p = nullptr; size_t bytes = 0;
        if ((rc = st_buffer_device_ptr(m->e[i], m->cams[h][i], name, &p, &bytes))) return rc;
        CK(cudaSetDevice(m->e[i]->device)); CK(cudaStreamSynchronize(m->e[i]->stream));
        size_t a = (size_t)bounds[i].first * per_row, b = (size_t)bounds[i].second * per_row;
        CK(cudaMemcpy(dst + a, (const float*)p + a, (b - a) * 4, cudaMemcpyDeviceToHost));
    }
    return ST_OK;
}
int st_multi_peer_errors(st_multi* m, st_camera_handle h, uint32_t* count) {
    if (!m || h < 0 || (size_t)h >= m->cams.size() || !count) return fail(ST_ERR_NOT_FOUND, "unknown camera");
    *count = 0;
    if (m->home[h] >= 0) return get_camera(m->e[m->home[h]], m->cams[h][m->home[h]]) ? ST_OK : fail(ST_ERR_NOT_FOUND, "unknown camera");   // no peer link
    for (size_t i = 0; i < m->e.size(); i++) { uint32_t c = 0; int rc = st_peer_errors(m->e[i], m->cams[h][i], &c); if (rc) return rc; *count += c; }
    return ST_OK;
}
// st_render_cameras for the group: every member renders the listed cameras that live on it as batched groups, all members at once.  Each
// step runs on every member before the next one starts, so that no member's enqueue waits on the host: every check; the LUTs (which
// synchronise their device); the passes and device-surface stores; the host-surface copies; the synchronisation of members that copied.
int st_multi_render_cameras(st_multi* m, const st_camera_handle* cameras, int n, void* const* dsts, const size_t* pitch_bytes, int format) {
    if (!m) return fail(ST_ERR_INVALID, "null group");
    if (n <= 0 || !cameras) return fail(ST_ERR_INVALID, "no cameras to render");
    const size_t world = m->e.size();
    std::vector<std::vector<st_camera_handle>> hs(world);   // per member, in list order: member handles, surfaces, pitches
    std::vector<std::vector<void*>> ds(world);
    std::vector<std::vector<size_t>> ps(world);
    for (int i = 0; i < n; i++) {
        const st_camera_handle h = cameras[i];
        if (h < 0 || (size_t)h >= m->cams.size()) return fail(ST_ERR_NOT_FOUND, "unknown camera " + std::to_string(h));
        if (std::find(cameras, cameras + i, h) != cameras + i) return fail(ST_ERR_INVALID, "camera " + std::to_string(h) + " is listed twice");
        if (m->home[h] < 0 && world > 1) return fail(ST_ERR_INVALID, "camera " + std::to_string(h) + " is a strip camera; st_multi_render_cameras takes placed cameras");
        const int r = m->home[h] >= 0 ? m->home[h] : 0;
        hs[r].push_back(m->cams[h][r]); ds[r].push_back(dsts ? dsts[i] : nullptr); ps[r].push_back(pitch_bytes ? pitch_bytes[i] : 0);
    }
    if (world == 1) return st_render_cameras(m->e[0], hs[0].data(), n, dsts, pitch_bytes, format);
    std::vector<CameraBatch> b(world);
    for (size_t r = 0; r < world; r++) if (!hs[r].empty()) { int rc = batch_check(m->e[r], hs[r].data(), (int)hs[r].size(), ds[r].data(), ps[r].data(), format, &b[r]); if (rc) return rc; }
    for (size_t r = 0; r < world; r++) if (!hs[r].empty()) { CK(cudaSetDevice(m->e[r]->device)); int rc = ensure_luts(m->e[r]); if (rc) return rc; }
    for (size_t r = 0; r < world; r++) if (!hs[r].empty()) { int rc = batch_enqueue(m->e[r], b[r], format); if (rc) return rc; }
    std::vector<char> host_out(world, 0);
    for (size_t r = 0; r < world; r++) if (!hs[r].empty()) { bool h = false; int rc = batch_copy_out(m->e[r], b[r], &h); if (rc) return rc; host_out[r] = h; }
    for (size_t r = 0; r < world; r++) if (host_out[r] && !m->e[r]->async_output) { CK(cudaSetDevice(m->e[r]->device)); CK(cudaStreamSynchronize(m->e[r]->stream)); }
    return ST_OK;
}

}  // extern "C"
