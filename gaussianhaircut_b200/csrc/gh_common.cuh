// Shared device/host definitions for the B200-native strand-aligned Gaussian rasterizer.
//
// Replaces (as a fresh design, not a translation) the per-stage plumbing of the reference's
// ext/diff_gaussian_rasterization_hair/cuda_rasterizer/{config.h, auxiliary.h, rasterizer_impl.h}.
//
// Rounding contract: every expression that feeds a *decision* of the reference (tile membership,
// depth key bits, alpha < 1/255, T < 1e-4) is written with explicit round-to-nearest intrinsics in
// exactly the operation order nvcc 12.9 + ptxas emit for the reference sources with its default
// flags (-fmad=true, IEEE div/sqrt, precise expf), read off the reference build's SASS
// (cuobjdump -sass oracle/_ref/obj/forward.cu.o): NVVM fuses the LEFT product of `a*b + c*d` into
// the add, ptxas then also fuses `a*b - c*d` into fma(a,b,-(c*d)) and `m*m - d` into fma(m,m,-d);
// 1.f/x is an IEEE reciprocal.  Writing the intrinsics out makes the result independent of this
// compiler's own contraction choices.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define GH_NUM_CHANNELS 10   // reference config.h:15
#define GH_BLOCK_X 16        // reference config.h:16
#define GH_BLOCK_Y 16        // reference config.h:17
#define GH_TILE_PIX (GH_BLOCK_X * GH_BLOCK_Y)

// error bits in GhCtrl::err_flags
#define GH_ERR_PREFILTERED 1u   // a point failed the near cull although prefiltered=true (auxiliary.h:156-160)

#define GH_MUL(a, b) __fmul_rn((a), (b))
#define GH_ADD(a, b) __fadd_rn((a), (b))
#define GH_SUB(a, b) __fsub_rn((a), (b))
#define GH_FMA(a, b, c) __fmaf_rn((a), (b), (c))
#define GH_DIV(a, b) __fdiv_rn((a), (b))
#define GH_RCP(a) __frcp_rn((a))
#define GH_SQRT(a) __fsqrt_rn((a))

// Per-Gaussian 2-D state consumed by both blend kernels: one 32-byte sector per Gaussian.
//   (x, y)      pixel-space mean                       (reference geomState.means2D)
//   (ca,cb,cc)  conic, op = opacity                     (reference geomState.conic_opacity)
//   thr         ln(255*op): the Gaussian can reach alpha >= 1/255 only where power >= -thr
//   pd          1.0f if the conic is positive definite (cull test valid), else 0.0f
struct __align__(16) GhGeo {
    float x, y, ca, cb;
    float cc, op, thr, pd;
};

struct GhCtrl {
    unsigned int num_rendered;   // R = sum of per-tile instance counts
    unsigned int max_tile_len;   // longest per-tile list
    unsigned int err_flags;
    unsigned int nseg;           // segments produced by the long-list split (gh_binning.cu)
};

static __host__ __device__ __forceinline__ size_t gh_align_up(size_t v, size_t a) {
    return (v + a - 1) / a * a;
}

// ---- opaque workspace layouts (new build is free to choose them: SURVEY.md section 8 a11) ----
struct GhGeomWS {
    GhGeo* geo;      // [P]
    float* depth;    // [P] view-space z (key low word)
    float* acc16;    // [P][16] backward accumulation records (64 B each): dL/d colors 0..9,
                     //         mean2D.x, mean2D.y, conic.x, conic.y, conic.w, opacity
    static __host__ __device__ size_t bytes(size_t P) {
        return gh_align_up(P * sizeof(GhGeo), 256) + gh_align_up(P * sizeof(float), 256) +
               gh_align_up(P * 64, 256) + 256;
    }
    static __host__ __device__ GhGeomWS carve(char* base, size_t P) {
        GhGeomWS w;
        size_t off = gh_align_up((size_t)base, 256) - (size_t)base;
        w.geo = (GhGeo*)(base + off); off += gh_align_up(P * sizeof(GhGeo), 256);
        w.depth = (float*)(base + off); off += gh_align_up(P * sizeof(float), 256);
        w.acc16 = (float*)(base + off);
        return w;
    }
};

struct GhImgWS {
    GhCtrl* ctrl;            // [1]
    uint32_t* tile_count;    // [T]   instances per tile
    uint32_t* tile_cursor;   // [T]   emit cursors
    uint2* ranges;           // [T]   (start, end) into the sorted instance list; (0,0) if empty
    uint32_t* tile_perm;     // [T]   launch order of the blend kernels: tiles by decreasing list length
    float* final_T;          // [W*H]
    uint32_t* n_contrib;     // [W*H] 1-based list position of the last blended instance
    static __host__ __device__ size_t bytes(size_t npix, size_t T) {
        return 256 + 3 * gh_align_up(T * 4, 256) + gh_align_up(T * 8, 256) +
               2 * gh_align_up(npix * 4, 256) + 256;
    }
    static __host__ __device__ GhImgWS carve(char* base, size_t npix, size_t T) {
        GhImgWS w;
        size_t off = gh_align_up((size_t)base, 256) - (size_t)base;
        w.ctrl = (GhCtrl*)(base + off); off += 256;
        w.tile_count = (uint32_t*)(base + off); off += gh_align_up(T * 4, 256);
        w.tile_cursor = (uint32_t*)(base + off); off += gh_align_up(T * 4, 256);
        w.ranges = (uint2*)(base + off); off += gh_align_up(T * 8, 256);
        w.tile_perm = (uint32_t*)(base + off); off += gh_align_up(T * 4, 256);
        w.final_T = (float*)(base + off); off += gh_align_up(npix * 4, 256);
        w.n_contrib = (uint32_t*)(base + off);
        return w;
    }
};

struct GhBinWS {
    uint64_t* inst;   // [R]  (depth_bits << 32 | gaussian_idx), bucketed by tile, sorted within a tile
    uint64_t* tmp;    // [R]  scratch of the long-list sort (MSD split target); then, written by the forward blend,
                      //      the backward block mask of each record at its list position (gh_blend.cu)
    uint2* seg;       // [R/768 + R/2048 + 2] (start, length) of the split segments
    static __host__ __device__ size_t max_segments(size_t R) { return R / 768 + R / 2048 + 2; }
    static __host__ __device__ size_t bytes(size_t R) {
        return 2 * gh_align_up(R * 8, 256) + gh_align_up(max_segments(R) * 8, 256) + 256;
    }
    static __host__ __device__ GhBinWS carve(char* base, size_t R) {
        GhBinWS w;
        size_t off = gh_align_up((size_t)base, 256) - (size_t)base;
        w.inst = (uint64_t*)(base + off); off += gh_align_up(R * 8, 256);
        w.tmp = (uint64_t*)(base + off); off += gh_align_up(R * 8, 256);
        w.seg = (uint2*)(base + off);
        return w;
    }
};

#ifdef __CUDACC__
// Tile rectangle of a splat (reference auxiliary.h:46-56, float->int truncation, clamp to grid).
// PTX of the reference: (p - r) * 0.0625 ; ((p + r) + 16) + (-1)) * 0.0625 ; cvt.rzi ; max.s32 0 ; min.u32 grid
__device__ __forceinline__ void gh_get_rect(float px, float py, int radius, int gx, int gy,
                                            int& minx, int& miny, int& maxx, int& maxy) {
    const float rf = (float)radius;
    int v;
    v = __float2int_rz(GH_MUL(GH_SUB(px, rf), 0.0625f)); minx = min(gx, max(0, v));
    v = __float2int_rz(GH_MUL(GH_SUB(py, rf), 0.0625f)); miny = min(gy, max(0, v));
    v = __float2int_rz(GH_MUL(GH_ADD(GH_ADD(GH_ADD(px, rf), 16.0f), -1.0f), 0.0625f)); maxx = min(gx, max(0, v));
    v = __float2int_rz(GH_MUL(GH_ADD(GH_ADD(GH_ADD(py, rf), 16.0f), -1.0f), 0.0625f)); maxy = min(gy, max(0, v));
}

// ---- stage-1 pieces shared by gh_preprocess_kernel and the fused projection kernel (gh_project.cu) -------------
__device__ __forceinline__ float gh_ndc2pix(float v, int S) {
    // auxiliary.h:41-44: ((v + 1.0) * S - 1.0) * 0.5 with double literals -> evaluated in FP64
    double t = __dadd_rn((double)v, 1.0);
    t = __fma_rn(t, (double)S, -1.0);
    t = __dmul_rn(t, 0.5);
    return __double2float_rn(t);
}

// View-space depth + near cull (auxiliary.h:154) and the NDC projection (forward.cu:201-206).  false = culled.
__device__ __forceinline__ bool gh_pre_project(float px, float py, float pz, const float* __restrict__ vm,
                                               const float* __restrict__ pm, float& zview, float& projx, float& projy) {
    zview = GH_ADD(__ldg(vm + 14), GH_FMA(pz, __ldg(vm + 10), GH_FMA(px, __ldg(vm + 2), GH_MUL(py, __ldg(vm + 6)))));
    if (zview <= 0.2f) return false;
    const float hx = GH_ADD(__ldg(pm + 12), GH_FMA(pz, __ldg(pm + 8), GH_FMA(px, __ldg(pm + 0), GH_MUL(py, __ldg(pm + 4)))));
    const float hy = GH_ADD(__ldg(pm + 13), GH_FMA(pz, __ldg(pm + 9), GH_FMA(px, __ldg(pm + 1), GH_MUL(py, __ldg(pm + 5)))));
    const float hw = GH_ADD(__ldg(pm + 15), GH_FMA(pz, __ldg(pm + 11), GH_FMA(px, __ldg(pm + 3), GH_MUL(py, __ldg(pm + 7)))));
    const float p_w = GH_RCP(GH_ADD(hw, 0.0000001f));
    projx = GH_MUL(hx, p_w); projy = GH_MUL(hy, p_w);
    return true;
}

// Caller-supplied conic: invert it to size the splat (forward.cu:238-248).  false = singular (not rendered).
__device__ __forceinline__ bool gh_pre_from_conic(float conx, float cony, float conz, float& covx, float& covz, float& det) {
    const float det_inv = GH_FMA(conx, conz, -GH_MUL(cony, cony));
    if (det_inv == 0.0f) return false;
    det = GH_RCP(det_inv);
    covx = GH_MUL(conz, det);
    covz = GH_MUL(conx, det);
    return true;
}

// Splat extent from the larger eigenvalue (forward.cu:254-257), pixel centre, tile rectangle and the 32-byte state
// record of the blend kernels.  Returns the radius (0 = not rendered; rect and g are then left untouched).
__device__ __forceinline__ int gh_pre_finish(float covx, float covz, float det, float conx, float cony, float conz,
                                             float projx, float projy, float op, int W, int H, int gx, int gy,
                                             int& minx, int& miny, int& maxx, int& maxy, GhGeo& g) {
    const float mid = GH_MUL(GH_ADD(covx, covz), 0.5f);
    const float sq = GH_SQRT(fmaxf(GH_FMA(mid, mid, -det), 0.1f));
    const float lam = fmaxf(GH_ADD(mid, sq), GH_SUB(mid, sq));
    const float my_radius = ceilf(GH_MUL(GH_SQRT(lam), 3.0f));
    const float pix_x = gh_ndc2pix(projx, W), pix_y = gh_ndc2pix(projy, H);
    const int ri = __float2int_rz(my_radius);
    // NaN covariance -> NaN radius -> 0: the reference counts such a Gaussian in tiles_touched but never
    // emits its key (duplicateWithKeys tests radii > 0), leaving an uninitialised record in the list;
    // dropping it here keeps the histogram and the emit consistent
    if (ri <= 0) return 0;
    int x0, y0, x1, y1;
    gh_get_rect(pix_x, pix_y, ri, gx, gy, x0, y0, x1, y1);
    if ((x1 - x0) * (y1 - y0) == 0) return 0;
    g.x = pix_x; g.y = pix_y; g.ca = conx; g.cb = cony; g.cc = conz; g.op = op;
    g.thr = __logf(255.0f * op);           // only used by the conservative cull (slack covers the approx)
    g.thr = (255.0f * op > 0.f) ? g.thr : -1e30f;
    const bool pd = (conx > 0.f) && (conz > 0.f) && (conx * conz - cony * cony > 0.f) && (op == op);
    g.pd = pd ? 1.0f : 0.0f;
    if (!(op == op)) g.thr = 1e30f;        // NaN opacity blends with alpha 0.99 in the reference (min.f32)
    minx = x0; miny = y0; maxx = x1; maxy = y1;
    return ri;
}

__device__ __forceinline__ GhGeo gh_geo_not_rendered() {
    GhGeo g; g.x = 0.f; g.y = 0.f; g.ca = 0.f; g.cb = 0.f; g.cc = 0.f; g.op = 0.f; g.thr = -1e30f; g.pd = 0.f;
    return g;
}

// Warp-cooperative enumeration of the (Gaussian, tile) instances of a warp's 32 tile rectangles.  Splat rectangles
// vary a lot in size (a strand segment seen end-on covers one tile, seen sideways a dozen), so a loop in which every
// lane walks its own rectangle runs as long as the warp's LARGEST one; here the rectangles are flattened into one
// list (warp prefix sum of their sizes) and lane l takes items l, l + 32, ...: ceil(sum / 32) rounds instead of max.
struct GhWarpRects {
    int incl, excl, w, minxy, total;
    uint32_t rw;       // ceil(2^32 / w): k / w == umulhi(k, rw) whenever k * w < 2^32 (w >= 2).  k < w * h for a
                       // rectangle of w x h tiles, so every tile grid with gx * gx * gy < 2^32 is safe (checked by the
                       // host entry points; 1080p: 120 * 120 * 68 = 979 200)
};
__device__ __forceinline__ GhWarpRects gh_warp_rects(int minx, int miny, int maxx, int maxy, int lane) {
    GhWarpRects r;
    r.w = maxx - minx;
    const int count = r.w * (maxy - miny);
    int v = count;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int nb = __shfl_up_sync(0xffffffffu, v, o); if (lane >= o) v += nb; }
    r.incl = v; r.excl = v - count;
    r.total = __shfl_sync(0xffffffffu, v, 31);
    r.minxy = minx | (miny << 16);
    r.rw = (r.w > 1) ? (0xffffffffu / (uint32_t)r.w + 1u) : 0u;
    return r;
}
// item j of the flattened list: returns its tile (y * gx + x) and the lane that owns the rectangle, -1 past the end
__device__ __forceinline__ int gh_warp_rect_item(const GhWarpRects& r, int j, int gx, int& owner) {
    int lo = 0;     // number of lanes whose inclusive sum is <= j == first lane whose rectangle contains item j
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
        const int v = __shfl_sync(0xffffffffu, r.incl, lo + s - 1);
        if (v <= j) lo += s;
    }
    owner = lo;
    const int oexcl = __shfl_sync(0xffffffffu, r.excl, lo);
    const int ow = __shfl_sync(0xffffffffu, r.w, lo);
    const uint32_t orw = __shfl_sync(0xffffffffu, r.rw, lo);
    const int oxy = __shfl_sync(0xffffffffu, r.minxy, lo);
    const uint32_t k = (uint32_t)(j - oexcl);
    const uint32_t q = (ow > 1) ? __umulhi(k, orw) : k;
    const int x = (oxy & 0xffff) + (int)(k - q * (uint32_t)ow), y = (oxy >> 16) + (int)q;
    return (j < r.total) ? y * gx + x : -1;
}

// per-tile histogram of a warp's rectangles (replaces the reference's per-Gaussian tiles_touched + prefix sum): the
// warp walks the flattened list of its (Gaussian, tile) instances.  Neighbouring Gaussians of a strand hit the same
// tiles: lanes asking for the same tile in the same round are grouped with match.any and counted with one atomic.
// Must be called by all 32 lanes (empty rectangle = nothing to count).
__device__ __forceinline__ void gh_warp_tile_histogram(int minx, int miny, int maxx, int maxy, int gx,
                                                       uint32_t* __restrict__ tile_count) {
    const int lane = threadIdx.x & 31;
    const GhWarpRects wr = gh_warp_rects(minx, miny, maxx, maxy, lane);
    for (int j0 = 0; j0 < wr.total; j0 += 32) {
        int owner;
        const int tile = gh_warp_rect_item(wr, j0 + lane, gx, owner);
        const uint32_t peers = __match_any_sync(0xffffffffu, tile);
        if (tile >= 0 && lane == __ffs(peers) - 1) atomicAdd(&tile_count[tile], (uint32_t)__popc(peers));
    }
}

// World-space 3-D covariance from scale * modifier and a RAW (un-normalised) quaternion
// (reference forward.cu:118-152; glm column-major products, see oracle/glm_shim).
// Order of operations transcribed from the reference PTX.
__device__ __forceinline__ void gh_cov3d(float s0, float s1, float s2, float mod,
                                         float r, float x, float y, float z, float* cov) {
    const float sx = GH_MUL(mod, s0), sy = GH_MUL(mod, s1), sz = GH_MUL(mod, s2);
    // operation order of the reference SASS (ptxas fuses one product of each +- pair into an FFMA)
    const float yy = GH_MUL(y, y), zz = GH_MUL(z, z);
    const float xz = GH_MUL(x, z), rx = GH_MUL(r, x), rz = GH_MUL(r, z);
    const float yy_zz = GH_ADD(yy, zz);
    const float xx_zz = GH_FMA(x, x, zz);
    const float xx_yy = GH_FMA(x, x, yy);
    // R columns (glm::mat3 ctor fills columns)
    const float R00 = GH_SUB(1.0f, GH_ADD(yy_zz, yy_zz));
    const float t01 = GH_FMA(x, y, -rz);   const float R01 = GH_ADD(t01, t01);   // 2(xy - rz)
    const float t02 = GH_FMA(r, y, xz);    const float R02 = GH_ADD(t02, t02);   // 2(xz + ry)
    const float t10 = GH_FMA(x, y, rz);    const float R10 = GH_ADD(t10, t10);   // 2(xy + rz)
    const float R11 = GH_SUB(1.0f, GH_ADD(xx_zz, xx_zz));
    const float t12 = GH_FMA(y, z, -rx);   const float R12 = GH_ADD(t12, t12);   // 2(yz - rx)
    const float t20 = GH_FMA(-r, y, xz);   const float R20 = GH_ADD(t20, t20);   // 2(xz - ry)
    const float t21 = GH_FMA(y, z, rx);    const float R21 = GH_ADD(t21, t21);   // 2(yz + rx)
    const float R22 = GH_SUB(1.0f, GH_ADD(xx_yy, xx_yy));
    // M = S * R  ->  M[c][r] = s_r * R[c][r]   (the zero terms of S do not change the rounding)
    const float M00 = GH_MUL(sx, R00), M01 = GH_MUL(sy, R01), M02 = GH_MUL(sz, R02);
    const float M10 = GH_MUL(sx, R10), M11 = GH_MUL(sy, R11), M12 = GH_MUL(sz, R12);
    const float M20 = GH_MUL(sx, R20), M21 = GH_MUL(sy, R21), M22 = GH_MUL(sz, R22);
    // Sigma = transpose(M) * M ; Sigma[j][i] = M[i][0]M[j][0] + M[i][1]M[j][1] + M[i][2]M[j][2]
    cov[0] = GH_FMA(M02, M02, GH_FMA(M00, M00, GH_MUL(M01, M01)));
    cov[1] = GH_FMA(M02, M12, GH_FMA(M00, M10, GH_MUL(M01, M11)));
    cov[2] = GH_FMA(M02, M22, GH_FMA(M00, M20, GH_MUL(M01, M21)));
    cov[3] = GH_FMA(M12, M12, GH_FMA(M10, M10, GH_MUL(M11, M11)));
    cov[4] = GH_FMA(M12, M22, GH_FMA(M10, M20, GH_MUL(M11, M21)));
    cov[5] = GH_FMA(M22, M22, GH_FMA(M20, M20, GH_MUL(M21, M21)));
}

// power = -0.5f*(ca*dx*dx + cc*dy*dy) - cb*dx*dy  in the reference's rounding order
// (forward.cu:358-361 / backward.cu:495-499).
__device__ __forceinline__ float gh_power(float dx, float dy, float ca, float cb, float cc) {
    const float t1 = GH_MUL(dx, ca);
    const float t3 = GH_MUL(dy, GH_MUL(dy, cc));
    const float s = GH_FMA(dx, t1, t3);
    const float t5 = GH_MUL(dy, GH_MUL(dx, cb));
    return GH_FMA(s, -0.5f, -t5);   // SASS: FFMA R, s, -0.5, -t5
}

// ---- per-tile sort network (used by the forward blend CTA for its own list and by gh_segment_sort_kernel)
#define GH_INKERNEL_SORT_MAX 2048u
// Normalised bitonic network (every comparator puts the smaller key at the lower index), so
// elements beyond n behave as +inf without being materialised: a comparator whose upper index
// is >= n is simply skipped.
__device__ __forceinline__ void gh_ce(uint64_t& a, uint64_t& b) {
    const uint64_t lo = a < b ? a : b, hi = a < b ? b : a;
    a = lo; b = hi;
}

template <typename KeyPtr>
__device__ __forceinline__ void gh_bitonic_sort(KeyPtr keys, const uint32_t n, const int tid, const int nt)
{
    const uint64_t INF = ~0ull;             // virtual padding: never stored, never moves
    uint32_t ln2 = 0;                       // n2 = 1 << ln2 >= n
    while ((1u << ln2) < n) ln2++;
    const uint32_t half = (1u << ln2) >> 1, quarter = half >> 1;
    for (uint32_t lk = 1; lk <= ln2; lk++) {      // merge blocks of size k = 1 << lk
        {   // first step of the merge: partner = mirror inside the block of size k
            const uint32_t k = 1u << lk, hk = k >> 1;
            for (uint32_t t = tid; t < half; t += nt) {
                const uint32_t blk = t >> (lk - 1), off = t & (hk - 1);
                const uint32_t i = (blk << lk) + off, j = (blk << lk) + (k - 1 - off);
                if (j < n) {
                    const uint64_t a = keys[i], b = keys[j];
                    if (a > b) { keys[i] = b; keys[j] = a; }
                }
            }
            __syncthreads();
        }
        int ls = (int)lk - 2;                      // remaining strides s = k/4 ... 1
        // two strides (s, s/2) per pass: a thread owns i, i+s/2, i+s, i+3s/2 and does 4 exchanges in registers
        for (; ls >= 1; ls -= 2) {
            const uint32_t sft = (uint32_t)ls, s = 1u << sft, h = s >> 1;
            for (uint32_t t = tid; t < quarter; t += nt) {
                const uint32_t i = ((t >> (sft - 1)) << (sft + 1)) | (t & (h - 1));
                if (i < n) {
                    const uint32_t ib = i + h, ic = i + s, id = ic + h;
                    uint64_t ka = keys[i];
                    uint64_t kb = ib < n ? keys[ib] : INF;
                    uint64_t kc = ic < n ? keys[ic] : INF;
                    uint64_t kd = id < n ? keys[id] : INF;
                    gh_ce(ka, kc); gh_ce(kb, kd);
                    gh_ce(ka, kb); gh_ce(kc, kd);
                    keys[i] = ka;
                    if (ib < n) keys[ib] = kb;
                    if (ic < n) keys[ic] = kc;
                    if (id < n) keys[id] = kd;
                }
            }
            __syncthreads();
        }
        if (ls == 0) {                             // odd number of strides left: the stride-1 stage
            for (uint32_t t = tid; t < half; t += nt) {
                const uint32_t i = t << 1, j = i + 1;
                if (j < n) {
                    const uint64_t a = keys[i], b = keys[j];
                    if (a > b) { keys[i] = b; keys[j] = a; }
                }
            }
            __syncthreads();
        }
    }
}

// Sort up to 2048 records held in shared memory with an NT-thread CTA (NT = 128 or 256) in linear time:
// one MSD split of the records into 1024 sub-buckets by linearly quantised depth (order preserving),
// then every thread insertion-sorts the records of its 1024 / NT consecutive sub-buckets (the range is
// already partitioned, so records move only inside their sub-bucket); ranges longer than 32 records
// fall back to the CTA-wide bitonic network.
#define GH_SORT_SUB 1024u
#define GH_SORT_SCRATCH_WORDS (GH_SORT_SUB + 512u)
template <int NT>
__device__ __forceinline__ void gh_bucket_sort_tile(uint64_t* A, uint64_t* B, uint32_t* cnt, int n, int tid) {
    // cnt: GH_SORT_SCRATCH_WORDS words of 16-byte aligned shared scratch (counters / cursors + list of long ranges)
    constexpr int NW = NT / 32;                    // warps
    constexpr int V4 = (int)GH_SORT_SUB / 4 / NT;  // uint4 of counters per thread (1 or 2)
    __shared__ uint32_t s_red[16];
    __shared__ uint32_t s_nbig;
    const int lane = tid & 31, warp = tid >> 5;
    uint32_t* big = cnt + GH_SORT_SUB;       // (start, length) of thread ranges too long for one thread
    // depth range of the list
    uint32_t dmin = 0xffffffffu, dmax = 0u;
    for (int i = tid; i < n; i += NT) { const uint32_t d = (uint32_t)(A[i] >> 32); dmin = min(dmin, d); dmax = max(dmax, d); }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        dmin = min(dmin, __shfl_xor_sync(0xffffffffu, dmin, o));
        dmax = max(dmax, __shfl_xor_sync(0xffffffffu, dmax, o));
    }
    if (lane == 0) { s_red[warp] = dmin; s_red[8 + warp] = dmax; }
#pragma unroll
    for (int q = 0; q < V4; q++) reinterpret_cast<uint4*>(cnt)[tid * V4 + q] = make_uint4(0u, 0u, 0u, 0u);
    if (tid == 0) s_nbig = 0u;
    __syncthreads();
#pragma unroll
    for (int w = 0; w < NW; w++) { dmin = min(dmin, s_red[w]); dmax = max(dmax, s_red[8 + w]); }
    // monotone map depth bits -> sub-bucket 0..1023
    const float inv = (float)GH_SORT_SUB / ((float)(dmax - dmin) + 1.0f);
    for (int i = tid; i < n; i += NT) {
        const uint32_t d = (uint32_t)(A[i] >> 32);
        const uint32_t b = min(GH_SORT_SUB - 1u, (uint32_t)((float)(d - dmin) * inv));
        atomicAdd(&cnt[b], 1u);
    }
    __syncthreads();
    int r0, r1;      // this thread's range of B: its 4 * V4 consecutive sub-buckets
    {   // exclusive scan of the counts
        uint4 c[V4];
        uint32_t sum = 0;
#pragma unroll
        for (int q = 0; q < V4; q++) { c[q] = reinterpret_cast<uint4*>(cnt)[tid * V4 + q]; sum += c[q].x + c[q].y + c[q].z + c[q].w; }
        uint32_t v = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t nb = __shfl_up_sync(0xffffffffu, v, o); if (lane >= o) v += nb; }
        if (lane == 31) s_red[warp] = v;
        __syncthreads();
        uint32_t start = v - sum;
#pragma unroll
        for (int w = 0; w < NW; w++) start += (w < warp) ? s_red[w] : 0u;
        r0 = (int)start; r1 = (int)(start + sum);
        // the counters become scatter cursors
        uint32_t run = start;
#pragma unroll
        for (int q = 0; q < V4; q++) {
            const uint4 cur = make_uint4(run, run + c[q].x, run + c[q].x + c[q].y, run + c[q].x + c[q].y + c[q].z);
            run += c[q].x + c[q].y + c[q].z + c[q].w;
            reinterpret_cast<uint4*>(cnt)[tid * V4 + q] = cur;
        }
    }
    __syncthreads();
    for (int i = tid; i < n; i += NT) {
        const uint64_t key = A[i];
        const uint32_t d = (uint32_t)(key >> 32);
        const uint32_t b = min(GH_SORT_SUB - 1u, (uint32_t)((float)(d - dmin) * inv));
        B[atomicAdd(&cnt[b], 1u)] = key;
    }
    __syncthreads();
    if (r1 - r0 > 32) {
        const uint32_t q = atomicAdd(&s_nbig, 1u);
        big[2 * q] = (uint32_t)r0; big[2 * q + 1] = (uint32_t)(r1 - r0);
    } else {
        for (int i = r0 + 1; i < r1; i++) {
            const uint64_t key = B[i];
            int j = i - 1;
            while (j >= r0 && B[j] > key) { B[j + 1] = B[j]; j--; }
            B[j + 1] = key;
        }
    }
    __syncthreads();
    const uint32_t nbig = s_nbig;
    for (uint32_t q = 0; q < nbig; q++)
        gh_bitonic_sort(B + big[2 * q], big[2 * q + 1], tid, NT);   // ends with a barrier
    for (int i = tid; i < n; i += NT) A[i] = B[i];
    __syncthreads();
}

#endif  // __CUDACC__
