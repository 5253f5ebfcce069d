// Stage 3 / 4: per-tile front-to-back alpha compositing of the 10-channel feature vector
// (RGB, label, ones, dir2D(3), orientation confidence, depth) and its back-to-front backward.
//
// Per-pixel arithmetic and every skip/stop decision follow the reference kernels renderCUDA
// (cuda_rasterizer/forward.cu:287-400, backward.cu:403-561) bit for bit.  The work decomposition is
// new and built around the shape of strand-aligned Gaussians (long thin ellipses: of the 256 pixels
// of a tile a splat typically reaches alpha >= 1/255 on ~15):
//
//   forward  (gh_blend_forward_kernel, CTA = tile, 8 warps, one pixel per lane)
//   * lists of <= 2048 records are depth-sorted by the CTA itself (gh_bucket_sort_tile) before blending;
//   * the sorted list is staged in chunks of 256 into shared memory with cp.async (LDGSTS), double
//     buffered, indices prefetched two chunks ahead;
//   * each staged Gaussian is scan-converted ONCE per tile: the exact-conservative x-span of
//     {alpha >= 1/255} on every pixel row (two rows per packed-FP32 instruction) gives 16-bit row masks,
//     a 5-step shuffle transpose turns the 32 (Gaussian) x 32 (pixel) bit matrix into one hit list per
//     pixel, and every lane walks only ITS pixel's list -- a skipped Gaussian costs nothing;
//   * the 10 colour channels are accumulated as 5 x (FMUL2 + FFMA2), bit-identical to FMUL + FFMA;
//   * from the same row masks each record's mask over the backward's 64 blocks of 2x2 pixels is written out.
//   backward (gh_blend_backward_kernel, CTA = tile, 4 warps, a vertical pixel pair per lane)
//   * one 384-position window at a time; only the records whose block mask is not zero are staged, and two
//     shuffle transposes of their masks leave one bit list per block;
//   * a block is owned by 2 lanes; the 16 blocks of a warp walk their own lists in lock-step (one warp
//     instruction works on SIXTEEN different Gaussians); blocks are assigned to warps by list length;
//   * the pixel pair is evaluated in packed FP32 (.x upper pixel, .y lower pixel); the 16 gradient
//     components are summed over the block's 2 lanes through shared memory and leave as TWO
//     REDG.E.ADD.F32x4 per lane into a 64-byte per-Gaussian record -- instead of 16 scalar atomicAdd
//     per (pixel, Gaussian) pair in the reference (backward.cu:527,549-558);
//   * dL/dalpha uses the scalar form of the reference's per-channel suffix recursion
//     (backward.cu:519-523):  sum_ch (c - accum_rec)[ch] dL[ch]  =  c.dL  -  A,   A' = a_last (c_last.dL) + (1-a_last) A.
// Both kernels take tiles by decreasing list length (gh_tile_scan_kernel's permutation `tile_perm`).
// DESIGN.md section 5 records the alternatives to these choices that were measured and rejected.
#include "gh_common.cuh"
#include "gh_kernels.h"

#define GH_HALF_C (GH_NUM_CHANNELS / 2)

#define GH_CHUNK 256             // forward staging chunk (records): one per thread, two chunks in flight
#define GH_FWD_MIN_CTAS 4        // __launch_bounds__ second argument of the forward kernel (register cap)
#define GH_BWD_THREADS 128
#define GH_BWD_CHUNK 384         // backward staging window (records)
#define GH_BWD_MIN_CTAS 5        // __launch_bounds__ second argument of the backward kernel (register cap)
#define GH_BWD_BLOCKS 64         // backward 2x2-pixel blocks per tile: 8 across, 8 down, 16 per warp

static_assert(GH_CHUNK == 256, "each of the forward kernel's 256 threads stages exactly one record per chunk");
static_assert(GH_BWD_CHUNK % GH_BWD_THREADS == 0, "every backward thread stages the same number of records of a full window");

namespace {

struct GhPixEval {
    float dx, dy, power, G, alpha;
    bool ok;   // passes the reference's `power > 0` and `alpha < 1/255` skips
};

__device__ __forceinline__ GhPixEval gh_eval(const float4 g0, const float4 g1, float pxf, float pyf) {
    GhPixEval e;
    e.dx = GH_SUB(g0.x, pxf);
    e.dy = GH_SUB(g0.y, pyf);
    e.power = gh_power(e.dx, e.dy, g0.z, g0.w, g1.x);
    e.G = 0.f; e.alpha = 0.f;
    e.ok = false;
    if (!(e.power > 0.0f)) {
        e.G = expf(e.power);
        e.alpha = fminf(0.99f, GH_MUL(g1.y, e.G));
        e.ok = !(e.alpha < 1.0f / 255.0f);
    }
    return e;
}

__device__ __forceinline__ void gh_cp_async16(void* smem, const void* gmem) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void gh_cp_async8(void* smem, const void* gmem) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void gh_cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
__device__ __forceinline__ void gh_cp_async_wait_all() { asm volatile("cp.async.wait_group 0;\n" ::: "memory"); }

// Packed FP32 (Blackwell FFMA2 / FMUL2 / FADD2: two IEEE-rounded results per issue slot).  The blend
// kernels are bound by instruction issue, not by the FP32 pipe, so pairing halves their FP32 cost.
__device__ __forceinline__ float2 gh_f2(float a) { return make_float2(a, a); }
__device__ __forceinline__ float2 gh_neg2(float2 a) { return make_float2(-a.x, -a.y); }
__device__ __forceinline__ float2 gh_mul2(float2 a, float2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ float2 gh_add2(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 gh_sub2(float2 a, float2 b) { return __fadd2_rn(a, gh_neg2(b)); }
__device__ __forceinline__ float2 gh_fma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ float gh_rcp_approx(float x) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

// forward staging, double buffered: chunk c sits in buffer c & 1, chunk c + 1 lands in the other while c is blended
struct GhStage {
    float4 g0[2][GH_CHUNK];
    float4 g1[2][GH_CHUNK];
    float2 feat[2][GH_CHUNK * GH_HALF_C];
    uint32_t id[2][GH_CHUNK];
};
static_assert(sizeof(GhStage::g0) + sizeof(GhStage::g1) >= 8u * GH_INKERNEL_SORT_MAX, "sort buffer A (g0+g1) too small");
static_assert(sizeof(GhStage::feat) >= 8u * GH_INKERNEL_SORT_MAX, "sort buffer B (feat) too small");

// issue the gather of one instance (geometry record + feature row) into slot `slot` of buffer `buf`
__device__ __forceinline__ void gh_stage_issue(GhStage& st, int buf, int slot, uint32_t id,
                                               const GhGeo* __restrict__ geo, const float* __restrict__ features) {
    const float4* gp = reinterpret_cast<const float4*>(geo + id);
    gh_cp_async16(&st.g0[buf][slot], gp);
    gh_cp_async16(&st.g1[buf][slot], gp + 1);
    const float2* fp = reinterpret_cast<const float2*>(features + (size_t)id * GH_NUM_CHANNELS);
#pragma unroll
    for (int k = 0; k < GH_HALF_C; k++) gh_cp_async8(&st.feat[buf][slot * GH_HALF_C + k], fp + k);
    st.id[buf][slot] = id;
}

// Per-PIXEL instance lists of one staged chunk (forward pass).  Warp w scan-converts Gaussians
// [32w, 32w+32) of the chunk (one per lane): on every pixel row the exact-conservative x-span of
// {alpha >= 1/255} becomes a 16-bit column mask; two rows form the
// 32-bit coverage word of the 32 pixels owned by one warp (pixel p = 32*(row/2) + 16*(row%2) + col).
// The 32 (Gaussian) x 32 (pixel) bit matrix is then transposed inside the warp with 5 shuffle steps,
// so lane P ends with "which of my warp's 32 Gaussians cover pixel P" and stores it: no atomics, no
// clearing pass.  pixbits is [word = builder warp][pixel] -> a warp reads consecutive banks.
__device__ __forceinline__ uint32_t gh_transpose32(uint32_t x, int lane) {
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) {
        const uint32_t m = (s == 16) ? 0x0000ffffu : (s == 8) ? 0x00ff00ffu : (s == 4) ? 0x0f0f0f0fu
                         : (s == 2) ? 0x33333333u : 0x55555555u;
        const uint32_t y = __shfl_xor_sync(0xffffffffu, x, s);
        x = (lane & s) ? (((y >> s) & m) | (x & ~m)) : ((x & m) | ((y & m) << s));
    }
    return x;
}

// Two 16-pixel rows (lo, hi halves of `rows`) -> one 8-bit row of 2x2 blocks: bit bx is set when column 2 bx
// or 2 bx + 1 is set in either row.
__device__ __forceinline__ uint32_t gh_block_row(uint32_t rows) {
    uint32_t x = (rows | (rows >> 16)) & 0xffffu;
    x = (x | (x >> 1)) & 0x5555u;
    x = (x | (x >> 1)) & 0x3333u;
    x = (x | (x >> 2)) & 0x0f0fu;
    return (x | (x >> 4)) & 0x00ffu;
}

// Besides the pixel lists, every record of the chunk leaves its mask over the backward's 64 blocks of 2x2
// pixels in bmask[j] (bit by * 8 + bx; .x = block rows 0..3, .y = rows 4..7), derived from the same row
// masks: the backward stages only the records whose mask is not zero and scan-converts nothing itself.
__device__ __forceinline__ void gh_build_pixel_lists(const GhStage& st, uint32_t* pixbits, int buf, int cnt,
                                                     int warp, int lane, float tx0, float ty0,
                                                     uint2* __restrict__ bmask) {
    // `warp` = index of the batch of 32 staged Gaussians this warp scan-converts (= list word index)
    const int j = warp * 32 + lane;
    uint32_t rowmask[16];
#pragma unroll
    for (int r = 0; r < 16; r++) rowmask[r] = 0u;
    float gx = 0.f, gy = 0.f, b = 0.f, ia = 0.f, aQ = -1.f, bbac = 0.f;
    int r0 = 16, r1 = -1;            // rows of the tile this Gaussian can reach
    bool all_pixels = false;
    if (j < cnt) {
        const float4 g0 = st.g0[buf][j], g1 = st.g1[buf][j];
        gx = g0.x; gy = g0.y; b = g0.w;
        const float a = g0.z, c = g1.x, thr = g1.z, pd = g1.w;
        const float mxd = fmaxf(fabsf(gx - tx0), fabsf(gx - (tx0 + 15.f)));
        const float myd = fmaxf(fabsf(gy - ty0), fabsf(gy - (ty0 + 15.f)));
        const float slack = 1e-3f + 2e-5f * (a * mxd * mxd + c * myd * myd + 2.f * fabsf(b) * mxd * myd);
        const float Q = 2.f * (thr + slack);
        if (pd == 0.f || Q != Q) {
            all_pixels = true; r0 = 0; r1 = 15;                     // no bound available: every pixel
        } else if (Q >= 0.f) {
            ia = __frcp_rn(a);
            aQ = a * Q;
            bbac = b * b - a * c;                                   // < 0 for a PD conic
            // rows with a real span: dy^2 < aQ / (ac - b^2)
            const float ry = sqrtf(aQ / (-bbac)) + 0.01f;
            r0 = 0; r1 = 15;
            if (ry == ry) { r0 = max(0, __float2int_ru(gy - ry - ty0)); r1 = min(15, __float2int_rd(gy + ry - ty0)); }
        }
    }
    // warp-uniform row window: the 32 Gaussians of a warp are neighbours in depth, not in space, but
    // strand Gaussians are small, so most rows are empty for the whole warp
    int wr0 = r0, wr1 = r1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        wr0 = min(wr0, __shfl_xor_sync(0xffffffffu, wr0, o));
        wr1 = max(wr1, __shfl_xor_sync(0xffffffffu, wr1, o));
    }
    // two pixel rows per instruction (FFMA2 / FMUL2 / FADD2); a row without a real span has
    // disc <= 0 and is masked out below
    const float2 bbac2 = gh_f2(bbac), aQ2 = gh_f2(aQ), b2 = gh_f2(b), ia2 = gh_f2(ia), gx2 = gh_f2(gx);
    const float2 off2 = gh_f2(-0.01f), ntx2 = gh_f2(-tx0);
#pragma unroll
    for (int t = 0; t < 8; t++) {
        if (2 * t + 1 < wr0 || 2 * t > wr1) continue;               // uniform
        const float2 dy = make_float2(gy - (ty0 + (float)(2 * t)), gy - (ty0 + (float)(2 * t + 1)));
        // a dx^2 + 2 b dy dx + (c dy^2 - Q) <= 0,  dx = gx - px
        const float2 disc = gh_fma2(gh_mul2(dy, dy), bbac2, aQ2);
        const float2 sq = gh_mul2(disc, make_float2(rsqrtf(disc.x), rsqrtf(disc.y)));
        const float2 hb = gh_mul2(b2, dy);
        const float2 lo = gh_add2(gh_add2(gh_fma2(gh_sub2(hb, sq), ia2, gx2), off2), ntx2);
        const float2 hi = gh_add2(gh_add2(gh_fma2(gh_add2(hb, sq), ia2, gx2), gh_neg2(off2)), ntx2);
        const int p0a = max(0, __float2int_ru(lo.x)), p1a = min(15, __float2int_rd(hi.x));
        const int p0b = max(0, __float2int_ru(lo.y)), p1b = min(15, __float2int_rd(hi.y));
        const uint32_t ma = (disc.x > 0.f && p0a <= p1a) ? (((2u << (p1a - p0a)) - 1u) << p0a) : 0u;
        const uint32_t mb = (disc.y > 0.f && p0b <= p1b) ? (((2u << (p1b - p0b)) - 1u) << p0b) : 0u;
        rowmask[2 * t] = all_pixels ? 0xffffu : ma;      // rows outside [r0, r1] have disc <= 0
        rowmask[2 * t + 1] = all_pixels ? 0xffffu : mb;
    }
    uint2 bm = make_uint2(0u, 0u);
#pragma unroll
    for (int t = 0; t < 8; t++) {
        const uint32_t word = rowmask[2 * t] | (rowmask[2 * t + 1] << 16);   // my coverage of warp t's pixels
        if (t < 4) bm.x |= gh_block_row(word) << (8 * t);
        else bm.y |= gh_block_row(word) << (8 * (t - 4));
        uint32_t col = 0u;
        if (__any_sync(0xffffffffu, word != 0u)) col = gh_transpose32(word, lane);
        pixbits[warp * 256 + t * 32 + lane] = col;                           // pixel 32t+lane: bits = Gaussians
    }
    if (j < cnt) bmask[j] = bm;
}

// ------------------------------------------------------------------------------------------ forward
__global__ void __launch_bounds__(256, GH_FWD_MIN_CTAS)
gh_blend_forward_kernel(const uint2* __restrict__ ranges, const uint32_t* __restrict__ tile_perm, uint64_t* inst,
                        const GhGeo* __restrict__ geo, const float* __restrict__ features,
                        int W, int H, int gx, const float* __restrict__ bg,
                        float* __restrict__ final_T, uint32_t* __restrict__ n_contrib,
                        float* __restrict__ out, uint2* __restrict__ bmask)
{
    // Forward needs no cross-pixel communication, so every lane walks the list of ITS OWN pixel:
    // a lane only ever touches Gaussians whose alpha >= 1/255 footprint (conservatively) contains
    // its pixel, whatever the other lanes of the warp are doing.
    extern __shared__ __align__(16) unsigned char gh_fwd_smem[];
    GhStage& st = *reinterpret_cast<GhStage*>(gh_fwd_smem);
    uint32_t* pixbits = reinterpret_cast<uint32_t*>(gh_fwd_smem + sizeof(GhStage));   // [word][pixel] (GH_CHUNK / 32 words x 256); also the sort's scratch

    const int tile = (int)tile_perm[blockIdx.x];      // heaviest tiles first
    const int tx = tile % gx, ty = tile / gx;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // a warp owns two pixel rows: lanes 0..15 row 2*warp, lanes 16..31 row 2*warp+1
    const int px = tx * GH_BLOCK_X + (lane & 15);
    const int py = ty * GH_BLOCK_Y + 2 * warp + (lane >> 4);
    const bool inside = (px < W) && (py < H);
    const float pxf = (float)px, pyf = (float)py;
    const float tx0 = (float)(tx * GH_BLOCK_X), ty0 = (float)(ty * GH_BLOCK_Y);

    const uint2 rg = ranges[tile];
    const int n = (int)(rg.y - rg.x);
    const int nchunks = (n + GH_CHUNK - 1) / GH_CHUNK;

    float T = 1.0f;
    float2 C2[GH_HALF_C];                      // channel pairs (2k, 2k+1)
#pragma unroll
    for (int k = 0; k < GH_HALF_C; k++) C2[k] = make_float2(0.f, 0.f);
    uint32_t last = 0;
    bool done = !inside;
    bool warp_done = (__ballot_sync(0xffffffffu, done) == 0xffffffffu);

    // Sort this tile's bucket by (depth bits, Gaussian index) right here when it fits the staging buffers
    // (<= 2048 records = 16 KB): the sort is latency/barrier bound, the blend is issue bound, and as
    // one kernel the two overlap across the CTAs of an SM.  The sorted bucket is written back for the
    // backward pass.  Longer lists were sorted by gh_tile_split_long_kernel + gh_segment_sort_kernel
    // (gh_binning.cu) before this launch.
    if (n >= 2 && n <= (int)GH_INKERNEL_SORT_MAX) {
        uint64_t* sbase = reinterpret_cast<uint64_t*>(&st.g0[0][0]);     // g0 + g1 = 16 KB contiguous
        uint64_t* spong = reinterpret_cast<uint64_t*>(&st.feat[0][0]);   // next 16 KB (feat is 20 KB)
        uint64_t* gl = inst + rg.x;
        // The bucket is one contiguous run of 8-byte records: the TMA engine copies it into shared memory
        // (cp.async.bulk, one request, completion on an mbarrier) instead of a load/store loop.  Bulk copies
        // move 16-byte granules, so the run is widened to even record indices; `skeys` skips the extra
        // leading record.  The rare run that would not fit after widening takes the loop.
        const uint32_t odd = rg.x & 1u;
        const uint32_t nrec = ((uint32_t)n + odd + 1u) & ~1u;
        uint64_t* skeys = sbase;                  // the loop path below uses the whole 2048-record buffer
        if (nrec <= GH_INKERNEL_SORT_MAX) {
            skeys = sbase + odd;
            __shared__ __align__(8) uint64_t s_mbar;
            const uint32_t mbar = (uint32_t)__cvta_generic_to_shared(&s_mbar);
            if (tid == 0) {
                asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(mbar) : "memory");
                asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            }
            __syncthreads();
            if (tid == 0) {
                const uint32_t bytes = nrec * 8u;
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                             ::"r"((uint32_t)__cvta_generic_to_shared(sbase)), "l"(gl - odd), "r"(bytes), "r"(mbar) : "memory");
            }
            uint32_t landed = 0;
            for (uint32_t it = 0; it < (1u << 24) && !landed; it++)
                asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n selp.u32 %0, 1, 0, p;\n}"
                             : "=r"(landed) : "r"(mbar) : "memory");
            if (!landed) __trap();            // the copy engine never reported completion
        } else {
            for (int i = tid; i < n; i += 256) skeys[i] = gl[i];
            __syncthreads();
        }
        if (n <= 64) gh_bitonic_sort(skeys, (uint32_t)n, tid, 256);
        else gh_bucket_sort_tile<256>(skeys, spong, pixbits, n, tid);
        for (int i = tid; i < n; i += 256) gl[i] = skeys[i];
        __syncthreads();
    }

    // prologue: chunk 0 in flight, indices of chunk 1 in a register
    uint32_t next_id = 0;
    if (nchunks > 0) {
        if (tid < min(GH_CHUNK, n)) gh_stage_issue(st, 0, tid, (uint32_t)inst[(size_t)rg.x + tid], geo, features);
        gh_cp_async_commit();
        if (GH_CHUNK + tid < n) next_id = (uint32_t)inst[(size_t)rg.x + GH_CHUNK + tid];
    }

    for (int c = 0; c < nchunks; c++) {
        const int base = c * GH_CHUNK;
        const int cnt = min(GH_CHUNK, n - base);
        const int buf = c & 1;
        gh_cp_async_wait_all();
        // chunk c landed for every thread; block-wide early exit like the reference's
        // __syncthreads_count(done) == BLOCK_SIZE
        if (__syncthreads_and(warp_done)) break;
        if (c + 1 < nchunks) {
            if (base + GH_CHUNK + tid < n) gh_stage_issue(st, buf ^ 1, tid, next_id, geo, features);
            gh_cp_async_commit();
            if (base + 2 * GH_CHUNK + tid < n) next_id = (uint32_t)inst[(size_t)rg.x + base + 2 * GH_CHUNK + tid];
        }
        gh_build_pixel_lists(st, pixbits, buf, cnt, warp, lane, tx0, ty0, bmask + rg.x + base);
        __syncthreads();

        if (!done) {
            // which of my pixel's 8 list words are non-empty
            uint32_t nz = 0u;
#pragma unroll
            for (int k = 0; k < GH_CHUNK / 32; k++)
                nz |= (pixbits[k * 256 + tid] != 0u) ? (1u << k) : 0u;
            int wi = 0;
            uint32_t cur = 0u;
            while (true) {
                if (cur == 0u) {
                    if (nz == 0u) break;
                    wi = __ffs(nz) - 1;
                    nz &= nz - 1;
                    cur = pixbits[wi * 256 + tid];
                }
                const int bpos = __ffs(cur) - 1;
                cur &= cur - 1;
                const int jj = wi * 32 + bpos;
                const float4 g0 = st.g0[buf][jj], g1 = st.g1[buf][jj];
                const GhPixEval e = gh_eval(g0, g1, pxf, pyf);
                if (e.ok) {
                    const float test_T = GH_MUL(T, GH_SUB(1.0f, e.alpha));
                    if (test_T < 0.0001f) { done = true; break; }
                    // C[ch] = fma(T, alpha * f[ch], C[ch]) (forward.cu:379-380 as ptxas fuses it), two
                    // channels per instruction with Blackwell's packed FP32 pipe: FMUL2 + FFMA2 round each
                    // half exactly like FMUL + FFMA
                    const float2 a2 = make_float2(e.alpha, e.alpha), T2 = make_float2(T, T);
#pragma unroll
                    for (int k = 0; k < GH_HALF_C; k++)
                        C2[k] = __ffma2_rn(T2, __fmul2_rn(a2, st.feat[buf][jj * GH_HALF_C + k]), C2[k]);
                    T = test_T;
                    last = (uint32_t)(base + jj + 1);
                }
            }
        }
        warp_done = (__ballot_sync(0xffffffffu, done) == 0xffffffffu);
    }
    gh_cp_async_wait_all();

    if (inside) {
        const size_t pix = (size_t)py * W + px;
        final_T[pix] = T;
        n_contrib[pix] = last;
        const size_t plane = (size_t)H * W;
#pragma unroll
        for (int ch = 0; ch < GH_NUM_CHANNELS; ch++)
            out[ch * plane + pix] = GH_FMA(T, __ldg(bg + ch), (ch & 1) ? C2[ch >> 1].y : C2[ch >> 1].x);
    }
}

// ------------------------------------------------------------------------------------------ backward
// Backward staging: ONE window of GH_BWD_CHUNK list positions at a time (single-buffered; the other resident
// CTAs of the SM cover the gather latency).  Only the LIVE records of the window are staged -- those whose
// block mask from the forward (gh_build_pixel_lists) is not zero -- packed into the first slots in list
// order.  The 16 blocks of a warp walk their lists in lock-step, so a warp spends max(list length over its
// blocks) steps per window: a wide window wastes fewer lanes on that maximum than several narrow ones
// (tools/imbalance.py), and 384 records still leave room for 5 CTAs per SM.
struct GhStageB {
    float4 g0[GH_BWD_CHUNK];                 // [slot]
    float4 g1[GH_BWD_CHUNK];
    float2 feat[GH_BWD_CHUNK * GH_HALF_C];
    uint2 ref[GH_BWD_CHUNK];                 // [slot] (Gaussian id, list position)
    uint2 mask[GH_BWD_CHUNK];                // [position - window base] block mask written by the forward
    uint32_t bits[GH_BWD_BLOCKS][GH_BWD_CHUNK / 32 + 1];   // [block][word]; +1 pad against bank conflicts
};

__device__ __forceinline__ void gh_stage_issue_b(GhStageB& st, int slot, uint32_t id, uint32_t pos,
                                                 const GhGeo* __restrict__ geo, const float* __restrict__ features) {
    const float4* gp = reinterpret_cast<const float4*>(geo + id);
    gh_cp_async16(&st.g0[slot], gp);
    gh_cp_async16(&st.g1[slot], gp + 1);
    const float2* fp = reinterpret_cast<const float2*>(features + (size_t)id * GH_NUM_CHANNELS);
#pragma unroll
    for (int k = 0; k < GH_HALF_C; k++) gh_cp_async8(&st.feat[slot * GH_HALF_C + k], fp + k);
    st.ref[slot] = make_uint2(id, pos);
}

// Live records of a window: ball[i] = which of the positions base + 32 i + [0, 32) are live.  Returns how many
// live records lie before window position p (0 <= p <= GH_BWD_CHUNK) = the slot of position p when it is live.
#define GH_BWD_BATCHES (GH_BWD_CHUNK / 32)
__device__ __forceinline__ uint32_t gh_live_before(const uint32_t (&ball)[GH_BWD_BATCHES], int p) {
    const int bi = p >> 5;
    const uint32_t part = (1u << (p & 31)) - 1u;
    uint32_t c = 0;
#pragma unroll
    for (int i = 0; i < GH_BWD_BATCHES; i++)
        c += __popc(i < bi ? ball[i] : (i == bi ? (ball[i] & part) : 0u));
    return c;
}

// batch `word` = slots [32 word, 32 word + 32) of the window, one per lane; two 5-step shuffle transposes turn
// the 32 block masks into one list word per block (lane = block `lane` and block 32 + lane).  The word is cut at
// the block's deepest blended list position here, once, rather than in the traversal loop: cut_lo / cut_hi =
// the number of staged slots whose position lies before that of block `lane` / of block 32 + lane (positions
// increase with the slot, so the cut is a prefix of the window).
__device__ __forceinline__ uint32_t gh_valid_bits(uint32_t cut, int first_slot) {
    const int lim = (int)cut - first_slot;
    return lim >= 32 ? 0xffffffffu : (lim <= 0 ? 0u : ((1u << lim) - 1u));
}

__device__ __forceinline__ void gh_build_lists_b(GhStageB& st, int nlive, int word, int lane, int base,
                                                 uint32_t cut_lo, uint32_t cut_hi) {
    const int j = word * 32 + lane;
    uint2 m = make_uint2(0u, 0u);
    if (j < nlive) m = st.mask[st.ref[j].y - (uint32_t)base];
    uint32_t lo = 0, hi = 0;
    if (__any_sync(0xffffffffu, m.x != 0u)) lo = gh_transpose32(m.x, lane);
    if (__any_sync(0xffffffffu, m.y != 0u)) hi = gh_transpose32(m.y, lane);
    st.bits[lane][word] = lo & gh_valid_bits(cut_lo, word * 32);
    st.bits[32 + lane][word] = hi & gh_valid_bits(cut_hi, word * 32);
}

// The even lane keeps components 0..7, the odd lane 8..15 (two REDG.E.ADD.F32x4 each).  Each lane
// stores the half its partner keeps (2 STS.128), loads the partner's contribution to its own half (2 LDS.128) and
// adds (4 FADD2): 4 shared-memory instructions where a shuffle exchange of 8 floats takes 8 SHFL (the kernel is
// bound by issue slots).  Record stride 48 B: the 8 lanes of a quarter-warp hit 8 disjoint groups of 4 banks.
#define GH_RED2_STRIDE4 3
__device__ __forceinline__ void gh_group2_reduce16(const float (&v)[16], float4* warp_buf, int lane, float4& out0, float4& out1) {
    const bool odd = (lane & 1) != 0;
    float4* mine = warp_buf + lane * GH_RED2_STRIDE4;
    // what the partner keeps: the even lane's partner (odd) keeps 8..15, the odd lane's partner keeps 0..7
    mine[0] = odd ? make_float4(v[0], v[1], v[2], v[3]) : make_float4(v[8], v[9], v[10], v[11]);
    mine[1] = odd ? make_float4(v[4], v[5], v[6], v[7]) : make_float4(v[12], v[13], v[14], v[15]);
    __syncwarp();
    const float4* theirs = warp_buf + (lane ^ 1) * GH_RED2_STRIDE4;
    const float4 a = theirs[0], b = theirs[1];
    __syncwarp();              // the next step overwrites the records
    const float4 k0 = odd ? make_float4(v[8], v[9], v[10], v[11]) : make_float4(v[0], v[1], v[2], v[3]);
    const float4 k1 = odd ? make_float4(v[12], v[13], v[14], v[15]) : make_float4(v[4], v[5], v[6], v[7]);
    const float2 s0 = gh_add2(make_float2(k0.x, k0.y), make_float2(a.x, a.y)), s1 = gh_add2(make_float2(k0.z, k0.w), make_float2(a.z, a.w));
    const float2 s2 = gh_add2(make_float2(k1.x, k1.y), make_float2(b.x, b.y)), s3 = gh_add2(make_float2(k1.z, k1.w), make_float2(b.z, b.w));
    out0 = make_float4(s0.x, s0.y, s1.x, s1.y);
    out1 = make_float4(s2.x, s2.y, s3.x, s3.y);
}

// State of the lane's pixel pair; .x = pixel (x, y0), .y = pixel (x, y0 + 1).
struct GhBwdPair {
    float2 T, A, last_alpha, last_cdot;
    float2 ntf_bg;                 // -T_final * (bg . dL_dpix)
    float2 npy;                    // -(pixel y)
    uint32_t last0, last1;
    float2 dL0[GH_HALF_C], dL1[GH_HALF_C];   // dL/dpixel of pixel 0 / pixel 1, channel pairs (2k, 2k+1)
};

// The pixel pair's share of one Gaussian, branch-free: every lane runs the same instruction stream and
// a pixel that does not blend this Gaussian (behind its last contributor, power > 0, alpha < 1/255 --
// the reference's three `continue`s, backward.cu:490-505) has alpha = G = 0, contributes exact zeros
// and keeps its state.  power / alpha are bit-identical to the forward pass (same operation order,
// FMUL2/FFMA2 round like FMUL/FFMA), so both passes agree on which pixels blend.  v = the 16 gradient
// components summed over the two pixels.
__device__ __forceinline__ bool gh_bwd_pair(GhBwdPair& p, const float4 g0, const float4 g1, const float2* feat,
                                            float pxf, uint32_t pos, float ddelx_dx, float ddely_dy, float (&v)[16]) {
    const float dx = GH_SUB(g0.x, pxf);
    const float2 dx2 = gh_f2(dx);
    const float2 dy = gh_add2(gh_f2(g0.y), p.npy);
    // gh_power: fma(fma(dx, dx*ca, dy*(dy*cc)), -0.5, -(dy*(dx*cb)))
    const float t1 = GH_MUL(dx, g0.z), dxcb = GH_MUL(dx, g0.w);
    const float2 t3 = gh_mul2(dy, gh_mul2(dy, gh_f2(g1.x)));
    const float2 sq = gh_fma2(dx2, gh_f2(t1), t3);
    const float2 power = gh_fma2(sq, gh_f2(-0.5f), gh_mul2(dy, gh_f2(-dxcb)));
    const float Gx0 = expf((power.x > 0.0f) ? 0.0f : power.x);   // expf(power) whenever the reference evaluates it
    const float Gx1 = expf((power.y > 0.0f) ? 0.0f : power.y);
    const float2 ao = gh_mul2(gh_f2(g1.y), make_float2(Gx0, Gx1));
    const float alpha0 = fminf(0.99f, ao.x), alpha1 = fminf(0.99f, ao.y);
    const bool ok0 = (pos < p.last0) & !(power.x > 0.0f) & !(alpha0 < 1.0f / 255.0f);
    const bool ok1 = (pos < p.last1) & !(power.y > 0.0f) & !(alpha1 < 1.0f / 255.0f);
    const float2 am = make_float2(ok0 ? alpha0 : 0.f, ok1 ? alpha1 : 0.f);
    const float2 G = make_float2(ok0 ? Gx0 : 0.f, ok1 ? Gx1 : 0.f);
    // T_{before this Gaussian} = T / (1 - alpha); gradients only need ~1 ulp here: MUFU.RCP, 1 - alpha
    // is in [0.01, 1] and rcp(1) == 1 exactly
    const float2 om = gh_sub2(gh_f2(1.0f), am);
    const float2 r = make_float2(gh_rcp_approx(om.x), gh_rcp_approx(om.y));
    p.T = gh_mul2(p.T, r);
    const float2 w = gh_mul2(am, p.T);                          // d(out)/d(color)
    const float2 w0 = gh_f2(w.x), w1 = gh_f2(w.y);
    float2 c0, c1;
#pragma unroll
    for (int k = 0; k < GH_HALF_C; k++) {
        const float2 f = feat[k];
        c0 = (k == 0) ? gh_mul2(f, p.dL0[0]) : gh_fma2(f, p.dL0[k], c0);
        c1 = (k == 0) ? gh_mul2(f, p.dL1[0]) : gh_fma2(f, p.dL1[k], c1);
        const float2 vc = gh_fma2(w1, p.dL1[k], gh_mul2(w0, p.dL0[k]));
        v[2 * k] = vc.x; v[2 * k + 1] = vc.y;
    }
    const float2 cdot = make_float2(c0.x + c0.y, c1.x + c1.y);
    // suffix recursion on the dot product (backward.cu:519-523), state advances only when blended
    const float2 A_new = gh_fma2(p.last_alpha, p.last_cdot, gh_mul2(gh_sub2(gh_f2(1.0f), p.last_alpha), p.A));
    // alpha also scales how much background shows through (backward.cu:535-538).  Not masked: every use
    // below is multiplied by G, which is 0 for a pixel that does not blend.
    const float2 dL_dalpha = gh_fma2(gh_sub2(cdot, A_new), p.T, gh_mul2(p.ntf_bg, r));
    // State update WITHOUT selects: a pixel that does not blend stores last_alpha = 0, so the next step computes
    // A_new = fma(0, last_cdot, 1 * A) = A exactly (cdot is finite) -- the recursion skips it just as the
    // reference's `continue` does, and A_new of this step is what the next blended step would have computed.
    p.A = A_new;
    p.last_cdot = cdot;
    p.last_alpha = am;
    const float2 dL_dG = gh_mul2(gh_f2(g1.y), dL_dalpha);
    const float2 gdx = gh_mul2(G, dx2), gdy = gh_mul2(G, dy);
    const float2 ncb = gh_f2(-g0.w);
    const float2 dG_ddelx = gh_fma2(gdx, gh_f2(-g0.z), gh_mul2(gdy, ncb));
    const float2 dG_ddely = gh_fma2(gdy, gh_f2(-g1.x), gh_mul2(gdx, ncb));
    const float2 t10 = gh_mul2(dL_dG, dG_ddelx), t11 = gh_mul2(dL_dG, dG_ddely);
    const float2 hg = gh_mul2(gh_f2(-0.5f), dL_dG);
    const float2 hgdx = gh_mul2(hg, gdx);
    const float2 t12 = gh_mul2(hgdx, dx2), t13 = gh_mul2(hgdx, dy), t14 = gh_mul2(gh_mul2(hg, gdy), dy);
    const float2 t15 = gh_mul2(G, dL_dalpha);
    v[10] = (t10.x + t10.y) * ddelx_dx; v[11] = (t11.x + t11.y) * ddely_dy;
    v[12] = t12.x + t12.y; v[13] = t13.x + t13.y; v[14] = t14.x + t14.y; v[15] = t15.x + t15.y;
    return ok0 | ok1;
}

// CTA = tile = 4 warps.  A lane owns a vertical pixel pair (x, y0), (x, y0+1); lanes 2i and 2i+1 own a 2x2
// block; block b covers tile pixels x = 2 (b % 8) + {0, 1}, y = 2 (b / 8) + {0, 1}.  The 16 blocks of a warp
// walk their own lists in lock-step, i.e. every warp instruction works on SIXTEEN different Gaussians.  The
// two pixels of a lane are summed in registers; the 16 gradient components are then summed over the block's
// 2 lanes through shared memory (gh_group2_reduce16), leaving eight adjacent components per lane = two
// REDG.E.ADD.F32x4 per lane.
__global__ void __launch_bounds__(GH_BWD_THREADS, GH_BWD_MIN_CTAS)
gh_blend_backward_kernel(const uint2* __restrict__ ranges, const uint32_t* __restrict__ tile_perm, const uint64_t* __restrict__ inst,
                         const GhGeo* __restrict__ geo, const float* __restrict__ features,
                         int W, int H, int gx, const float* __restrict__ bg,
                         const float* __restrict__ final_T, const uint32_t* __restrict__ n_contrib,
                         const float* __restrict__ dL_dpix, const uint2* __restrict__ bmask,
                         float* __restrict__ acc16)   // [P][16]: colors 0..9, mean2D x,y, conic x,y,w, opacity
{
    extern __shared__ __align__(16) unsigned char gh_bwd_smem[];
    GhStageB& st = *reinterpret_cast<GhStageB*>(gh_bwd_smem);
    float4* red_buf = reinterpret_cast<float4*>(gh_bwd_smem + sizeof(GhStageB)) + (threadIdx.x >> 5) * 32 * GH_RED2_STRIDE4;
    __shared__ uint32_t s_warp_last[GH_BWD_THREADS / 32];
    __shared__ uint32_t s_glast[GH_BWD_BLOCKS];              // per block: deepest list position any of its pixels blended
    __shared__ uint8_t s_perm[GH_BWD_THREADS / 32][GH_BWD_BLOCKS];   // per warp (redundant copies): rank -> block
    __shared__ uint32_t s_ball[GH_BWD_BATCHES];              // live records of the window being staged (gh_live_before)

    const int tile = (int)tile_perm[blockIdx.x];      // heaviest tiles first
    const int tx = tile % gx, ty = tile / gx;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const size_t plane = (size_t)H * W;
    const uint2 rg = ranges[tile];

    // ---- how far do the blocks / the tile reach into the list?  (natural block order here: warp w owns
    // blocks 16 w .. 16 w + 15)
    {
        const int nb = 16 * warp + lane / 2;
        const int nx = tx * GH_BLOCK_X + 2 * (nb % 8) + (lane % 2);
        const int ny = ty * GH_BLOCK_Y + 2 * (nb / 8);
        uint32_t gl = 0;
        if (nx < W && ny < H) gl = n_contrib[(size_t)ny * W + nx];
        if (nx < W && ny + 1 < H) gl = max(gl, n_contrib[(size_t)(ny + 1) * W + nx]);
        gl = max(gl, __shfl_xor_sync(0xffffffffu, gl, 1));      // over the block's two lanes
        if ((lane % 2) == 0) s_glast[nb] = gl;
        uint32_t wl = gl;
#pragma unroll
        for (int o = 2; o < 32; o <<= 1) wl = max(wl, __shfl_xor_sync(0xffffffffu, wl, o));
        if (lane == 0) s_warp_last[warp] = wl;
    }
    __syncthreads();
    uint32_t tile_last = 0;
#pragma unroll
    for (int w = 0; w < GH_BWD_THREADS / 32; w++) tile_last = max(tile_last, s_warp_last[w]);
    const int n = (int)tile_last;             // nothing beyond is blended by any pixel of this tile
    const int nchunks = (n + GH_BWD_CHUNK - 1) / GH_BWD_CHUNK;
    if (nchunks == 0) return;
    constexpr int PER_THREAD = GH_BWD_CHUNK / GH_BWD_THREADS;
    constexpr int WARPS = GH_BWD_THREADS / 32;
    // the builder's lane == block after the transposes: blocks `lane` and `32 + lane`
    const uint32_t glast_lo = s_glast[lane];
    const uint32_t glast_hi = s_glast[32 + lane];
    const uint32_t* ids = reinterpret_cast<const uint32_t*>(inst + rg.x);   // low word of a record = Gaussian id
    const uint2* masks = bmask + rg.x;

    // Thread tid covers window positions base + tid + 128 h (batch h * 4 + warp of s_ball).  The ids of the next
    // window wait in registers; its masks (st.mask) and live ballots (s_ball) are published as soon as the
    // current window's lists are built.
    uint32_t next_id[PER_THREAD];
    uint2 next_m[PER_THREAD];
    auto fetch = [&](int base, int cnt) {
#pragma unroll
        for (int h = 0; h < PER_THREAD; h++) {
            const int p = tid + h * GH_BWD_THREADS;
            next_id[h] = 0u;
            next_m[h] = make_uint2(0u, 0u);
            if (p < cnt) { next_id[h] = ids[2 * (size_t)(base + p)]; next_m[h] = masks[base + p]; }
        }
    };
    auto publish = [&]() {
#pragma unroll
        for (int h = 0; h < PER_THREAD; h++) {
            st.mask[tid + h * GH_BWD_THREADS] = next_m[h];
            const uint32_t b = __ballot_sync(0xffffffffu, (next_m[h].x | next_m[h].y) != 0u);
            if (lane == 0) s_ball[h * WARPS + warp] = b;
        }
    };
    // After a __syncthreads that follows publish(): stage the live records of window [base, base + GH_BWD_CHUNK)
    // and build its per-block lists.  Returns the number of live records = staged slots.
    auto stage = [&](int base, bool prefetch) -> int {
        uint32_t ball[GH_BWD_BATCHES];
#pragma unroll
        for (int i = 0; i < GH_BWD_BATCHES; i++) ball[i] = s_ball[i];
#pragma unroll
        for (int h = 0; h < PER_THREAD; h++) {
            const int p = tid + h * GH_BWD_THREADS;
            if ((s_ball[h * WARPS + warp] >> lane) & 1u)
                gh_stage_issue_b(st, (int)gh_live_before(ball, p), next_id[h], (uint32_t)(base + p), geo, features);
        }
        gh_cp_async_commit();
        const int nlive = (int)gh_live_before(ball, GH_BWD_CHUNK);
        const uint32_t b0 = (uint32_t)base;
        const uint32_t cut_lo = gh_live_before(ball, (int)min(max(glast_lo, b0) - b0, (uint32_t)GH_BWD_CHUNK));
        const uint32_t cut_hi = gh_live_before(ball, (int)min(max(glast_hi, b0) - b0, (uint32_t)GH_BWD_CHUNK));
        if (prefetch) fetch(base - GH_BWD_CHUNK, GH_BWD_CHUNK);
        gh_cp_async_wait_all();
        __syncthreads();
        // per-block lists: each of the 4 warps transposes every fourth batch of 32 staged records
        for (int word = warp; word * 32 < nlive; word += WARPS)
            gh_build_lists_b(st, nlive, word, lane, base, cut_lo, cut_hi);
        __syncthreads();
        if (prefetch) publish();        // st.mask and s_ball are free again
        return nlive;
    };

    // ---- stage the last window (windows are visited last to first) and build its lists
    {
        const int base = (nchunks - 1) * GH_BWD_CHUNK;
        fetch(base, n - base);
        publish();
        __syncthreads();
    }
    int nlive = stage((nchunks - 1) * GH_BWD_CHUNK, nchunks > 1);

    // ---- block -> (warp, lane group) assignment.  The blocks of a warp advance in lock-step, so a warp pays for
    // its LONGEST list: blocks are ranked by the length of their list in the window just built (lane b counts block
    // b -- and block 32 + b; every warp computes the same ranking for itself) and each warp takes 16
    // neighbours of that ranking.  Any assignment gives the same gradients up to the order of the float atomics.
    int blk;
    {
        const int nw = (nlive + 31) >> 5;
        uint32_t len0 = 0, len1 = 0;
        for (int w = 0; w < nw; w++) {
            len0 += __popc(st.bits[lane][w]);
            len1 += __popc(st.bits[32 + lane][w]);
        }
        const uint32_t key0 = (len0 << 6) | (uint32_t)lane, key1 = (len1 << 6) | (uint32_t)(32 + lane);
        int rank0 = 0, rank1 = 0;
#pragma unroll
        for (int k = 0; k < 32; k++) {
            const uint32_t a = __shfl_sync(0xffffffffu, key0, k);
            const uint32_t b = __shfl_sync(0xffffffffu, key1, k);
            rank0 += ((a < key0) ? 1 : 0) + ((b < key0) ? 1 : 0);
            rank1 += ((a < key1) ? 1 : 0) + ((b < key1) ? 1 : 0);
        }
        s_perm[warp][rank0] = (uint8_t)lane;
        s_perm[warp][rank1] = (uint8_t)(32 + lane);
        __syncwarp();
        blk = s_perm[warp][16 * warp + lane / 2];
    }
    const int px = tx * GH_BLOCK_X + 2 * (blk % 8) + (lane % 2);
    const int py0 = ty * GH_BLOCK_Y + 2 * (blk / 8);
    const float pxf = (float)px;

    GhBwdPair pr;
    {
        float tf[2], bgd[2];
        uint32_t lastv[2];
#pragma unroll
        for (int r = 0; r < 2; r++) {
            const int py = py0 + r;
            const bool inside = (px < W) && (py < H);
            const size_t pi = (size_t)py * W + px;
            tf[r] = inside ? final_T[pi] : 0.f;
            lastv[r] = inside ? n_contrib[pi] : 0u;     // pixel blends list positions 1..last
            float d[GH_NUM_CHANNELS];
            bgd[r] = 0.f;
#pragma unroll
            for (int ch = 0; ch < GH_NUM_CHANNELS; ch++) {
                d[ch] = inside ? dL_dpix[ch * plane + pi] : 0.f;
                bgd[r] += __ldg(bg + ch) * d[ch];
            }
#pragma unroll
            for (int k = 0; k < GH_HALF_C; k++) {
                if (r == 0) pr.dL0[k] = make_float2(d[2 * k], d[2 * k + 1]);
                else pr.dL1[k] = make_float2(d[2 * k], d[2 * k + 1]);
            }
        }
        pr.T = make_float2(tf[0], tf[1]);
        pr.ntf_bg = make_float2(-tf[0] * bgd[0], -tf[1] * bgd[1]);
        pr.npy = make_float2(-(float)py0, -(float)(py0 + 1));
        pr.A = gh_f2(0.f); pr.last_alpha = gh_f2(0.f); pr.last_cdot = gh_f2(0.f);
        pr.last0 = lastv[0]; pr.last1 = lastv[1];
    }
    // pixel-coordinate -> NDC chain rule factors (backward.cu:464-465)
    const float ddelx_dx = 0.5f * W, ddely_dy = 0.5f * H;

    uint32_t wlast = s_glast[blk];
#pragma unroll
    for (int o = 2; o < 32; o <<= 1) wlast = max(wlast, __shfl_xor_sync(0xffffffffu, wlast, o));   // over the warp's blocks

    for (int c = nchunks - 1; c >= 0; c--) {
        const int base = c * GH_BWD_CHUNK;
        if (c != nchunks - 1) {
            __syncthreads();                       // everyone is done with the previous window
            nlive = stage(base, c > 0);
        }
        if ((uint32_t)base >= wlast) continue;

        int wi = (nlive + 31) >> 5;
        uint32_t cur = 0;
        while (true) {
            while (cur == 0 && wi > 0) cur = st.bits[blk][--wi];
            const bool act = (cur != 0);
            if (!__any_sync(0xffffffffu, act)) break;

            // blocks whose list is exhausted run the same code on slot 0 with pos = UINT_MAX (-> all zeros)
            const int bpos = act ? 31 - __clz(cur) : 0;   // back to front
            cur &= ~(1u << bpos);
            const int jj = act ? wi * 32 + bpos : 0;
            const uint2 rf = st.ref[jj];
            const uint32_t id = rf.x;
            const float4 g0 = st.g0[jj], g1 = st.g1[jj];
            const float2* feat = &st.feat[jj * GH_HALF_C];
            const uint32_t pos = act ? rf.y : 0xffffffffu;
            float v[16];
            const bool contrib = gh_bwd_pair(pr, g0, g1, feat, pxf, pos, ddelx_dx, ddely_dy, v);
            const uint32_t cm = __ballot_sync(0xffffffffu, contrib);
            if (cm == 0u) continue;
            float4 s0, s1;
            gh_group2_reduce16(v, red_buf, lane, s0, s1);
            if ((cm >> (lane & 30)) & 3u) {            // either lane of my block contributed
                float4* dst = reinterpret_cast<float4*>(acc16 + (size_t)id * 16) + 2 * (lane & 1);
                atomicAdd(dst, s0);       // REDG.E.ADD.F32x4: components 0..3 / 8..11
                atomicAdd(dst + 1, s1);   //                              4..7 / 12..15
            }
        }
    }
    gh_cp_async_wait_all();
}

// ---------------------------------------------------------------------------- gradient unpack
// acc16 -> the reference binding's layouts (rasterize_points.cu:160-168): dL_dcolor (P,10),
// dL_dmean2D (P,3) [z never written by the reference: 0], dL_dconic (P,2,2) [.z unused: 0], dL_dopacity (P,1)
__global__ void __launch_bounds__(256)
gh_unpack_grads_kernel(int P, const float* __restrict__ acc16, float* __restrict__ dL_dmean2D,
                       float* __restrict__ dL_dconic, float* __restrict__ dL_dopacity, float* __restrict__ dL_dcolor,
                       float* __restrict__ dL_dmean3D, float* __restrict__ dL_dcov3D,
                       float* __restrict__ dL_dscale, float* __restrict__ dL_drot)
{
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= P) return;
    const float4* a = reinterpret_cast<const float4*>(acc16 + (size_t)idx * 16);
    const float4 a0 = a[0], a1 = a[1], a2 = a[2], a3 = a[3];
    float2* dc = reinterpret_cast<float2*>(dL_dcolor + (size_t)idx * GH_NUM_CHANNELS);
    dc[0] = make_float2(a0.x, a0.y); dc[1] = make_float2(a0.z, a0.w);
    dc[2] = make_float2(a1.x, a1.y); dc[3] = make_float2(a1.z, a1.w);
    dc[4] = make_float2(a2.x, a2.y);
    dL_dmean2D[3 * idx + 0] = a2.z; dL_dmean2D[3 * idx + 1] = a2.w; dL_dmean2D[3 * idx + 2] = 0.f;
    reinterpret_cast<float4*>(dL_dconic)[idx] = make_float4(a3.x, a3.y, 0.f, a3.z);
    dL_dopacity[idx] = a3.w;
    // conic supplied by the caller: nothing flows through the geometry (reference backward.cu:371,398,588)
    if (dL_dmean3D) { dL_dmean3D[3 * idx + 0] = 0.f; dL_dmean3D[3 * idx + 1] = 0.f; dL_dmean3D[3 * idx + 2] = 0.f; }
    if (dL_dcov3D) {
#pragma unroll
        for (int k = 0; k < 6; k++) dL_dcov3D[6 * idx + k] = 0.f;
    }
    if (dL_dscale) { dL_dscale[3 * idx + 0] = 0.f; dL_dscale[3 * idx + 1] = 0.f; dL_dscale[3 * idx + 2] = 0.f; }
    if (dL_drot) reinterpret_cast<float4*>(dL_drot)[idx] = make_float4(0.f, 0.f, 0.f, 0.f);
}

}  // namespace

void gh_launch_blend_forward(int W, int H, int gx, int gy, GhGeomWS geom, GhImgWS img, GhBinWS bin,
                             const float* features, const float* bg, float* out_color,
                             cudaStream_t stream)
{
    // ask for the largest shared-memory carve-out so that 4 CTAs (4 x 48 KB) are resident per SM.
    // The block masks for the backward go to bin.tmp: the long-list sort (gh_tile_split_long_kernel /
    // gh_segment_sort_kernel) uses it as scratch, but that ran to completion before this launch on the same stream.
    const int smem = (int)(sizeof(GhStage) + (GH_CHUNK / 32) * 256 * sizeof(uint32_t));
    cudaFuncSetAttribute(gh_blend_forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    cudaFuncSetAttribute(gh_blend_forward_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    gh_blend_forward_kernel<<<gx * gy, 256, smem, stream>>>(img.ranges, img.tile_perm, bin.inst, geom.geo, features,
                                                         W, H, gx, bg, img.final_T, img.n_contrib, out_color,
                                                         reinterpret_cast<uint2*>(bin.tmp));
}

void gh_launch_blend_backward(int W, int H, int gx, int gy, GhGeomWS geom, GhImgWS img, GhBinWS bin,
                              const float* features, const float* bg, const float* dL_dpix,
                              cudaStream_t stream)
{
    const int smem = (int)(sizeof(GhStageB) + GH_BWD_THREADS * GH_RED2_STRIDE4 * sizeof(float4));
    cudaFuncSetAttribute(gh_blend_backward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    cudaFuncSetAttribute(gh_blend_backward_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    gh_blend_backward_kernel<<<gx * gy, GH_BWD_THREADS, smem, stream>>>(img.ranges, img.tile_perm, bin.inst, geom.geo, features,
                                                          W, H, gx, bg, img.final_T, img.n_contrib, dL_dpix,
                                                          reinterpret_cast<const uint2*>(bin.tmp), geom.acc16);
}

void gh_launch_unpack_grads(int P, GhGeomWS geom, float* dL_dmean2D, float* dL_dconic, float* dL_dopacity,
                            float* dL_dcolor, float* dL_dmean3D, float* dL_dcov3D, float* dL_dscale, float* dL_drot,
                            cudaStream_t stream)
{
    gh_unpack_grads_kernel<<<(P + 255) / 256, 256, 0, stream>>>(P, geom.acc16, dL_dmean2D, dL_dconic,
                                                                dL_dopacity, dL_dcolor, dL_dmean3D, dL_dcov3D,
                                                                dL_dscale, dL_drot);
}
