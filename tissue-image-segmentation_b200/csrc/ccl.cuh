// K3 — connected-component labelling building blocks (union-find, raster-order ids, areas).
//
// Covers skimage.measure.label (unet.py:85, dist.py:107,123, inst_metrics.py:12-13), scipy.ndimage.label
// (hovernet.py:296,358), and the component analysis inside remove_small_objects / binary_fill_holes.
//
// Image access is a functor `Img`:  __device__ bool operator()(int n, long long gi, int& v) const
//   returns whether pixel gi (global index n*P + idx) is foreground; v = the value compared for equality.
//
// par[n*P + idx] = tile-local flat index of the parent (root = lowest index of the component = first pixel
// in raster order, which is what makes skimage's numbering reproducible), -1 for background.
#pragma once
#include <climits>

#include "common.cuh"

namespace tiseg {

// ---- image functors ----------------------------------------------------------------------------
struct ImgEqI32 {               // equal-value components of an int32 image, `bg` is background
    const int32_t* p; int bg;
    __device__ __forceinline__ bool operator()(int n, long long gi, int& v) const { v = p[gi]; return v != bg; }
};
struct ImgEqU8 {                // equal-value components of a uint8 image, bg < 0 => no background
    const uint8_t* p; int bg;
    __device__ __forceinline__ bool operator()(int n, long long gi, int& v) const { v = p[gi]; return v != bg; }
};
struct ImgEqU8Where {           // equal-value components of a uint8 image restricted to the pixels flagged in `on`
    const uint8_t* p; const uint8_t* on;
    __device__ __forceinline__ bool operator()(int n, long long gi, int& v) const { v = p[gi]; return on[gi] != 0; }
};
struct ImgMaskU8 {              // binary: non-zero is foreground
    const uint8_t* p;
    __device__ __forceinline__ bool operator()(int n, long long gi, int& v) const { v = 1; return p[gi] != 0; }
};
struct ImgNotMaskU8 {           // binary complement: zero is foreground (fill-holes background analysis)
    const uint8_t* p;
    __device__ __forceinline__ bool operator()(int n, long long gi, int& v) const { v = 1; return p[gi] == 0; }
};
struct ImgClassU8 {             // binary: pixels of one class id
    const uint8_t* p; int cls;
    __device__ __forceinline__ bool operator()(int n, long long gi, int& v) const { v = 1; return p[gi] == cls; }
};
struct ImgNotClassU8 {          // binary: pixels NOT of one class id
    const uint8_t* p; int cls;
    __device__ __forceinline__ bool operator()(int n, long long gi, int& v) const { v = 1; return p[gi] != cls; }
};
struct ImgEqI32TileBg {         // equal-value components, background value given per tile (arrange_label)
    const int32_t* p; const int* bg;
    __device__ __forceinline__ bool operator()(int n, long long gi, int& v) const { v = p[gi]; return v != bg[n]; }
};
struct ImgAll {                 // every pixel foreground, one value (mask == NULL)
    __device__ __forceinline__ bool operator()(int, long long, int& v) const { v = 1; return true; }
};
struct ImgBelowU8 {             // binary: uint8 value < thr
    const uint8_t* p; int thr;
    __device__ __forceinline__ bool operator()(int, long long gi, int& v) const { v = 1; return p[gi] < thr; }
};
struct ImgOrI32U8 {             // binary: labelled pixel OR foreground pixel (align_foreground's reachable set)
    const int32_t* lab; const uint8_t* fg;
    __device__ __forceinline__ bool operator()(int, long long gi, int& v) const { v = 1; return lab[gi] != 0 || fg[gi] != 0; }
};
struct ImgEqU8Drop {            // equal-value components of a uint8 image, values 0 and `drop` are background
    const uint8_t* p; int drop;
    __device__ __forceinline__ bool operator()(int, long long gi, int& v) const { v = p[gi]; return v != 0 && v != drop; }
};
struct ImgNonZeroI32 {          // binary: non-zero int32
    const int32_t* p;
    __device__ __forceinline__ bool operator()(int n, long long gi, int& v) const { v = 1; return p[gi] != 0; }
};

#ifdef __CUDACC__
// =====================================================================================================
// Three launches per labelling:
//   k_ccl_local   one CTA per 32-row x 128-column tile, FOUR PIXELS PER THREAD (a warp = 128 pixels of a row): values
//                 staged in shared memory, union-find entirely in shared memory — row runs from in-thread compares
//                 plus one ballot (which threads are one unbroken run), merges with the row above by shared
//                 atomicMin — flattened locally, then one 128-bit global write per thread: the tile-global index
//                 of each pixel's local root.  (A pixel-per-lane version of this kernel issued 132 instructions
//                 per 32 pixels and ran issue-bound at 3.4 IPC, profiles/r1_ccl_local_*.)
//   k_ccl_border  only the pixels on tile borders (~4 %) merge across tiles with global atomicMin unions.
//   k_ccl_flatten every pixel points at its global root (lowest flat index of the component = first pixel in
//                 raster order); also leaves the bitmap of the roots for the id ranking that usually follows.
// =====================================================================================================
#define CCL_WARPS 8                     // warps per tile CTA
#define CCL_RPW 4                       // rows per warp
#define CCL_TH (CCL_RPW * CCL_WARPS)    // tile rows
#define CCL_TW 128                      // tile columns: one warp x four pixels
#define CCL_BG INT_MIN                  // background marker inside the shared value tile

static __device__ __noinline__ void uf_union_tile(int* lab, int a, int b) { uf_union(lab, a, b); }

// four consecutive pixels gi .. gi+3 of one row: value, or CCL_BG on the background.  The generic form asks the functor
// pixel by pixel; the functors of the hot paths read the four pixels with one 128-bit / 32-bit load when the address
// is aligned.
template <class Img>
__device__ __forceinline__ void img_quad(const Img& img, int n, long long gi, int (&v)[4]) {
#pragma unroll
    for (int k = 0; k < 4; ++k) { int vv = 0; v[k] = img(n, gi + k, vv) ? vv : CCL_BG; }
}
__device__ __forceinline__ bool quad_u8(const uint8_t* q, int (&b)[4]) {
    if (((uintptr_t)q) & 3) return false;
    const unsigned w = *reinterpret_cast<const unsigned*>(q);
    b[0] = w & 255u; b[1] = (w >> 8) & 255u; b[2] = (w >> 16) & 255u; b[3] = w >> 24;
    return true;
}
__device__ __forceinline__ bool quad_i32(const int32_t* q, int (&b)[4]) {
    if (((uintptr_t)q) & 15) return false;
    const int4 w = *reinterpret_cast<const int4*>(q);
    b[0] = w.x; b[1] = w.y; b[2] = w.z; b[3] = w.w;
    return true;
}
#define TISEG_IMG_QUAD(Type, LOAD, PTR, FG, VAL)                                                                  \
    __device__ __forceinline__ void img_quad(const Type& img, int n, long long gi, int (&v)[4]) {                 \
        int b[4];                                                                                                 \
        if (LOAD(PTR + gi, b)) {                                                                                  \
            _Pragma("unroll") for (int k = 0; k < 4; ++k) v[k] = (FG) ? (VAL) : CCL_BG;                           \
        } else {                                                                                                  \
            _Pragma("unroll") for (int k = 0; k < 4; ++k) { int vv = 0; v[k] = img(n, gi + k, vv) ? vv : CCL_BG; } \
        }                                                                                                         \
    }
TISEG_IMG_QUAD(ImgEqI32, quad_i32, img.p, b[k] != img.bg, b[k])
TISEG_IMG_QUAD(ImgNonZeroI32, quad_i32, img.p, b[k] != 0, 1)
TISEG_IMG_QUAD(ImgEqU8, quad_u8, img.p, b[k] != img.bg, b[k])
TISEG_IMG_QUAD(ImgMaskU8, quad_u8, img.p, b[k] != 0, 1)
TISEG_IMG_QUAD(ImgNotMaskU8, quad_u8, img.p, b[k] == 0, 1)
TISEG_IMG_QUAD(ImgClassU8, quad_u8, img.p, b[k] == img.cls, 1)
TISEG_IMG_QUAD(ImgNotClassU8, quad_u8, img.p, b[k] != img.cls, 1)
TISEG_IMG_QUAD(ImgBelowU8, quad_u8, img.p, b[k] < img.thr, 1)
TISEG_IMG_QUAD(ImgEqU8Drop, quad_u8, img.p, b[k] != 0 && b[k] != img.drop, b[k])
#undef TISEG_IMG_QUAD

template <class Img, int CONN, bool LISTED>
__global__ void __launch_bounds__(32 * CCL_WARPS, LISTED ? 1 : 5) k_ccl_local(Geom g, Img img, int* __restrict__ par, bool vec) {
    __shared__ __align__(16) int sval[CCL_TH * CCL_TW];
    __shared__ __align__(16) int slab[CCL_TH * CCL_TW];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int tilesX = (g.W + CCL_TW - 1) / CCL_TW;
    const int ty = blockIdx.x / tilesX, tx = blockIdx.x - ty * tilesX;
    const int x0 = tx * CCL_TW + lane * 4, yt = ty * CCL_TH;
    // rows are dealt to the warps round-robin (warp w owns rows w, w + CCL_WARPS, ...): a nucleus spreads over all the
    // warps, so they reach the barriers together instead of one warp doing a blob's unions while the others wait
    FOR_TILES(LISTED, g, n) {
    const long long base = (long long)n * g.P;
    // phase A: loads (all rows of the thread in flight), in-thread runs, run starts across threads, staging
    int v[CCL_RPW][4];
    unsigned cm[CCL_RPW];               // bit k: pixel k continues the run of the pixel to its left
    unsigned fgm[CCL_RPW];              // bit k: pixel k is foreground
    int l0[CCL_RPW];                    // label (tile-local index of the run start) of the run pixel 0 belongs to
#pragma unroll
    for (int r = 0; r < CCL_RPW; ++r) {
        const int y = yt + r * CCL_WARPS + warp;
        if (y < g.H && x0 + 3 < g.W) img_quad(img, n, base + (long long)y * g.W + x0, v[r]);
        else {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                int vv = 0;
                v[r][k] = CCL_BG;
                if (y < g.H && x0 + k < g.W && img(n, base + (long long)y * g.W + x0 + k, vv)) v[r][k] = vv;
            }
        }
    }
#pragma unroll
    for (int r = 0; r < CCL_RPW; ++r) {
        const int row = r * CCL_WARPS + warp, li0 = row * CCL_TW + lane * 4;
        int left = __shfl_up_sync(0xffffffffu, v[r][3], 1);
        if (lane == 0) left = CCL_BG;
        const unsigned f = (v[r][0] != CCL_BG ? 1u : 0u) | (v[r][1] != CCL_BG ? 2u : 0u) | (v[r][2] != CCL_BG ? 4u : 0u) |
                           (v[r][3] != CCL_BG ? 8u : 0u);
        const unsigned c = ((v[r][0] == left ? 1u : 0u) | (v[r][1] == v[r][0] ? 2u : 0u) | (v[r][2] == v[r][1] ? 4u : 0u) |
                            (v[r][3] == v[r][2] ? 8u : 0u)) & f;
        fgm[r] = f; cm[r] = c;
        // threads that are one unbroken continuation of the run to their left; the run of my pixel 0 (if it
        // continues) started in the nearest lower lane that is not one, at that lane's last in-thread start
        const unsigned full = __ballot_sync(0xffffffffu, c == 15u);
        const unsigned lower = ~full & ((1u << lane) - 1u);
        const int src = lower ? 31 - __clz(lower) : 0;
        const int s3 = 31 - __clz((~c & 15u) | 1u);                 // in-thread start of the run of pixel 3 (0 if unbroken)
        const int inherited = __shfl_sync(0xffffffffu, li0 + s3, src);
        l0[r] = (c & 1u) ? inherited : li0;
        // label of pixel k = last break at or below k (the run start inside the thread), or the inherited one
        const unsigned brk = ~c & 15u;
        int4 lab;
        lab.x = (f & 1u) ? l0[r] : -1;
        lab.y = (f & 2u) ? ((brk & 2u) ? li0 + 1 : l0[r]) : -1;
        lab.z = (f & 4u) ? ((brk & 4u) ? li0 + 2 : (brk & 2u) ? li0 + 1 : l0[r]) : -1;
        lab.w = (f & 8u) ? ((brk & 14u) ? li0 + s3 : l0[r]) : -1;
        *reinterpret_cast<int4*>(&sval[li0]) = make_int4(v[r][0], v[r][1], v[r][2], v[r][3]);
        *reinterpret_cast<int4*>(&slab[li0]) = lab;
    }
    __syncthreads();
    // phase B: merge with the row above (same redundancy rule as documented at k_ccl_border), decided for the four
    // pixels at once as bit masks; the inside of a blob needs no union at all
#pragma unroll
    for (int r = 0; r < CCL_RPW; ++r) {
        const int row = r * CCL_WARPS + warp, li0 = row * CCL_TW + lane * 4;
        if (row == 0 || !fgm[r]) continue;
        const int4 up = *reinterpret_cast<const int4*>(&sval[li0 - CCL_TW]);
        const int ul = lane > 0 ? sval[li0 - CCL_TW - 1] : CCL_BG;
        const int ur = lane < 31 ? sval[li0 - CCL_TW + 4] : CCL_BG;
        const unsigned eU = ((up.x == v[r][0] ? 1u : 0u) | (up.y == v[r][1] ? 2u : 0u) | (up.z == v[r][2] ? 4u : 0u) |
                             (up.w == v[r][3] ? 8u : 0u)) & fgm[r];
        const unsigned eL = ((ul == v[r][0] ? 1u : 0u) | (up.x == v[r][1] ? 2u : 0u) | (up.y == v[r][2] ? 4u : 0u) |
                             (up.z == v[r][3] ? 8u : 0u)) & fgm[r];
        unsigned need_u = eU & ~(cm[r] & eL), need_l = 0, need_r = 0;
        if (CONN == 2) {
            const unsigned eR = ((up.y == v[r][0] ? 1u : 0u) | (up.z == v[r][1] ? 2u : 0u) | (up.w == v[r][2] ? 4u : 0u) |
                                 (ur == v[r][3] ? 8u : 0u)) & fgm[r];
            need_l = ~eU & eL & ~cm[r];
            need_r = ~eU & eR;
        }
        unsigned todo = need_u | (need_l << 4) | (need_r << 8);
        while (todo) {
            const int b = __ffs(todo) - 1;
            todo &= todo - 1;
            const int k = b & 3, li = li0 + k;
            uf_union_tile(slab, li, li - CCL_TW + (b >> 2 == 0 ? 0 : b >> 2 == 1 ? -1 : 1));
        }
    }
    __syncthreads();
    // phase C1: the threads that hold a run START point it at its local root (the inside of a blob has nothing to do)
#pragma unroll
    for (int r = 0; r < CCL_RPW; ++r) {
        const int li0 = (r * CCL_WARPS + warp) * CCL_TW + lane * 4;
        unsigned starts = fgm[r] & ~cm[r];
        while (starts) {
            const int k = __ffs(starts) - 1;
            starts &= starts - 1;
            const int root = uf_find(slab, li0 + k);
            if (root != li0 + k) slab[li0 + k] = root;
        }
    }
    __syncthreads();
    // phase C2: every pixel reads the root through its run start (its own label); one 128-bit global write per thread
#pragma unroll
    for (int r = 0; r < CCL_RPW; ++r) {
        const int row = r * CCL_WARPS + warp, y = yt + row, li0 = row * CCL_TW + lane * 4;
        if (y >= g.H || x0 >= g.W) continue;
        const int4 lab = *reinterpret_cast<const int4*>(&slab[li0]);
        const int q0 = slab[max(lab.x, 0)], q1 = slab[max(lab.y, 0)], q2 = slab[max(lab.z, 0)], q3 = slab[max(lab.w, 0)];
        const int off = yt * g.W + tx * CCL_TW;
        int4 out;
        out.x = lab.x >= 0 ? (q0 >> 7) * g.W + (q0 & (CCL_TW - 1)) + off : -1;
        out.y = lab.y >= 0 ? (q1 >> 7) * g.W + (q1 & (CCL_TW - 1)) + off : -1;
        out.z = lab.z >= 0 ? (q2 >> 7) * g.W + (q2 & (CCL_TW - 1)) + off : -1;
        out.w = lab.w >= 0 ? (q3 >> 7) * g.W + (q3 & (CCL_TW - 1)) + off : -1;
        int* dst = par + base + (long long)y * g.W + x0;
        if (vec) *reinterpret_cast<int4*>(dst) = out;
        else {
            if (x0 < g.W) dst[0] = out.x;
            if (x0 + 1 < g.W) dst[1] = out.y;
            if (x0 + 2 < g.W) dst[2] = out.z;
            if (x0 + 3 < g.W) dst[3] = out.w;
        }
    }
    if (LISTED) __syncthreads();        // the shared tile is reused by the next listed tile
    }
}

// Cross-tile merges.  Candidates: A) pixels of a tile's top row (y = 32k, k >= 1) look up / up-left / up-right;
// B) pixels of a tile's left column (x = 128k, k >= 1) look left / up-left; C) (8-connectivity) pixels of a tile's
// right column (x = 128k - 1) look up-right.  A diagonal union is skipped when the vertical neighbour has the same
// value (it is then connected through that neighbour's own row).
template <class Img, int CONN>
__device__ __forceinline__ void ccl_border_one(const Geom& g, const Img& img, int* par, int n, int t) {
    const int tilesY = (g.H + CCL_TH - 1) / CCL_TH, tilesX = (g.W + CCL_TW - 1) / CCL_TW;
    const int nA = (tilesY - 1) * g.W, nB = (tilesX - 1) * g.H, nC = CONN == 2 ? nB : 0;
    if (t >= nA + nB + nC) return;
    int y, x, kind;
    if (t < nA) { kind = 0; y = (t / g.W + 1) * CCL_TH; x = t - (t / g.W) * g.W; }
    else if (t < nA + nB) { t -= nA; kind = 1; x = (t / g.H + 1) * CCL_TW; y = t - (t / g.H) * g.H; }
    else { t -= nA + nB; kind = 2; x = (t / g.H + 1) * CCL_TW - 1; y = t - (t / g.H) * g.H; }
    const long long base = (long long)n * g.P;
    const int idx = y * g.W + x;
    int v = 0;
    if (!img(n, base + idx, v)) return;
    int* tp = par + base;
    int w = 0;
    bool sU = y > 0 && img(n, base + idx - g.W, w) && w == v;
    if (kind == 0) {
        if (sU) uf_union(tp, idx, idx - g.W);
        else if (CONN == 2) {
            if (x > 0 && img(n, base + idx - g.W - 1, w) && w == v) uf_union(tp, idx, idx - g.W - 1);
            if (x + 1 < g.W && img(n, base + idx - g.W + 1, w) && w == v) uf_union(tp, idx, idx - g.W + 1);
        }
    } else if (kind == 1) {
        if (img(n, base + idx - 1, w) && w == v) uf_union(tp, idx, idx - 1);
        else if (CONN == 2 && !sU && y > 0 && img(n, base + idx - g.W - 1, w) && w == v) uf_union(tp, idx, idx - g.W - 1);
    } else {
        if (!sU && y > 0 && x + 1 < g.W && img(n, base + idx - g.W + 1, w) && w == v) uf_union(tp, idx, idx - g.W + 1);
    }
}
template <class Img, int CONN, bool LISTED>
__global__ void __launch_bounds__(256) k_ccl_border(Geom g, Img img, int* par) {
    FOR_TILES(LISTED, g, n) ccl_border_one<Img, CONN>(g, img, par, n, blockIdx.x * blockDim.x + threadIdx.x);
}

// flatten + bitmap of the roots; defined in ccl.cu
int ccl_flatten(tiseg_ctx* c, const Geom& g, int* par);

// build + flatten.  par: [N*P] int
template <class Img>
int ccl_build(tiseg_ctx* c, const Geom& g, Img img, int conn, int* par) {
    const int tilesY = (g.H + CCL_TH - 1) / CCL_TH, tilesX = (g.W + CCL_TW - 1) / CCL_TW;
    dim3 lg((unsigned)(tilesX * tilesY), grid_tiles(g));
    const int nb = (tilesY - 1) * g.W + (tilesX - 1) * g.H * (conn == 2 ? 2 : 1);
    const bool vec = (g.W % 4 == 0) && aligned16(par);
    if (g.tl) {
        if (conn == 1) {
            TISEG_LAUNCH(c, (k_ccl_local<Img, 1, true>), lg, 32 * CCL_WARPS, 0, g, img, par, vec);
            if (nb > 0) TISEG_LAUNCH(c, (k_ccl_border<Img, 1, true>), dim3((nb + 255) / 256, 1), 256, 0, g, img, par);
        } else {
            TISEG_LAUNCH(c, (k_ccl_local<Img, 2, true>), lg, 32 * CCL_WARPS, 0, g, img, par, vec);
            if (nb > 0) TISEG_LAUNCH(c, (k_ccl_border<Img, 2, true>), dim3((nb + 255) / 256, 1), 256, 0, g, img, par);
        }
    } else if (conn == 1) {
        TISEG_LAUNCH(c, (k_ccl_local<Img, 1, false>), lg, 32 * CCL_WARPS, 0, g, img, par, vec);
        if (nb > 0) TISEG_LAUNCH(c, (k_ccl_border<Img, 1, false>), dim3((nb + 255) / 256, g.N), 256, 0, g, img, par);
    } else {
        TISEG_LAUNCH(c, (k_ccl_local<Img, 2, false>), lg, 32 * CCL_WARPS, 0, g, img, par, vec);
        if (nb > 0) TISEG_LAUNCH(c, (k_ccl_border<Img, 2, false>), dim3((nb + 255) / 256, g.N), 256, 0, g, img, par);
    }
    return ccl_flatten(c, g, par);
}
#endif

// ---- raster-order ranks ------------------------------------------------------------------------
// Selection is a functor  __device__ bool operator()(long long gi, int idx) const  (e.g. "is a root").
// rank[gi] = 1-based raster rank among the selected pixels of its tile (written only where selected);
// counts[n] = number selected (may be null).
// The selection is first reduced to a BITMAP, one 32-bit ballot word per row segment (bits[n, y, seg]); ranking then
// touches P/32 words instead of P pixels: k_rank_fused (one cluster of CTAs per tile: popcount per row, exclusive scan
// over the rows, then one warp per row: warp scan over the row's words, one store per selected pixel).
struct SelRoot {                // roots of a flattened forest
    const int* par;
    __device__ __forceinline__ bool operator()(long long gi, int idx) const { return par[gi] == idx; }
};
struct SelFlagU8 {
    const uint8_t* f;
    __device__ __forceinline__ bool operator()(long long gi, int) const { return f[gi] != 0; }
};

#ifdef __CUDACC__
// bits[n, y, seg] = ballot of the selected pixels of that 32-pixel row segment
template <class Sel>
__global__ void __launch_bounds__(TISEG_THREADS) k_rank_bits(Geom g, Sel sel, unsigned* __restrict__ bits) {
    Strip s;
    if (!warp_strip(g, s)) return;
    bool f[STRIP_R];
#pragma unroll
    for (int r = 0; r < STRIP_R; ++r) {
        int y = s.y0 + r;
        f[r] = s.okx && y < g.H && sel(s.base + (long long)y * g.W + s.x, y * g.W + s.x);
    }
#pragma unroll
    for (int r = 0; r < STRIP_R; ++r) {
        unsigned m = __ballot_sync(0xffffffffu, f[r]);
        int y = s.y0 + r;
        if (s.lane == 0 && y < g.H) bits[((long long)s.n * g.H + y) * g.SEG + s.seg] = m;
    }
}

// bitmap -> ranks (defined in ccl.cu)
int rank_from_bits(tiseg_ctx* c, const Geom& g, const unsigned* bits, int* rank, int* counts);

template <class Sel>
int rank_generic(tiseg_ctx* c, const Geom& g, Sel sel, int* rank, int* counts) {
    unsigned* bits = ws<unsigned>(c, (size_t)g.N * g.H * g.SEG);
    if (!bits) return TISEG_ERR_CUDA;
    TISEG_LAUNCH(c, k_rank_bits<Sel>, strip_grid(g), TISEG_THREADS, 0, g, sel, bits);
    return rank_from_bits(c, g, bits, rank, counts);
}
#endif

// roots of a flattened forest: rank[root] = raster rank (1-based); counts[n] = K
int rank_roots(tiseg_ctx* c, const Geom& g, const int* par, int* rank, int* counts);
// out[gi] = par[gi] >= 0 ? rank[par[gi]] : 0
int apply_rank(tiseg_ctx* c, const Geom& g, const int* par, const int* rank, int32_t* out);
// area[root] = component size (this zeroes `area` itself; valid at root positions only)
int ccl_areas(tiseg_ctx* c, const Geom& g, const int* par, int* area);

// full label: img functor -> out ids (1..K raster order), counts
template <class Img>
int ccl_label(tiseg_ctx* c, const Geom& g, Img img, int conn, int32_t* out, int* counts) {
#ifdef __CUDACC__
    size_t total = (size_t)g.N * g.P;
    int* par = ws<int>(c, total);
    int* rank = ws<int>(c, total);
    if (!par || !rank) return TISEG_ERR_CUDA;
    TISEG_TRY(ccl_build(c, g, img, conn, par));
    TISEG_TRY(rank_roots(c, g, par, rank, counts));
    TISEG_TRY(apply_rank(c, g, par, rank, out));
#endif
    return TISEG_OK;
}

}  // namespace tiseg
