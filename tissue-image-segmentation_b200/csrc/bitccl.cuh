// Connected components on BIT PLANES: the per-pixel work of a labelling is reduced to one streaming pass that turns the
// image into five bit planes (one 32-bit ballot word per 32-pixel row segment and plane); everything after that — the
// union-find, the cross-tile merges, the root bitmaps, and the consumers that only need to know WHICH component a pixel
// run belongs to (pair histogram, blob boxes, flood staging) — works on words and on the horizontal RUNS they describe,
// never on pixels.  The pixel-level shared-memory union-find of ccl.cuh issues ~4.4 warp instructions per pixel and map
// (profiles/r2_pair_local_*: 566 M warp instructions for two 64 x 1000^2 labellings, 45 % of them in single-lane
// union / find loops); here the streaming pass costs ~0.7 and the rest is proportional to the number of runs.
//
// Planes (bit x of word [n, y, seg] = pixel 32 * seg + x of row y; bits beyond W are zero):
//   F   pixel is foreground
//   C   foreground and equal to its left neighbour            (same run)
//   EU  foreground and equal to the pixel above
//   EL  foreground and equal to the pixel above-left
//   ER  foreground and equal to the pixel above-right
// For a binary mask only F is stored and the other four are derived with shifts (BitPlanes::C == nullptr).
//
// Nodes of the union-find are the runs of a TILE ROW: a run is cut where it crosses a tile's left edge, so that every
// node lies inside one tile of BT_TH rows x BT_TWW words and the tile kernel needs no neighbour.  A node's id is the
// tile-local / tile-global flat index of its first pixel; `par` is a pixel-indexed int array that is only ever touched
// at run starts (root = lowest index of the component = its first pixel in raster order, as everywhere in this library).
//   k_bitccl_tile     one CTA per tile, one thread per word: unions inside the tile in shared memory, then
//                     par[run start] = local root (global index) and the bitmap of the local roots
//   k_bitccl_border   the unions that cross tile edges (top rows of tiles, first / last column of tiles)
//   k_bitccl_resolve  local roots -> final roots; bitmap of the final roots (what the raster-order ranking consumes)
#pragma once
#include "common.cuh"

namespace tiseg {

#define BT_TH 32                 // tile rows
#define BT_TWW 8                 // tile width in words (256 pixels)
#define BT_TW (32 * BT_TWW)
#define BT_THREADS (BT_TH * BT_TWW)

struct BitPlanes {
    const unsigned* F;
    const unsigned* C;           // nullptr: binary mask, planes derived from F
    const unsigned* EU;
    const unsigned* EL;
    const unsigned* ER;
};
struct BitPlanesW { unsigned *F, *C, *EU, *EL, *ER; };
inline BitPlanes as_const(const BitPlanesW& w) { return BitPlanes{w.F, w.C, w.EU, w.EL, w.ER}; }

// allocation of the five planes of `maps` tile batches in the call workspace
inline int bitplanes_alloc(tiseg_ctx* c, const Geom& g, int maps, BitPlanesW& p) {
    const size_t words = (size_t)maps * g.N * g.H * g.SEG;
    p.F = ws<unsigned>(c, words); p.C = ws<unsigned>(c, words); p.EU = ws<unsigned>(c, words);
    p.EL = ws<unsigned>(c, words); p.ER = ws<unsigned>(c, words);
    return (p.F && p.C && p.EU && p.EL && p.ER) ? TISEG_OK : TISEG_ERR_CUDA;
}

#ifdef __CUDACC__
// read-only find (the forest is final: no concurrent unions)
__device__ __forceinline__ int find_ro(const int* __restrict__ par, int x) {
    int q = par[x];
    while (q != x) { x = q; q = par[x]; }
    return x;
}

struct Masks { unsigned f, c, eu, el, er; };

// the five masks of word (y, seg) of tile-batch entry `n` (wo = n * H * SEG), as the image defines them (not cut at
// tile edges)
__device__ __forceinline__ Masks bit_masks(const BitPlanes& p, const Geom& g, long long wo, int y, int seg) {
    Masks m;
    const long long i = wo + (long long)y * g.SEG + seg;
    m.f = p.F[i];
    if (p.C) {
        m.c = p.C[i]; m.eu = p.EU[i]; m.el = p.EL[i]; m.er = p.ER[i];
        return m;
    }
    const unsigned fl = seg > 0 ? p.F[i - 1] : 0u;
    m.c = m.f & ((m.f << 1) | (fl >> 31));
    m.eu = m.el = m.er = 0u;
    if (y > 0) {
        const unsigned u = p.F[i - g.SEG];
        const unsigned ul = seg > 0 ? p.F[i - g.SEG - 1] : 0u, ur = seg + 1 < g.SEG ? p.F[i - g.SEG + 1] : 0u;
        m.eu = m.f & u;
        m.el = m.f & ((u << 1) | (ul >> 31));
        m.er = m.f & ((u >> 1) | (ur << 31));
    }
    return m;
}

// run starts of word (y, seg) with runs cut at the left edge of every tile
__device__ __forceinline__ unsigned bit_starts(const BitPlanes& p, const Geom& g, long long wo, int y, int seg) {
    const long long i = wo + (long long)y * g.SEG + seg;
    const unsigned f = p.F[i];
    unsigned c;
    if (p.C) c = p.C[i];
    else c = f & ((f << 1) | (seg > 0 ? p.F[i - 1] >> 31 : 0u));
    if (seg % BT_TWW == 0) c &= ~1u;
    return f & ~c;
}

// tile-global flat index of the first pixel of the tile-row run that contains foreground pixel (y, x)
__device__ __forceinline__ int bit_node_of(const BitPlanes& p, const Geom& g, long long wo, int y, int x) {
    int seg = x >> 5;
    unsigned m = bit_starts(p, g, wo, y, seg) & (0xffffffffu >> (31 - (x & 31)));
    while (!m) { --seg; m = bit_starts(p, g, wo, y, seg); }      // ends inside the tile row: its first pixel starts a run
    return y * g.W + seg * 32 + 31 - __clz(m);
}

// ---- streaming pass: int32 label map -> planes (equal-value components, background 0) ---------------------------------
// One warp = one 256-pixel column strip x EQ_BAND rows, walking down, EIGHT pixels per thread (two 128-bit loads per row).
// The row above stays in registers, so every pixel is loaded once (plus the two strip-edge columns).  The pass is
// ISSUE-bound (profiles/r2_*: 180 warp instructions per 128 pixels of a row at 2.5 IPC in its first form), so
//   * per pixel k, eq_px<k> ORs bit k of byte 0 / 1 / 2 of A (planes F, C, EU) and of byte 0 / 1 of B (EL, ER): one
//     ISETP (the "pixel is foreground" predicate rides along as the AND input) + one predicated LOP3 per plane;
//   * eq_words5 assembles the 32-bit words of the five planes from the bytes of the four lanes of a word group with a
//     reduce-scatter — TWO shuffles instead of two per plane: step 1 (lane ^ 1) even lanes collect the 16-bit halves of
//     F, C, EU, odd lanes those of EL, ER; step 2 (lane ^ 2) the words.  Lane (group + 0) ends with the words of F and C,
//     lanes + 2, + 1, + 3 with EU, EL, ER, and each stores its own;
//   * eight pixels per thread halve the per-row overhead (neighbour shuffles, vote, assembly, stores) per pixel.
#define EQ_BAND 32
#define EQ_UNROLL 2
template <int K>
__device__ __forceinline__ void eq_px(int v, int left, int up, int upl, int upr, unsigned& A, unsigned& B) {
    asm("{\n\t.reg .pred pf, p;\n\t"
        "setp.ne.s32 pf, %2, 0;\n\t"
        "@pf or.b32 %0, %0, %7;\n\t"
        "setp.eq.and.s32 p, %2, %3, pf;\n\t"
        "@p or.b32 %0, %0, %8;\n\t"
        "setp.eq.and.s32 p, %2, %4, pf;\n\t"
        "@p or.b32 %0, %0, %9;\n\t"
        "setp.eq.and.s32 p, %2, %5, pf;\n\t"
        "@p or.b32 %1, %1, %7;\n\t"
        "setp.eq.and.s32 p, %2, %6, pf;\n\t"
        "@p or.b32 %1, %1, %8;\n\t}"
        : "+r"(A), "+r"(B)
        : "r"(v), "r"(left), "r"(up), "r"(upl), "r"(upr), "n"(1 << K), "n"(256 << K), "n"(65536 << K));
}
// -> w0: the word of F (lane & 3 == 0), EL (1), EU (2), ER (3); w1: the word of C (lane & 3 == 0)
__device__ __forceinline__ void eq_words5(unsigned A, unsigned B, bool b0, bool b1, unsigned& w0, unsigned& w1) {
    const unsigned r1 = __shfl_xor_sync(0xffffffffu, b0 ? A : B, 1), own = b0 ? B : A;
    const unsigned lo = b0 ? r1 : own, hi = b0 ? own : r1;
    const unsigned Xlo = __byte_perm(lo, hi, 0x5140), Xhi = __byte_perm(lo, hi, 0x3362);
    const unsigned r2 = __shfl_xor_sync(0xffffffffu, b0 ? (b1 ? (Xlo & 0xffffu) : (Xlo >> 16)) : (b1 ? Xlo : Xhi), 2);
    w0 = b1 ? (b0 ? __byte_perm(r2, Xlo, 0x7610) : __byte_perm(r2, Xhi, 0x5410)) : __byte_perm(Xlo, r2, 0x5410);
    w1 = __byte_perm(Xlo, r2, 0x7632);
}
// T = int32_t, or uint16_t (instance maps with ids below 65536 shipped at half the bytes).  VEC: rows are 16-byte aligned
// and W % 4 == 0, so each aligned group of four pixels is inside the row or outside it as a whole.
template <class T, bool VEC>
__device__ __forceinline__ void eq_load8(const T* __restrict__ rp, int x, int W, int (&v)[8]) {
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = 0;
    if (VEC) {
        if (sizeof(T) == 4) {
            if (x + 3 < W) { const int4 q = *reinterpret_cast<const int4*>(rp); v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w; }
            if (x + 7 < W) { const int4 q = *reinterpret_cast<const int4*>(rp + 4); v[4] = q.x; v[5] = q.y; v[6] = q.z; v[7] = q.w; }
        } else {
            if (x + 3 < W) { const uint2 q = *reinterpret_cast<const uint2*>(rp); v[0] = q.x & 0xffffu; v[1] = q.x >> 16; v[2] = q.y & 0xffffu; v[3] = q.y >> 16; }
            if (x + 7 < W) { const uint2 q = *reinterpret_cast<const uint2*>(rp + 4); v[4] = q.x & 0xffffu; v[5] = q.x >> 16; v[6] = q.y & 0xffffu; v[7] = q.y >> 16; }
        }
    } else {
#pragma unroll
        for (int k = 0; k < 8; ++k) if (x + k < W) v[k] = (int)rp[k];
    }
}
struct EqRow { int pv[8], pvL, pvR; };
// one row: the words of the five planes from the row `v` (+ the strip's outer neighbour `e`) and the row above (st)
__device__ __forceinline__ void eq_row(const int (&v)[8], int e, EqRow& st, int lane, bool b0, bool b1, unsigned* mp, unsigned* mp2) {
    int vL = __shfl_up_sync(0xffffffffu, v[7], 1), vR = __shfl_down_sync(0xffffffffu, v[0], 1);
    if (lane == 0) vL = e;
    if (lane == 31) vR = e;
    unsigned w0 = 0u, w1 = 0u;
    if (__any_sync(0xffffffffu, (v[0] | v[1] | v[2] | v[3] | v[4] | v[5] | v[6] | v[7]) != 0)) {   // (uniform) background rows are cheap
        unsigned A = 0u, B = 0u;
        eq_px<0>(v[0], vL, st.pv[0], st.pvL, st.pv[1], A, B);
        eq_px<1>(v[1], v[0], st.pv[1], st.pv[0], st.pv[2], A, B);
        eq_px<2>(v[2], v[1], st.pv[2], st.pv[1], st.pv[3], A, B);
        eq_px<3>(v[3], v[2], st.pv[3], st.pv[2], st.pv[4], A, B);
        eq_px<4>(v[4], v[3], st.pv[4], st.pv[3], st.pv[5], A, B);
        eq_px<5>(v[5], v[4], st.pv[5], st.pv[4], st.pv[6], A, B);
        eq_px<6>(v[6], v[5], st.pv[6], st.pv[5], st.pv[7], A, B);
        eq_px<7>(v[7], v[6], st.pv[7], st.pv[6], st.pvR, A, B);
        eq_words5(A, B, b0, b1, w0, w1);
    }
    if (mp) *mp = w0;
    if (mp2) *mp2 = w1;
#pragma unroll
    for (int k = 0; k < 8; ++k) st.pv[k] = v[k];
    st.pvL = vL; st.pvR = vR;
}
template <class T, bool VEC>
__device__ __forceinline__ void eq_strip(const Geom& g, const T* __restrict__ t, int lane, int x, int y0, int y1, unsigned* mp, unsigned* mp2) {
    // the strip's outer neighbours: lane 0 looks one pixel to the left of the strip, lane 31 one to the right
    const int xe = lane == 0 ? x - 1 : x + 8;
    const bool oke = (lane == 0 || lane == 31) && xe >= 0 && xe < g.W;
    const bool b0 = lane & 1, b1 = lane & 2;
    const T* rp = t + (long long)y0 * g.W + x;            // walks down one row at a time
    const T* ep = t + (long long)y0 * g.W + xe;
    EqRow st;
#pragma unroll
    for (int k = 0; k < 8; ++k) st.pv[k] = 0;
    st.pvL = st.pvR = 0;
    if (y0 > 0) {
        eq_load8<T, VEC>(rp - g.W, x, g.W, st.pv);
        const int e = oke ? (int)*(ep - g.W) : 0;
        st.pvL = __shfl_up_sync(0xffffffffu, st.pv[7], 1);
        st.pvR = __shfl_down_sync(0xffffffffu, st.pv[0], 1);
        if (lane == 0) st.pvL = e;
        if (lane == 31) st.pvR = e;
    }
    // software pipeline: the loads of chunk i + 1 are issued before the arithmetic of chunk i (a warp's walk is a chain of
    // load latencies otherwise: 16 iterations x ~2 us left the pass at 40 % of the HBM rate)
    int nxt[EQ_UNROLL][8], next[EQ_UNROLL];
    auto issue = [&](int yy) {                               // rows yy .. yy + EQ_UNROLL - 1 (zeros beyond y1)
#pragma unroll
        for (int u = 0; u < EQ_UNROLL; ++u) {
            if (yy + u < y1) {
                eq_load8<T, VEC>(rp + (long long)u * g.W, x, g.W, nxt[u]);
                next[u] = oke ? (int)ep[(long long)u * g.W] : 0;
            } else {
#pragma unroll
                for (int k = 0; k < 8; ++k) nxt[u][k] = 0;
                next[u] = 0;
            }
        }
        rp += (long long)EQ_UNROLL * g.W; ep += (long long)EQ_UNROLL * g.W;
    };
    issue(y0);
    for (int y = y0; y < y1; y += EQ_UNROLL) {
        int cur[EQ_UNROLL][8], ext[EQ_UNROLL];
#pragma unroll
        for (int u = 0; u < EQ_UNROLL; ++u) {
#pragma unroll
            for (int k = 0; k < 8; ++k) cur[u][k] = nxt[u][k];
            ext[u] = next[u];
        }
        if (y + EQ_UNROLL < y1) issue(y + EQ_UNROLL);
#pragma unroll
        for (int u = 0; u < EQ_UNROLL; ++u) {
            if (y + u >= y1) break;                           // (uniform)
            eq_row(cur[u], ext[u], st, lane, b0, b1, mp, mp2);
            if (mp) mp += g.SEG;
            if (mp2) mp2 += g.SEG;
        }
    }
}
template <class T>
__global__ void __launch_bounds__(TISEG_THREADS)
k_eqbits(Geom g, const T* __restrict__ img, BitPlanesW out, bool vec) {
    const int lane = threadIdx.x & 31;
    const int bands = (g.H + EQ_BAND - 1) / EQ_BAND, strips = (g.W + 255) >> 8;
    const long long wi = (long long)blockIdx.x * TISEG_WARPS_PER_BLOCK + (threadIdx.x >> 5);
    if (wi >= (long long)strips * bands) return;
    const int band = (int)(wi / strips), strip = (int)(wi - (long long)band * strips), n = blockIdx.y;
    const int x = strip * 256 + lane * 8, y0 = band * EQ_BAND, y1 = min(y0 + EQ_BAND, g.H);
    const T* t = img + (long long)n * g.P;
    const int seg = strip * 8 + (lane >> 2);
    unsigned *mp = nullptr, *mp2 = nullptr;         // the plane(s) whose words this lane ends up with (eq_words5)
    if (seg < g.SEG) {
        const int role = lane & 3;
        const long long o = ((long long)n * g.H + y0) * g.SEG + seg;
        mp = (role == 0 ? out.F : role == 2 ? out.EU : role == 1 ? out.EL : out.ER) + o;
        if (role == 0) mp2 = out.C + o;
    }
    if (vec) eq_strip<T, true>(g, t, lane, x, y0, y1, mp, mp2);
    else eq_strip<T, false>(g, t, lane, x, y0, y1, mp, mp2);
}

// ---- tile union-find on the planes -------------------------------------------------------------------------------------
static __device__ __noinline__ void bt_union(int* par, int a, int b) { uf_union(par, a, b); }

// tile-local node (row * BT_TW + column of the run start) of foreground pixel (row, x) from the tile's start masks
__device__ __forceinline__ int bt_node_of(const unsigned (*sS)[BT_TWW], int row, int x) {
    int w = x >> 5;
    unsigned m = sS[row][w] & (0xffffffffu >> (31 - (x & 31)));
    while (!m) { --w; m = sS[row][w]; }
    return row * BT_TW + w * 32 + 31 - __clz(m);
}

// p: planes of `g.N` tile-batch entries; par [g.N, P]; lbits [g.N, H, SEG].  conn 1: 4-neighbourhood, 2: 8.
// `bad` / `low` (may be null): a bit plane of flagged pixels; low[local root] = 1 for every tile component that holds one
// (k_bitccl_resolve carries the flags on to the final roots).  `low` is cleared at every node first (each tile clears its
// own nodes before its first barrier); it is only meaningful at the nodes.
template <int CONN>
__global__ void __launch_bounds__(BT_THREADS)
k_bitccl_tile(Geom g, BitPlanes p, int* __restrict__ par, unsigned* __restrict__ lbits, const unsigned* __restrict__ bad,
              uint8_t* __restrict__ low) {
    __shared__ int spar[BT_TH * BT_TW];
    __shared__ unsigned sS[BT_TH][BT_TWW];
    const int tilesX = (g.SEG + BT_TWW - 1) / BT_TWW;
    const int ty = blockIdx.x / tilesX, tx = blockIdx.x - ty * tilesX, n = blockIdx.y;
    const int r = threadIdx.x / BT_TWW, w = threadIdx.x - r * BT_TWW;
    const int y = ty * BT_TH + r, seg = tx * BT_TWW + w;
    const long long wo = (long long)n * g.H * g.SEG;
    const bool live = y < g.H && seg < g.SEG;
    Masks m = {0u, 0u, 0u, 0u, 0u};
    if (live) m = bit_masks(p, g, wo, y, seg);
    // connections that leave the tile belong to k_bitccl_border
    if (w == 0) { m.c &= ~1u; m.el &= ~1u; }
    if (w == BT_TWW - 1) m.er &= 0x7fffffffu;
    if (r == 0) m.eu = m.el = m.er = 0u;
    const unsigned S = m.f & ~m.c;
    sS[r][w] = S;
    const int node0 = r * BT_TW + w * 32;
    // the flags of the tile's own nodes start at 0 (they are raised after the second barrier, on nodes of this tile only)
    uint8_t* lown = low ? low + (long long)n * g.P + (long long)y * g.W + seg * 32 : nullptr;
    for (unsigned s = S; s; s &= s - 1) {
        const int b = __ffs(s) - 1;
        spar[node0 + b] = node0 + b;
        if (lown) lown[b] = 0;
    }
    __syncthreads();
    // unions with the row above; a pixel that continues its run and whose left neighbour already sits under the same
    // upper run needs none (rule of k_ccl_local)
    unsigned need_u = m.eu & ~(m.c & m.el), need_l = 0u, need_r = 0u;
    if (CONN == 2) { need_l = ~m.eu & m.el & ~m.c; need_r = ~m.eu & m.er; }
    for (unsigned s = need_u; s; s &= s - 1) {
        const int x = w * 32 + __ffs(s) - 1;
        bt_union(spar, bt_node_of(sS, r, x), bt_node_of(sS, r - 1, x));
    }
    for (unsigned s = need_l; s; s &= s - 1) {
        const int x = w * 32 + __ffs(s) - 1;
        bt_union(spar, bt_node_of(sS, r, x), bt_node_of(sS, r - 1, x - 1));
    }
    for (unsigned s = need_r; s; s &= s - 1) {
        const int x = w * 32 + __ffs(s) - 1;
        bt_union(spar, bt_node_of(sS, r, x), bt_node_of(sS, r - 1, x + 1));
    }
    __syncthreads();
    // every node: global par entry = global index of its local root; bitmap of the local roots
    unsigned roots = 0u;
    const int gy0 = ty * BT_TH, gx0 = tx * BT_TW;
    int* tp = par + (long long)n * g.P;
    for (unsigned s = S; s; s &= s - 1) {
        const int b = __ffs(s) - 1, node = node0 + b;
        const int root = uf_find(spar, node);
        if (root == node) roots |= 1u << b;
        tp[y * g.W + gx0 + w * 32 + b] = (gy0 + root / BT_TW) * g.W + gx0 + (root & (BT_TW - 1));
    }
    if (live) lbits[wo + (long long)y * g.SEG + seg] = roots;
    if (bad && live) {
        unsigned bw = bad[wo + (long long)y * g.SEG + seg] & m.f;
        while (bw) {                                         // one step per run piece that holds a flagged pixel
            const int b = __ffs(bw) - 1;
            const unsigned rest = ~m.f >> b;
            const int len = rest ? __ffs(rest) - 1 : 32 - b;
            bw = (b + len >= 32) ? 0u : bw & (0xffffffffu << (b + len));
            const int root = uf_find(spar, bt_node_of(sS, r, w * 32 + b));
            low[(long long)n * g.P + (gy0 + root / BT_TW) * g.W + gx0 + (root & (BT_TW - 1))] = 1;
        }
    }
}

// unions across tile edges.  Work items per tile-batch entry: (a) every word of every tile-top row (rows BT_TH * k,
// k >= 1): the vertical / diagonal connections into the tile above, plus run continuations across tile columns;
// (b) for every other row, each inner tile-column boundary: the continuation across it and the two diagonals the tile
// kernel dropped there.
template <int CONN>
__global__ void __launch_bounds__(256)
k_bitccl_border(Geom g, BitPlanes p, int* par) {
    const int tilesX = (g.SEG + BT_TWW - 1) / BT_TWW, tilesY = (g.H + BT_TH - 1) / BT_TH;
    const int nA = (tilesY - 1) * g.SEG, nB = g.H * (tilesX - 1);
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nA + nB) return;
    const int n = blockIdx.y;
    const long long wo = (long long)n * g.H * g.SEG;
    int* tp = par + (long long)n * g.P;
    if (t < nA) {
        const int y = (t / g.SEG + 1) * BT_TH, seg = t - (t / g.SEG) * g.SEG;
        const Masks m = bit_masks(p, g, wo, y, seg);
        if (!m.f) return;
        unsigned need_u = m.eu & ~(m.c & m.el), need_l = 0u, need_r = 0u;
        if (CONN == 2) { need_l = ~m.eu & m.el & ~m.c; need_r = ~m.eu & m.er; }
        for (unsigned s = need_u; s; s &= s - 1) {
            const int x = seg * 32 + __ffs(s) - 1;
            uf_union(tp, bit_node_of(p, g, wo, y, x), bit_node_of(p, g, wo, y - 1, x));
        }
        for (unsigned s = need_l; s; s &= s - 1) {
            const int x = seg * 32 + __ffs(s) - 1;
            uf_union(tp, bit_node_of(p, g, wo, y, x), bit_node_of(p, g, wo, y - 1, x - 1));
        }
        for (unsigned s = need_r; s; s &= s - 1) {
            const int x = seg * 32 + __ffs(s) - 1;
            uf_union(tp, bit_node_of(p, g, wo, y, x), bit_node_of(p, g, wo, y - 1, x + 1));
        }
        return;
    }
    t -= nA;
    const int y = t / (tilesX - 1), j = t - y * (tilesX - 1) + 1;     // boundary between tile columns j-1 and j
    const int segR = j * BT_TWW, xr = segR * 32;                      // first pixel of the right tile
    if (xr >= g.W) return;
    const bool top = y % BT_TH == 0;                                  // (the diagonals of tile-top rows are items (a))
    const Masks mr = bit_masks(p, g, wo, y, segR);
    if (mr.c & 1u) uf_union(tp, y * g.W + xr, bit_node_of(p, g, wo, y, xr - 1));
    if (CONN == 2 && !top && y > 0) {
        if (~mr.eu & mr.el & ~mr.c & 1u) uf_union(tp, y * g.W + xr, bit_node_of(p, g, wo, y - 1, xr - 1));
        const Masks ml = bit_masks(p, g, wo, y, segR - 1);
        if ((~ml.eu & ml.er) >> 31) uf_union(tp, bit_node_of(p, g, wo, y, xr - 1), bit_node_of(p, g, wo, y - 1, xr));
    }
}

// local roots -> final roots (path compression on the way); fbits = bitmap of the final roots
static __global__ void __launch_bounds__(TISEG_THREADS)
k_bitccl_resolve(Geom g, int* par, const unsigned* __restrict__ lbits, unsigned* __restrict__ fbits, uint8_t* low) {
    const long long words = (long long)g.H * g.SEG;
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= words) return;
    const int n = blockIdx.y;
    unsigned m = lbits[(long long)n * words + t], keep = m;
    if (m) {
        const int y = (int)(t / g.SEG), seg = (int)(t - (long long)y * g.SEG);
        int* tp = par + (long long)n * g.P;
        const int idx0 = y * g.W + seg * 32;
        while (m) {
            const int b = __ffs(m) - 1;
            m &= m - 1;
            const int r = idx0 + b, G = uf_find(tp, r);
            if (G != r) {
                tp[r] = G; keep &= ~(1u << b);
                if (low && low[(long long)n * g.P + r]) low[(long long)n * g.P + G] = 1;
            }
        }
    }
    fbits[(long long)n * words + t] = keep;
}

// planes -> forest (par at run starts) + bitmap of the final roots.  lbits / fbits: [g.N, H, SEG] scratch / output.
inline int bitccl_build(tiseg_ctx* c, const Geom& g, const BitPlanes& p, int conn, int* par, unsigned* lbits, unsigned* fbits,
                        const unsigned* bad = nullptr, uint8_t* low = nullptr) {
    const int tilesX = (g.SEG + BT_TWW - 1) / BT_TWW, tilesY = (g.H + BT_TH - 1) / BT_TH;
    const dim3 tg((unsigned)(tilesX * tilesY), (unsigned)g.N);
    const int nb = (tilesY - 1) * g.SEG + g.H * (tilesX - 1);
    const dim3 bg((unsigned)((nb + 255) / 256), (unsigned)g.N);
    if (conn == 2) {
        TISEG_LAUNCH(c, k_bitccl_tile<2>, tg, BT_THREADS, 0, g, p, par, lbits, bad, low);
        if (nb > 0) TISEG_LAUNCH(c, k_bitccl_border<2>, bg, 256, 0, g, p, par);
    } else {
        TISEG_LAUNCH(c, k_bitccl_tile<1>, tg, BT_THREADS, 0, g, p, par, lbits, bad, low);
        if (nb > 0) TISEG_LAUNCH(c, k_bitccl_border<1>, bg, 256, 0, g, p, par);
    }
    const dim3 wg((unsigned)(((long long)g.H * g.SEG + TISEG_THREADS - 1) / TISEG_THREADS), (unsigned)g.N);
    TISEG_LAUNCH(c, k_bitccl_resolve, wg, TISEG_THREADS, 0, g, par, lbits, fbits, low);
    return TISEG_OK;
}
#endif

}  // namespace tiseg
