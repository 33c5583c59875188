// K3 — connected-component labelling entry points (tiseg_label*, tiseg_re_instance) and the
// non-template parts of the CCL toolbox declared in ccl.cuh.
#include <cooperative_groups.h>
#include "ccl.cuh"

namespace tiseg {

// every foreground pixel points directly at its root; bits[n, y, seg] (zeroed beforehand) gets the bit of every root.
// Four pixels per thread (one 128-bit load / store; the pixels of a run share one chase): a pixel-per-lane version of
// this pass was issue-bound at a quarter of the HBM rate (profiles/r1_flatten_*).
template <bool LISTED>
__global__ void __launch_bounds__(TISEG_THREADS) k_ccl_flatten(Geom g, int* par, unsigned* bits, bool vec) {
    const int W4 = (g.W + 3) >> 2;
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (long long)W4 * g.H) return;
    const int y = (int)(t / W4), x = (int)(t - (long long)y * W4) * 4, idx = y * g.W + x;
    FOR_TILES(LISTED, g, n) {
    int* tp = par + (long long)n * g.P;
    int p[4], a[4];
    if (vec) {
        const int4 v = *reinterpret_cast<const int4*>(tp + idx);
        p[0] = v.x; p[1] = v.y; p[2] = v.z; p[3] = v.w;
    } else {
#pragma unroll
        for (int k = 0; k < 4; ++k) p[k] = x + k < g.W ? tp[idx + k] : -1;
    }
    int q[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) q[k] = p[k] >= 0 ? tp[p[k]] : -1;           // second hops, independent
    bool changed = false;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        a[k] = p[k];
        if (p[k] < 0) continue;
        if (k > 0 && p[k] == p[k - 1]) a[k] = a[k - 1];
        else {
            int r = p[k], nx = q[k];
            while (nx != r) { r = nx; nx = tp[r]; }
            a[k] = r;
        }
        changed |= a[k] != p[k];
        if (a[k] == idx + k) atomicOr(&bits[((long long)n * g.H + y) * g.SEG + ((x + k) >> 5)], 1u << ((x + k) & 31));
    }
    if (changed) {
        if (vec) *reinterpret_cast<int4*>(tp + idx) = make_int4(a[0], a[1], a[2], a[3]);
        else {
#pragma unroll
            for (int k = 0; k < 4; ++k) if (x + k < g.W && a[k] != p[k]) tp[idx + k] = a[k];
        }
    }
    }
}

// out = par >= 0 ? rank[par] : 0, four pixels per thread
template <bool LISTED>
__global__ void __launch_bounds__(TISEG_THREADS)
k_apply_rank(Geom g, const int* __restrict__ par, const int* __restrict__ rank, int32_t* __restrict__ out, bool vec) {
    const long long P = g.P, i = flat4_index();
    if (i >= P) return;
    FOR_TILES(LISTED, g, n) {
        const long long base = (long long)n * P;
        Pack4<int> p = ld4(par + base, i, P, vec), o;
#pragma unroll
        for (int k = 0; k < 4; ++k) o.v[k] = (i + k < P && p.v[k] >= 0) ? rank[base + p.v[k]] : 0;
        st4(out + base, i, P, vec, o);
    }
}

// area[root] += length of each run of pixels sharing the root (one atomic per run of the warp's 128 pixels)
__global__ void __launch_bounds__(TISEG_THREADS) k_ccl_areas(Geom g, const int* __restrict__ par, int* area, bool vec) {
    Quad q;
    if (!warp_quad(g, q)) return;
    int p[4];
    quad_load_i32(g, q, par + q.base, -1, vec, p);
    if (!__any_sync(0xffffffffu, p[0] >= 0 || p[1] >= 0 || p[2] >= 0 || p[3] >= 0)) return;      // (uniform)
    const QuadRuns r = quad_runs(p, -1, q.lane);
    FOR_QUAD_RUNS(r, k, len) atomicAdd(&area[q.base + p[k]], (int)len);
}

int ccl_flatten(tiseg_ctx* c, const Geom& g, int* par) {
    unsigned* bits = ws<unsigned>(c, (size_t)g.N * g.H * g.SEG);
    if (!bits) return TISEG_ERR_CUDA;
    TISEG_TRY(zero(c, bits, (size_t)g.N * g.H * g.SEG * sizeof(unsigned)));
    const dim3 qg((unsigned)(((long long)((g.W + 3) / 4) * g.H + TISEG_THREADS - 1) / TISEG_THREADS), grid_tiles(g));
    TISEG_LAUNCH_TILES(c, k_ccl_flatten, g, qg, TISEG_THREADS, 0, g, par, bits, (g.W % 4 == 0) && aligned16(par));
    c->rootblk_par = par;             // rank_roots on this forest can skip its bitmap pass
    c->rootblk = (int*)bits;
    return TISEG_OK;
}

// rank[n, pixel] = 1-based raster rank of each set bit of bits[n] (written at the set bits only); counts[n] = set bits
// (may be null).  A tile belongs to a thread-block CLUSTER of RF_CTAS 1024-thread CTAs (a tile per CTA left 84 of the 148
// SMs idle on a 64-tile batch): every CTA ranks a quarter of the rows — row totals (one warp per row, four rows of loads
// in flight), block scan over its rows, placement (one warp per row: warp scan over the row's words, one store per set
// bit) — and the CTAs exchange their totals through distributed shared memory: the ranks of CTA r start after the set
// bits of CTAs 0 .. r-1.  The bitmap of a tile is P / 8 bytes (125 KB at 1000^2): the second read comes from L1 / L2.
#define RF_ROWS 4096                    // rows scanned per round (4 per thread)
#define RF_CTAS 4
template <bool LISTED>
__global__ void __cluster_dims__(RF_CTAS, 1, 1) __launch_bounds__(1024, 2)
k_rank_fused(Geom g, const unsigned* __restrict__ bits, int* __restrict__ rank, int* counts) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    __shared__ int srow[RF_ROWS];
    __shared__ int wsum[32];
    __shared__ int s_carry;
    __shared__ int s_total;             // set bits of this CTA's rows (read by the other CTAs of the cluster)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int cr = (int)cluster.block_rank();
    const int ya = (int)((long long)g.H * cr / RF_CTAS), yb = (int)((long long)g.H * (cr + 1) / RF_CTAS);     // this CTA's rows
    FOR_TILES_OF(LISTED, g, (int)(blockIdx.x / RF_CTAS), n) {
    const unsigned* B = bits + (long long)n * g.H * g.SEG;
    int* out = rank + (long long)n * g.P;
    // set bits of the own rows -> the start of the own ranks
    {
        int t = 0;
        for (long long k = (long long)ya * g.SEG + threadIdx.x; k < (long long)yb * g.SEG; k += 1024) t += __popc(B[k]);
#pragma unroll
        for (int d = 16; d; d >>= 1) t += __shfl_xor_sync(0xffffffffu, t, d);
        if (lane == 0) wsum[warp] = t;
        __syncthreads();
        if (warp == 0) {
            int w = wsum[lane];
#pragma unroll
            for (int d = 16; d; d >>= 1) w += __shfl_xor_sync(0xffffffffu, w, d);
            if (lane == 0) s_total = w;
        }
    }
    cluster.sync();
    if (threadIdx.x == 0) {
        int before = 0, all = 0;
        for (int r = 0; r < RF_CTAS; ++r) {
            const int t = *cluster.map_shared_rank(&s_total, r);
            if (r < cr) before += t;
            all += t;
        }
        s_carry = before;
        if (cr == 0 && counts) counts[n] = all;
    }
    cluster.sync();                     // (nobody rewrites s_total, or leaves, while it is being read)
    for (int base = ya; base < yb; base += RF_ROWS) {
        const int rows = min(RF_ROWS, yb - base);
        // row totals
        for (int r0 = warp; r0 < rows; r0 += 128) {
            int v[4] = {0, 0, 0, 0};
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int r = r0 + 32 * u;
                if (r < rows) for (int k = lane; k < g.SEG; k += 32) v[u] += __popc(B[(long long)(base + r) * g.SEG + k]);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                v[u] = (int)__reduce_add_sync(0xffffffffu, (unsigned)v[u]);
                if (lane == 0 && r0 + 32 * u < rows) srow[r0 + 32 * u] = v[u];
            }
        }
        __syncthreads();
        // exclusive scan of the row totals (four rows per thread)
        int a[4], tot = 0;
#pragma unroll
        for (int u = 0; u < 4; ++u) { const int r = threadIdx.x * 4 + u; a[u] = r < rows ? srow[r] : 0; tot += a[u]; }
        int incl = tot;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += t; }
        if (lane == 31) wsum[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            const int w = wsum[lane];
            int wi = w;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { const int t = __shfl_up_sync(0xffffffffu, wi, d); if (lane >= d) wi += t; }
            wsum[lane] = wi - w;
        }
        __syncthreads();
        const int c0 = s_carry;
        int run = c0 + wsum[warp] + incl - tot;
#pragma unroll
        for (int u = 0; u < 4; ++u) { const int r = threadIdx.x * 4 + u; if (r < rows) srow[r] = run; run += a[u]; }
        __syncthreads();
        if (threadIdx.x == 1023) s_carry = run;
        // placement: one warp per row, four rows of loads in flight
        for (int r0 = warp; r0 < rows; r0 += 128) {
            int pre[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) pre[u] = r0 + 32 * u < rows ? srow[r0 + 32 * u] : 0;
            for (int k0 = 0; k0 < g.SEG; k0 += 32) {
                const int seg = k0 + lane;
                unsigned m[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int r = r0 + 32 * u;
                    m[u] = (r < rows && seg < g.SEG) ? B[(long long)(base + r) * g.SEG + seg] : 0u;
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int r = r0 + 32 * u;
                    if (r >= rows) break;                            // (uniform)
                    if (!__any_sync(0xffffffffu, m[u] != 0u)) continue;  // (uniform) nothing to place in this piece of the row
                    int inc = __popc(m[u]);
#pragma unroll
                    for (int d = 1; d < 32; d <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += t; }
                    int k = pre[u] + inc - __popc(m[u]);
                    int* dst = out + (long long)(base + r) * g.W + seg * 32;
                    for (unsigned q = m[u]; q; q &= q - 1) dst[__ffs(q) - 1] = ++k;
                    pre[u] += __shfl_sync(0xffffffffu, inc, 31);
                }
            }
        }
        __syncthreads();
    }
    }
}

int rank_from_bits(tiseg_ctx* c, const Geom& g, const unsigned* bits, int* rank, int* counts) {
    TISEG_LAUNCH_TILES(c, k_rank_fused, g, grid_tiles(g) * RF_CTAS, 1024, 0, g, bits, rank, counts);
    return TISEG_OK;
}

int rank_roots(tiseg_ctx* c, const Geom& g, const int* par, int* rank, int* counts) {
    if (c->rootblk_par == par && c->rootblk) {
        // the flatten pass already left the bitmap of the roots
        const unsigned* bits = (const unsigned*)c->rootblk;
        c->rootblk_par = nullptr;
        return rank_from_bits(c, g, bits, rank, counts);
    }
    return rank_generic(c, g, SelRoot{par}, rank, counts);
}

int apply_rank(tiseg_ctx* c, const Geom& g, const int* par, const int* rank, int32_t* out) {
    const long long P = g.P;
    const bool vec = (P % 4 == 0) && aligned16(par, out);
    TISEG_LAUNCH_TILES(c, k_apply_rank, g, dim3(flat4_grid(P), grid_tiles(g)), TISEG_THREADS, 0, g, par, rank, out, vec);
    return TISEG_OK;
}

int ccl_areas(tiseg_ctx* c, const Geom& g, const int* par, int* area) {
    TISEG_TRY(zero(c, area, (size_t)g.N * g.P * sizeof(int)));
    TISEG_LAUNCH(c, k_ccl_areas, quad_grid(g), TISEG_THREADS, 0, g, par, area, (g.W % 4 == 0) && aligned16(par));
    return TISEG_OK;
}

// ---- re_instance: ranks of the distinct non-zero values (instance_semantic.py:5-15) -----------------
// first[n, v] = 1 if value v occurs; rank over the value axis.  Values must be < vmax.
__global__ void k_mark_values(Geom g, const int32_t* __restrict__ img, uint8_t* seen, int vmax, int* bad) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    int v = img[px.base + px.idx];
    if (v == 0) return;
    if (v < 0 || v >= vmax) { *bad = 1; return; }
    seen[(long long)px.n * vmax + v] = 1;
}
__global__ void k_lookup_values(Geom g, const int32_t* __restrict__ img, const int* __restrict__ vr, int vmax,
                                int32_t* __restrict__ out) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    int v = img[px.base + px.idx];
    out[px.base + px.idx] = (v > 0 && v < vmax) ? vr[(long long)px.n * vmax + v] : 0;
}

}  // namespace tiseg

using namespace tiseg;

extern "C" {

int tiseg_label(tiseg_ctx* c, const int32_t* img, int N, int H, int W, int32_t background, int connectivity,
                int32_t* out, int32_t* count) {
    if (!c || !img || !out || (connectivity != 1 && connectivity != 2)) { set_error("tiseg_label: bad argument"); return TISEG_ERR_ARG; }
    TISEG_TRY(check_geom(N, H, W));
    begin_call(c);
    Geom g = make_geom(N, H, W);
    size_t total = (size_t)N * g.P;
    const int32_t* d_img = in(c, img, total);
    int32_t* d_out = tiseg::out(c, out, total);
    int32_t* d_cnt = count ? tiseg::out(c, count, (size_t)N) : nullptr;
    if (!d_img || !d_out) return TISEG_ERR_CUDA;
    TISEG_TRY(ccl_label(c, g, ImgEqI32{d_img, background}, connectivity, d_out, d_cnt));
    return end_call(c);
}

int tiseg_label_u8(tiseg_ctx* c, const uint8_t* img, int N, int H, int W, int32_t background, int connectivity,
                   int32_t* out, int32_t* count) {
    if (!c || !img || !out || (connectivity != 1 && connectivity != 2)) { set_error("tiseg_label_u8: bad argument"); return TISEG_ERR_ARG; }
    TISEG_TRY(check_geom(N, H, W));
    begin_call(c);
    Geom g = make_geom(N, H, W);
    size_t total = (size_t)N * g.P;
    const uint8_t* d_img = in(c, img, total);
    int32_t* d_out = tiseg::out(c, out, total);
    int32_t* d_cnt = count ? tiseg::out(c, count, (size_t)N) : nullptr;
    if (!d_img || !d_out) return TISEG_ERR_CUDA;
    TISEG_TRY(ccl_label(c, g, ImgEqU8{d_img, background}, connectivity, d_out, d_cnt));
    return end_call(c);
}

int tiseg_re_instance(tiseg_ctx* c, const int32_t* img, int N, int H, int W, int32_t* out, int32_t* count) {
    if (!c || !img || !out) { set_error("tiseg_re_instance: bad argument"); return TISEG_ERR_ARG; }
    TISEG_TRY(check_geom(N, H, W));
    begin_call(c);
    Geom g = make_geom(N, H, W);
    size_t total = (size_t)N * g.P;
    const int32_t* d_img = in(c, img, total);
    int32_t* d_out = tiseg::out(c, out, total);
    int32_t* d_cnt = count ? tiseg::out(c, count, (size_t)N) : nullptr;
    if (!d_img || !d_out) return TISEG_ERR_CUDA;
    // value axis: ids are bounded by a generous multiple of the pixel count (instance ids never exceed it
    // in the reference's datasets); larger ids are reported as an argument error rather than mis-ranked
    int vmax = g.P + 1 < (1 << 16) ? (1 << 16) : g.P + 1;
    vmax = (vmax + 1023) / 1024 * 1024;          // the value axis is ranked as a [vmax / 1024, 1024] raster
    uint8_t* seen = ws<uint8_t>(c, (size_t)N * vmax);
    int* vr = ws<int>(c, (size_t)N * vmax);
    int* bad = c->d_err;                 // deferred: reported by this call if it synchronises, else by the next that does
    if (!seen || !vr) return TISEG_ERR_CUDA;
    TISEG_TRY(zero(c, seen, (size_t)N * vmax));
    TISEG_LAUNCH(c, k_mark_values, warp_grid(g), TISEG_THREADS, 0, g, d_img, seen, vmax, bad);
    // rank over the value axis: reuse the raster-rank machinery on a [N, vmax / 1024, 1024] "image"
    Geom gv = make_geom(N, vmax / 1024, 1024);
    TISEG_TRY(rank_generic(c, gv, SelFlagU8{seen}, vr, d_cnt));
    TISEG_LAUNCH(c, k_lookup_values, warp_grid(g), TISEG_THREADS, 0, g, d_img, vr, vmax, d_out);
    return end_call(c);
}

}  // extern "C"
