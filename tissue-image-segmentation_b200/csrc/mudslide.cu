// mudslide_watershed (tiseg/models/utils/postprocess.py:158-181) with its helpers get_graph_degree (:12-28) and
// prepare (:31-120) — CDNet's direction-graph refinement.  No shipped config enables it (if_mudslide = False) and its
// one call site is commented out (cdnet.py:146); it is built because the reference exports it
// (models/utils/__init__.py:3-5).  SURVEY.md §8f rank 3.
//
// Everything but `prepare` is masks and component filters (K2/K3).  `prepare` is an ORDERED breadth-first pass: the
// queue starts with the boundary pixels of the inner mask and the contour pixels in raster order; every round first
// follows each queued pixel's direction pointer, then expands to the 8-neighbours nobody points at, and the first
// visitor of a pixel decides its level and (if it has none) its direction — so the result depends on the queue
// order.  Queued pixels are inner-mask or contour pixels and every step moves to an adjacent inner-mask pixel, so the
// order restricted to one 8-connected component of (inner mask | contour) does not depend on the other components:
// each component is processed sequentially and exactly by one lane with its own FIFO slice, the same decomposition
// as align_foreground (align.cu) and the watershed.
#include "ccl.cuh"
#include "morph.cuh"
#include "watershed.cuh"

namespace tiseg {

#define FULL 0xffffffffu
// (row, col) offset of direction k = 1..8 (postprocess.py:37-38)
__constant__ int c_mdr[9] = {0, 0, -1, -1, -1, 0, 1, 1, 1};
__constant__ int c_mdc[9] = {0, -1, -1, 0, 1, 1, 1, 0, -1};

__global__ void k_mud_binarise(Geom g, const uint8_t* __restrict__ a, uint8_t* __restrict__ out) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    out[px.base + px.idx] = a[px.base + px.idx] != 0;
}
// seg[fore == 0] = 0; contour = fore ^ seg
__global__ void k_mud_masks(Geom g, const uint8_t* __restrict__ segf, const uint8_t* __restrict__ fore, uint8_t* __restrict__ seg,
                            uint8_t* __restrict__ contour) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    const long long i = px.base + px.idx;
    const uint8_t s = segf[i] && fore[i];
    seg[i] = s;
    contour[i] = (fore[i] != 0) != (s != 0);
}
__global__ void k_mud_dir_clean(Geom g, uint8_t* dir, const uint8_t* __restrict__ keep) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    const long long i = px.base + px.idx;
    if (!keep[i]) dir[i] = 0;
}
__global__ void k_mud_xor(Geom g, const uint8_t* __restrict__ a, const uint8_t* __restrict__ b, uint8_t* __restrict__ out) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    const long long i = px.base + px.idx;
    out[i] = (a[i] != 0) != (b[i] != 0);
}
// degree[n] = pixels p with a direction k whose BACKWARD neighbour (p - dir(k)) is n; out = degree > 1
__global__ void k_mud_degree(Geom g, const uint8_t* __restrict__ dir, uint8_t* __restrict__ du) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    const uint8_t* t = dir + px.base;
    int deg = 0;
#pragma unroll
    for (int k = 1; k <= 8; ++k) {
        const int y = px.y + c_mdr[k], x = px.x + c_mdc[k];           // p = n + dir(k)  <=>  n = p - dir(k)
        if (y >= 0 && y < g.H && x >= 0 && x < g.W && t[y * g.W + x] == k) ++deg;
    }
    du[px.base + px.idx] = deg > 1;
}
// seg[degree > 0] = 0 (postprocess.py:50-53)
__global__ void k_mud_cut(Geom g, uint8_t* seg, const uint8_t* __restrict__ du) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    const long long i = px.base + px.idx;
    if (du[i]) seg[i] = 0;
}
// the initial queue membership (:55-72), hfa (:73-78), level = 1, vis = 0 / 1
__global__ void k_mud_init(Geom g, const uint8_t* __restrict__ seg, const uint8_t* __restrict__ contour,
                           const uint8_t* __restrict__ dir, uint8_t* __restrict__ inq, uint8_t* __restrict__ hfa,
                           int* __restrict__ level, int* __restrict__ vis, uint8_t* __restrict__ domain) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    const long long i = px.base + px.idx;
    const uint8_t* ts = seg + px.base;
    const uint8_t* td = dir + px.base;
    bool edge = false, pointed = false;
#pragma unroll
    for (int k = 1; k <= 8; ++k) {
        const int y = px.y + c_mdr[k], x = px.x + c_mdc[k];
        const bool inb = y >= 0 && y < g.H && x >= 0 && x < g.W;
        if (!inb || ts[y * g.W + x] != 1) edge = true;
        // somebody points at me: p = me - dir(k) has direction k
        const int py = px.y - c_mdr[k], pxx = px.x - c_mdc[k];
        if (py >= 0 && py < g.H && pxx >= 0 && pxx < g.W && td[py * g.W + pxx] == k) pointed = true;
    }
    const bool q = (ts[px.idx] == 1 && edge) || contour[i] > 0;
    inq[i] = q;
    hfa[i] = pointed;
    level[i] = 1;
    vis[i] = q ? 1 : 0;
    domain[i] = ts[px.idx] > 0 || contour[i] > 0;
}

__global__ void __launch_bounds__(TISEG_THREADS)
k_mud_bfs(Geom g, const uint8_t* __restrict__ segm, const uint8_t* __restrict__ inqm, const uint8_t* __restrict__ hfam,
          const int* __restrict__ par, BlobInfo b, int* work, int* queue, uint8_t* dirm, int* levelm, int* vism) {
    const int lane = threadIdx.x & 31;
    const int n = blockIdx.y;
    const int B = b.count[n];
    const long long base = (long long)n * g.P, ko = (long long)n * b.KS;
    const uint8_t* seg = segm + base;
    const uint8_t* inq = inqm + base;
    const uint8_t* hfa = hfam + base;
    const int* tp = par + base;
    uint8_t* dir = dirm + base;
    int* level = levelm + base;
    int* vis = vism + base;
    const int W = g.W, H = g.H;
    for (;;) {
        int bid = 0;
        if (lane == 0) bid = atomicAdd(&work[n], 1) + 1;
        bid = __shfl_sync(FULL, bid, 0);
        if (bid > B) break;
        const int root = b.root[ko + bid];
        const int y0 = root / W, y1 = b.ymax[ko + bid], x0 = b.xmin[ko + bid], x1 = b.xmax[ko + bid];
        int* q = queue + base + b.off[ko + bid];
        int tail = 0;
        for (int y = y0; y <= y1; ++y) {                    // the initial queue, in raster order
            for (int xb = x0; xb <= x1; xb += 32) {
                int x = xb + lane;
                bool in = false;
                if (x <= x1) { int idx = y * W + x; in = tp[idx] == root && inq[idx] != 0; }
                unsigned m = __ballot_sync(FULL, in);
                if (in) q[tail + __popc(m & ((1u << lane) - 1))] = y * W + x;
                tail += __popc(m);
            }
        }
        __syncwarp();
        if (lane == 0) {
            int start = 0, end = tail, iter = 1;
            while (end > start) {
                ++iter;
                for (int ix = start; ix < end; ++ix) {      // follow the direction pointers (:88-101)
                    const int pix = q[ix];
                    const int k = dir[pix];
                    if (k == 0) continue;
                    const int r = pix / W + c_mdr[k], cc = pix % W + c_mdc[k];
                    if (r < 0 || r >= H || cc < 0 || cc >= W) continue;
                    const int nb = r * W + cc;
                    if (seg[nb] == 0) continue;
                    if (vis[nb] == 0) { q[tail++] = nb; vis[nb] = iter; }
                    if (vis[nb] == iter) {
                        level[nb] = min(level[nb], level[pix] - 1);
                        if (dir[nb] == 0) dir[nb] = (uint8_t)k;
                    }
                }
                for (int ix = start; ix < end; ++ix) {      // expand to the neighbours nobody points at (:103-117)
                    const int pix = q[ix];
                    const int r0 = pix / W, c0 = pix % W;
                    const int lp = level[pix];
#pragma unroll
                    for (int k = 1; k <= 8; ++k) {
                        const int r = r0 + c_mdr[k], cc = c0 + c_mdc[k];
                        if (r < 0 || r >= H || cc < 0 || cc >= W) continue;
                        const int nb = r * W + cc;
                        if (seg[nb] > 0 && vis[nb] == 0 && hfa[nb] == 0) {
                            q[tail++] = nb; vis[nb] = iter;
                            if (dir[nb] == 0) { dir[nb] = (uint8_t)k; level[nb] = min(level[nb], lp - 1); }
                            if (lp <= -1) level[nb] = min(level[nb], lp);
                        }
                    }
                }
                start = end;
                end = tail;
            }
        }
        __syncwarp();
    }
}

__global__ void k_mud_levels_out(Geom g, const int* __restrict__ level, uint8_t* __restrict__ pred0, uint8_t* __restrict__ boundary) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    const long long i = px.base + px.idx;
    pred0[i] = level[i] <= 0;
    boundary[i] = level[i] > 0;
}

}  // namespace tiseg

using namespace tiseg;

extern "C" int tiseg_mudslide_watershed(tiseg_ctx* c, const uint8_t* seg, uint8_t* dir_graph, const uint8_t* fore, int N, int H,
                                        int W, uint8_t* pred_out, uint8_t* boundary_out) {
    if (!c || !seg || !dir_graph || !fore || !pred_out || !boundary_out) { set_error("tiseg_mudslide_watershed: bad argument"); return TISEG_ERR_ARG; }
    Call call(c, "tiseg_mudslide_watershed", N, H, W);
    const Geom& g = call.g;
    const size_t total = call.total;
    const uint8_t* d_seg = call.in(seg, total);
    uint8_t* d_dir = call.inout(dir_graph, total);
    const uint8_t* d_fore = call.in(fore, total);
    uint8_t* d_pred = call.out(pred_out, total);
    uint8_t* d_bnd = call.out(boundary_out, total);
    TISEG_TRY(call.status());
    uint8_t* m[10];
    for (auto& p : m) { p = ws<uint8_t>(c, total); if (!p) return TISEG_ERR_CUDA; }
    int* par = ws<int>(c, total); int* rank = ws<int>(c, total);
    int* level = ws<int>(c, total); int* vis = ws<int>(c, total); int* queue = ws<int>(c, total);
    int* work = ws<int>(c, (size_t)N);
    if (!par || !rank || !level || !vis || !queue || !work) return TISEG_ERR_CUDA;
    uint8_t *segb = m[0], *segf = m[1], *foref = m[2], *forec = m[3], *segc = m[4], *contour = m[5], *small = m[6], *du = m[7], *tmp = m[8], *aux = m[9];
    // seg = fill_holes(seg); fore = remove_small_objects(fill_holes(fore), 20); seg[fore == 0] = 0; contour = fore ^ seg
    TISEG_LAUNCH(c, k_mud_binarise, warp_grid(g), TISEG_THREADS, 0, g, d_seg, segb);
    TISEG_TRY(ccl_build(c, g, ImgNotMaskU8{segb}, 1, par));
    TISEG_TRY(fill_from_complement_forest(c, g, par, segf));
    TISEG_LAUNCH(c, k_mud_binarise, warp_grid(g), TISEG_THREADS, 0, g, d_fore, tmp);
    TISEG_TRY(ccl_build(c, g, ImgNotMaskU8{tmp}, 1, par));
    TISEG_TRY(fill_from_complement_forest(c, g, par, foref));
    TISEG_TRY(remove_small_mask(c, g, foref, 20, 1, forec));
    TISEG_LAUNCH(c, k_mud_masks, warp_grid(g), TISEG_THREADS, 0, g, segf, forec, segc, contour);
    // dir_graph[remove_small_objects(dir_graph > 0, 20) == 0] = 0
    TISEG_LAUNCH(c, k_mud_binarise, warp_grid(g), TISEG_THREADS, 0, g, (const uint8_t*)d_dir, tmp);
    TISEG_TRY(remove_small_mask(c, g, tmp, 20, 1, aux));
    TISEG_LAUNCH(c, k_mud_dir_clean, warp_grid(g), TISEG_THREADS, 0, g, d_dir, aux);
    // small_area = remove_small_objects(seg, 60) ^ seg
    TISEG_TRY(remove_small_mask(c, g, segc, 60, 1, tmp));
    TISEG_LAUNCH(c, k_mud_xor, warp_grid(g), TISEG_THREADS, 0, g, tmp, segc, small);
    // du = remove_small_objects(get_graph_degree(dir_graph) > 1, 3)
    TISEG_LAUNCH(c, k_mud_degree, warp_grid(g), TISEG_THREADS, 0, g, (const uint8_t*)d_dir, tmp);
    TISEG_TRY(remove_small_mask(c, g, tmp, 3, 1, du));
    // prepare
    TISEG_LAUNCH(c, k_mud_cut, warp_grid(g), TISEG_THREADS, 0, g, segc, du);
    uint8_t *inq = tmp, *hfa = aux, *domain = segb;
    TISEG_LAUNCH(c, k_mud_init, warp_grid(g), TISEG_THREADS, 0, g, segc, contour, (const uint8_t*)d_dir, inq, hfa, level, vis, domain);
    BlobInfo b;
    TISEG_TRY(blobs_build(c, g, ImgMaskU8{domain}, par, rank, b, true, 2));
    TISEG_TRY(zero(c, work, (size_t)N * sizeof(int)));
    int per_tile = (c->sm_count * 8 * 4 + N - 1) / N;
    per_tile = per_tile < 1 ? 1 : (per_tile > 512 ? 512 : per_tile);
    TISEG_LAUNCH(c, k_mud_bfs, dim3(per_tile, N), TISEG_THREADS, 0, g, segc, inq, hfa, par, b, work, queue, d_dir, level, vis);
    // pred = remove_small_objects(level <= 0, 15, connectivity=1) ^ small_area; boundary = level > 0
    TISEG_LAUNCH(c, k_mud_levels_out, warp_grid(g), TISEG_THREADS, 0, g, level, segf, d_bnd);
    TISEG_TRY(remove_small_mask(c, g, segf, 15, 1, foref));
    TISEG_LAUNCH(c, k_mud_xor, warp_grid(g), TISEG_THREADS, 0, g, foref, small, d_pred);
    return call.finish();
}
