// Train-time label generation on the GPU (SURVEY.md §8f rank 4), the two targets whose test-time counterparts are the
// DIST and HoVer-Net post-processes:
//   tiseg_gen_hv_map            gen_instance_hv_map (tiseg/datasets/ops/hv_map.py:18-97)
//   tiseg_instance_distance_map the per-instance chessboard distance of DistanceLabelMake.__call__
//                               (tiseg/datasets/ops/distance_map.py:59-110; after its _fix_inst relabelling)
//   tiseg_fix_inst              the _fix_inst every label maker starts with (distance_map.py:41-57, bound_map.py:18-33,
//                               unet_map.py:36-51, direction_map.py:17-32)
//   tiseg_bound_label           BoundLabelMake.__call__ after _fix_inst (bound_map.py:62-88)
// The reference loops over instances, crops a box around each and works on the crop; here per-instance statistics
// (bounding box, coordinate sums, extremes) are accumulated once with atomics into tables dense by instance id, and one
// pass over the pixels evaluates the crop-relative formulas — same integers, same fp32 divisions.
#include "common.cuh"
#include "ccl.cuh"

namespace tiseg {

#define LG_INF 0x3fffffff

struct InstBox {
    int* ymin; int* ymax; int* xmin; int* xmax; int* cnt;       // [N, VM]
    unsigned long long* sy; unsigned long long* sx;             // [N, VM] coordinate sums
    int VM;
};

// The kernels that read a raw ground-truth instance map (gen_instance_hv_map, _fix_inst) are templated on its id type T,
// int32 or uint16 (common.cuh); the maps they produce are int32 either way.
template <class T>
__global__ void __launch_bounds__(TISEG_THREADS)
k_inst_stats(Geom g, const T* __restrict__ inst, InstBox b, int* bad) {
    Pix px;
    if (!warp_pixel(g, px)) return;
    int v = px.ok ? (int)inst[px.base + px.idx] : 0;
    int vl = __shfl_up_sync(0xffffffffu, v, 1);
    bool cont = px.lane > 0 && v == vl;
    unsigned m = __ballot_sync(0xffffffffu, cont);
    if (v != 0 && !cont) {                                       // one set of atomics per in-segment run
        if (v < 0 || v >= b.VM) { *bad = 1; return; }
        const int len = run_end_lane(m, px.lane) - px.lane + 1;
        const long long o = (long long)px.n * b.VM + v;
        atomicMin(&b.ymin[o], px.y); atomicMax(&b.ymax[o], px.y);
        atomicMin(&b.xmin[o], px.x); atomicMax(&b.xmax[o], px.x + len - 1);
        atomicAdd(&b.cnt[o], len);
        atomicAdd(&b.sy[o], (unsigned long long)px.y * len);
        atomicAdd(&b.sx[o], (unsigned long long)(2 * px.x + len - 1) * len / 2);
    }
}
__global__ void k_inst_box_init(InstBox b, int N, int H, int W) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)N * b.VM) return;
    b.ymin[i] = H; b.ymax[i] = -1; b.xmin[i] = W; b.xmax[i] = -1; b.cnt[i] = 0; b.sy[i] = 0ull; b.sx[i] = 0ull;
}

// hv_map.py:36-95 per pixel: crop box = bbox expanded by 2 (clipped); centre of mass of the crop rounded to a pixel;
// x = (col - box_x0 + 1) - com_x; negative side divided by its most negative value, positive side by its largest.
template <class T>
__global__ void __launch_bounds__(TISEG_THREADS)
k_hv_map(Geom g, const T* __restrict__ inst, InstBox b, float2* __restrict__ hv) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    const int v = (int)inst[px.base + px.idx];
    float xv = 0.f, yv = 0.f;
    if (v > 0 && v < b.VM) {
        const long long o = (long long)px.n * b.VM + v;
        const int by0 = max(b.ymin[o] - 2, 0), by1 = min(b.ymax[o] + 1 + 2, g.H);
        const int bx0 = max(b.xmin[o] - 2, 0), bx1 = min(b.xmax[o] + 1 + 2, g.W);
        if (by1 - by0 >= 2 && bx1 - bx0 >= 2) {
            const double cnt = (double)b.cnt[o];
            // scipy.ndimage.center_of_mass on the crop: sum(coordinate * mask) / sum(mask) in float64, then int(. + 0.5)
            const int comy = (int)(((double)(b.sy[o] - (unsigned long long)b.cnt[o] * by0)) / cnt + 0.5);
            const int comx = (int)(((double)(b.sx[o] - (unsigned long long)b.cnt[o] * bx0)) / cnt + 0.5);
            const int xi = (px.x - bx0 + 1) - comx, yi = (px.y - by0 + 1) - comy;
            const int xlo = (b.xmin[o] - bx0 + 1) - comx, xhi = (b.xmax[o] - bx0 + 1) - comx;
            const int ylo = (b.ymin[o] - by0 + 1) - comy, yhi = (b.ymax[o] - by0 + 1) - comy;
            xv = (float)xi; yv = (float)yi;
            if (xi < 0) xv = __fdiv_rn(xv, -(float)xlo); else if (xi > 0) xv = __fdiv_rn(xv, (float)xhi);
            if (yi < 0) yv = __fdiv_rn(yv, -(float)ylo); else if (yi > 0) yv = __fdiv_rn(yv, (float)yhi);
        }
    }
    hv[px.base + px.idx] = make_float2(xv, yv);
}

// ---- per-instance chessboard distance --------------------------------------------------------------------------
// distance_transform_cdt of one instance's crop = chessboard distance to the nearest pixel that is NOT of this
// instance inside the crop; the crop keeps a two-pixel ring of such pixels wherever the image allows, so this is the
// distance to the nearest differently-labelled pixel of the image (-1 for an instance that fills the image).
__global__ void __launch_bounds__(TISEG_THREADS)
k_idm_columns(Geom g, const int32_t* __restrict__ inst, int* __restrict__ col) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, n = blockIdx.y;
    if (x >= g.W) return;
    const int32_t* m = inst + (long long)n * g.P + x;
    int* c = col + (long long)n * g.P + x;
    int d = LG_INF, prev = 0;
    for (int y = 0; y < g.H; ++y) {                      // distance to the nearest pixel above with another label
        const int v = m[(long long)y * g.W];
        if (y > 0 && v != prev) d = 1; else if (d != LG_INF) ++d;
        c[(long long)y * g.W] = d;
        prev = v;
    }
    d = LG_INF;
    for (int y = g.H - 1; y >= 0; --y) {
        const int v = m[(long long)y * g.W];
        if (y < g.H - 1 && v != prev) d = 1; else if (d != LG_INF) ++d;
        if (d < c[(long long)y * g.W]) c[(long long)y * g.W] = d;
        prev = v;
    }
}
__global__ void __launch_bounds__(TISEG_THREADS)
k_idm_rows(Geom g, const int32_t* __restrict__ inst, const int* __restrict__ col, int* __restrict__ dist, int* maxd, int VM) {
    const int y = blockIdx.x, n = blockIdx.y;
    const long long ro = (long long)n * g.P + (long long)y * g.W;
    for (int x = threadIdx.x; x < g.W; x += blockDim.x) {
        const int v = inst[ro + x];
        int best = 0;
        if (v != 0) {
            best = col[ro + x];
            for (int d = 1; d < g.W && d < best; ++d) {
                if (x - d >= 0) { const int gv = inst[ro + x - d] != v ? 0 : col[ro + x - d]; best = min(best, max(d, gv)); }
                if (x + d < g.W) { const int gv = inst[ro + x + d] != v ? 0 : col[ro + x + d]; best = min(best, max(d, gv)); }
            }
            if (best >= LG_INF) best = -1;
            else if (v > 0 && v < VM) atomicMax(&maxd[(long long)n * VM + v], best);
        }
        dist[ro + x] = best;
    }
}
__global__ void __launch_bounds__(TISEG_THREADS)
k_idm_finish(Geom g, const int32_t* __restrict__ inst, const int* __restrict__ dist, const int* __restrict__ maxd, int VM,
             int normalise, float* __restrict__ out) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    const long long i = px.base + px.idx;
    const int v = inst[i];
    float r = 0.f;
    // an instance whose expanded crop is thinner than two pixels is skipped (distance_map.py:85-86): with the
    // two-pixel expansion that only happens when the image itself is
    if (v > 0 && v < VM && g.H >= 2 && g.W >= 2) {
        const int mx = maxd[(long long)px.n * VM + v];
        if (!normalise) r = (float)dist[i];
        else if (mx > 0) r = __fdiv_rn((float)dist[i], (float)mx);         // max <= 0: the instance is skipped (:100-102)
    }
    out[i] = r;
}

// ---- _fix_inst ------------------------------------------------------------------------------------------------
// Per id: remove_small_objects(mask, 5) (4-connected pieces), measure.label (8-connected), ids handed out in
// (id, raster order of the piece) order.  Two equal-value CCL passes do the per-id work for every id at once; the
// new id of a piece = pieces of smaller ids (scan over the id axis) + its raster rank among the pieces of its id + 1.
// The kept map has the id type of the input, so both labellings read the ids at the input's width.
template <class T>
__global__ void __launch_bounds__(TISEG_THREADS)
k_fix_keep(long long total, long long P, const T* __restrict__ inst, const int* __restrict__ par,
           const int* __restrict__ area, T* __restrict__ out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int p = par[i];
    out[i] = (p >= 0 && area[i - i % P + p] >= 5) ? inst[i] : (T)0;
}
// every root: slot within its id, max id per tile
template <class T>
__global__ void __launch_bounds__(TISEG_THREADS)
k_fix_root_slots(Geom g, const T* __restrict__ lab, const int* __restrict__ par, int* cnt, int* slot, int* vmax,
                 int VM, int* bad) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    const long long i = px.base + px.idx;
    if (par[i] != px.idx) return;
    const int v = (int)lab[i];
    if (v < 0 || v >= VM) { *bad = 1; return; }
    slot[i] = atomicAdd(&cnt[(long long)px.n * VM + v], 1);
    atomicMax(&vmax[px.n], v);
}
// exclusive scan of cnt over the id axis, one CTA per tile, 1024 ids per round
__global__ void __launch_bounds__(1024) k_fix_scan(const int* __restrict__ cnt, int* __restrict__ base, const int* __restrict__ vmax, int VM) {
    __shared__ int wsum[32];
    __shared__ int carry;
    const int n = blockIdx.x, lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int top = vmax[n];
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int v0 = 0; v0 <= top; v0 += 1024) {
        const int v = v0 + threadIdx.x;
        const int x = v <= top ? cnt[(long long)n * VM + v] : 0;
        int s = x;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, s, o); if (lane >= o) s += t; }
        if (lane == 31) wsum[w] = s;
        __syncthreads();
        if (w == 0) {
            int t = wsum[lane], u = t;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { int q = __shfl_up_sync(0xffffffffu, u, o); if (lane >= o) u += q; }
            wsum[lane] = u - t;
        }
        __syncthreads();
        const int c0 = carry;
        if (v <= top) base[(long long)n * VM + v] = c0 + wsum[w] + s - x;
        __syncthreads();
        if (threadIdx.x == 1023) carry = c0 + wsum[w] + s;
        __syncthreads();
    }
}
template <class T>
__global__ void __launch_bounds__(TISEG_THREADS)
k_fix_list(Geom g, const T* __restrict__ lab, const int* __restrict__ par, const int* __restrict__ base,
           const int* __restrict__ slot, int* __restrict__ lst, int VM) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    const long long i = px.base + px.idx;
    if (par[i] != px.idx) return;
    lst[px.base + base[(long long)px.n * VM + (int)lab[i]] + slot[i]] = px.idx;
}
template <class T>
__global__ void __launch_bounds__(TISEG_THREADS)
k_fix_newid(Geom g, const T* __restrict__ lab, const int* __restrict__ par, const int* __restrict__ base,
            const int* __restrict__ cnt, const int* __restrict__ lst, int* __restrict__ newid, int VM) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    const long long i = px.base + px.idx;
    if (par[i] != px.idx) return;
    const long long o = (long long)px.n * VM + (int)lab[i];
    const int b = base[o], k = cnt[o];
    int before = 0;
    for (int j = 0; j < k; ++j) before += lst[px.base + b + j] < px.idx;
    newid[i] = b + before + 1;
}

// ---- BoundLabelMake -----------------------------------------------------------------------------------------------
// bound_k = dilation(mask_k, diamond(r0)) & ~erosion(mask_k, diamond(r1)), union over the instances k.  Per pixel p:
// some instance other than p's own lies within L1 distance r0, or (p labelled) some pixel within L1 distance r1 is
// not of p's instance.  Pixels outside the image never count (scipy 'reflect' maps them back inside the diamond).
__global__ void __launch_bounds__(TISEG_THREADS)
k_bound_label(Geom g, const uint8_t* __restrict__ sem, const int32_t* __restrict__ inst, int edge_id, int r0, int r1,
              uint8_t* __restrict__ sem_out, uint8_t* __restrict__ bound_out) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    const long long i = px.base + px.idx;
    const int v = inst[i];
    const uint8_t s = v != 0 ? sem[i] : (uint8_t)0;
    bool edge = false;
    const int R = max(r0, r1);
    for (int dy = -R; dy <= R && !edge; ++dy) {
        const int y = px.y + dy;
        if (y < 0 || y >= g.H) continue;
        const int span = R - abs(dy);
        for (int dx = -span; dx <= span; ++dx) {
            const int x = px.x + dx;
            if (x < 0 || x >= g.W) continue;
            const int q = inst[px.base + (long long)y * g.W + x];
            if (q == v) continue;
            const int l1 = abs(dy) + abs(dx);
            if ((q != 0 && l1 <= r0) || (v != 0 && l1 <= r1)) { edge = true; break; }
        }
    }
    if (sem_out) sem_out[i] = s;
    bound_out[i] = edge ? (uint8_t)edge_id : s;
}

// ---- UNetLabelMake ------------------------------------------------------------------------------------------------
// _remove_1px_boundary (unet_map.py:53-63): erosion of every instance by diamond(1) = a pixel keeps its id iff its
// four in-image neighbours carry the same id.
__global__ void __launch_bounds__(TISEG_THREADS)
k_unet_inner(Geom g, const int32_t* __restrict__ inst, int32_t* __restrict__ inner, uint8_t* seen, int VM, int* bad) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    const long long i = px.base + px.idx;
    const int v = inst[i];
    int o = 0;
    if (v != 0) {
        bool keep = true;
        if (px.x > 0) keep &= inst[i - 1] == v;
        if (px.x + 1 < g.W) keep &= inst[i + 1] == v;
        if (px.y > 0) keep &= inst[i - g.W] == v;
        if (px.y + 1 < g.H) keep &= inst[i + g.W] == v;
        if (keep) {
            o = v;
            if (v < 0 || v >= VM) *bad = 1; else if (!seen[(long long)px.n * VM + v]) seen[(long long)px.n * VM + v] = 1;
        }
    }
    inner[i] = o;
}
__global__ void k_count_seen(const uint8_t* __restrict__ seen, int VM, int* count) {
    int n = blockIdx.y, c = 0;
    for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < VM; v += gridDim.x * blockDim.x) c += seen[(long long)n * VM + v];
    for (int d = 16; d; d >>= 1) c += __shfl_xor_sync(0xffffffffu, c, d);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(&count[n], c);
}
// _get_weight_map (unet_map.py:65-98) needs, per pixel, the Euclidean distances to the nearest and to the second
// nearest INSTANCE.  Per column only the two vertically nearest distinct ids can matter (a third one is farther than
// both from every pixel of the row), so a column sweep leaves (distance, id) x 2 per pixel and a bounded row search
// combines them — the exact squared distances scipy's EDT takes the square root of.
struct Top2 { int g1, l1, g2, l2; };            // vertical distance / id of the nearest and the second nearest id
__device__ __forceinline__ void top2_offer(long long d, int l, long long& d1, int& l1, long long& d2, int& l2) {
    if (l == l1) { if (d < d1) d1 = d; return; }
    if (d < d1) { d2 = d1; l2 = l1; d1 = d; l1 = l; return; }
    if (l == l2) { if (d < d2) d2 = d; return; }
    if (d < d2) { d2 = d; l2 = l; }
}
__global__ void __launch_bounds__(TISEG_THREADS)
k_unet_columns(Geom g, const int32_t* __restrict__ inner, int4* __restrict__ col) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, n = blockIdx.y;
    if (x >= g.W) return;
    const int32_t* m = inner + (long long)n * g.P + x;
    int4* c = col + (long long)n * g.P + x;
    int la = 0, ya = 0, lb = 0, yb = 0;               // last id seen and the id seen before it (distinct), with their rows
    for (int y = 0; y < g.H; ++y) {
        const int v = m[(long long)y * g.W];
        if (v != 0) { if (v != la) { lb = la; yb = ya; la = v; } ya = y; }
        c[(long long)y * g.W] = make_int4(la ? y - ya : LG_INF, la, lb ? y - yb : LG_INF, lb);
    }
    la = lb = 0;
    for (int y = g.H - 1; y >= 0; --y) {
        const int v = m[(long long)y * g.W];
        if (v != 0) { if (v != la) { lb = la; yb = ya; la = v; } ya = y; }
        const int4 t = c[(long long)y * g.W];
        long long d1 = t.y ? t.x : (long long)LG_INF, d2 = t.w ? t.z : (long long)LG_INF;
        int l1 = t.y, l2 = t.w;
        if (la) top2_offer(ya - y, la, d1, l1, d2, l2);
        if (lb) top2_offer(yb - y, lb, d1, l1, d2, l2);
        c[(long long)y * g.W] = make_int4((int)d1, l1, (int)d2, l2);
    }
}
__global__ void __launch_bounds__(TISEG_THREADS)
k_unet_weight(Geom g, const int32_t* __restrict__ inner, const int4* __restrict__ col, const int* __restrict__ count,
              double w0, double sigma, double* __restrict__ wmap) {
    const int y = blockIdx.x, n = blockIdx.y;
    const long long ro = (long long)n * g.P + (long long)y * g.W;
    const bool several = count[n] > 1;
    for (int x = threadIdx.x; x < g.W; x += blockDim.x) {
        double pen = 0.0;
        if (several && inner[ro + x] == 0) {
            const long long INF2 = (long long)LG_INF * LG_INF;
            long long d1 = INF2, d2 = INF2;
            int l1 = 0, l2 = 0;
            for (int dx = 0; dx < g.W && (long long)dx * dx < d2; ++dx) {
#pragma unroll
                for (int sgn = 0; sgn < 2; ++sgn) {
                    if (sgn && dx == 0) continue;
                    const int xx = sgn ? x - dx : x + dx;
                    if (xx < 0 || xx >= g.W) continue;
                    const int4 t = col[ro + xx];
                    if (t.y) top2_offer((long long)dx * dx + (long long)t.x * t.x, t.y, d1, l1, d2, l2);
                    if (t.w) top2_offer((long long)dx * dx + (long long)t.z * t.z, t.w, d1, l1, d2, l2);
                }
            }
            const double n1 = sqrt((double)d1), s2 = sqrt((double)d2);
            // the reference's order of operations: near2 = (d_k - near1 minimised) + near1; ties -> near1
            double n2 = d2 == d1 ? n1 : (s2 - n1) + n1;
            const double pix = n1 + n2;
            const double p = pix / sigma;
            pen = w0 * exp(-(p * p) / 2.0);
        }
        wmap[ro + x] = pen + 1.0;                        // wc is None: uniform class weight (unet_map.py:118-119)
    }
}

template <class T>
static int inst_tables(tiseg_ctx* c, const Geom& g, const T* d_inst, InstBox& b) {
    const int VM = g.P + 1 < (1 << 16) ? (1 << 16) : g.P + 1;
    const size_t n = (size_t)g.N * VM;
    b.VM = VM;
    b.ymin = ws<int>(c, n); b.ymax = ws<int>(c, n); b.xmin = ws<int>(c, n); b.xmax = ws<int>(c, n); b.cnt = ws<int>(c, n);
    b.sy = ws<unsigned long long>(c, n); b.sx = ws<unsigned long long>(c, n);
    if (!b.ymin || !b.ymax || !b.xmin || !b.xmax || !b.cnt || !b.sy || !b.sx) return TISEG_ERR_CUDA;
    TISEG_LAUNCH(c, k_inst_box_init, (unsigned)((n + 255) / 256), 256, 0, b, g.N, g.H, g.W);
    TISEG_LAUNCH_AS(c, TISEG_ID_NAME(T, "k_inst_stats"), k_inst_stats<T>, warp_grid(g), TISEG_THREADS, 0, g, d_inst, b, c->d_err);
    return TISEG_OK;
}

// the int32 / uint16 twins of the C entries below share these bodies
template <class T>
static int gen_hv_map_any(tiseg_ctx* c, const T* inst, int N, int H, int W, float* hv_out) {
    if (!c || !inst || !hv_out) { set_error("tiseg_gen_hv_map: bad argument"); return TISEG_ERR_ARG; }
    Call call(c, "tiseg_gen_hv_map", N, H, W);
    const T* d_inst = call.in(inst, call.total);
    float* d_hv = call.out(hv_out, call.total * 2);
    TISEG_TRY(call.status());
    const Geom& g = call.g;
    InstBox b;
    TISEG_TRY(inst_tables(c, g, d_inst, b));
    TISEG_LAUNCH_AS(c, TISEG_ID_NAME(T, "k_hv_map"), k_hv_map<T>, warp_grid(g), TISEG_THREADS, 0, g, d_inst, b, (float2*)d_hv);
    return call.finish();
}

template <class T>
static int fix_inst_any(tiseg_ctx* c, const T* inst, int N, int H, int W, int32_t* out) {
    if (!c || !inst || !out) { set_error("tiseg_fix_inst: bad argument"); return TISEG_ERR_ARG; }
    Call call(c, "tiseg_fix_inst", N, H, W);
    const Geom& g = call.g;
    const size_t total = call.total;
    const T* d_inst = call.in(inst, total);
    int32_t* d_out = call.out(out, total);
    TISEG_TRY(call.status());
    const int VM = g.P + 1 < (1 << 16) ? (1 << 16) : g.P + 1;
    int* par = ws<int>(c, total); int* aux = ws<int>(c, total); int* lst = ws<int>(c, total);
    T* kept = ws<T>(c, total);
    int* cnt = ws<int>(c, (size_t)N * VM); int* base = ws<int>(c, (size_t)N * VM); int* vmax = ws<int>(c, N);
    if (!par || !aux || !lst || !kept || !cnt || !base || !vmax) return TISEG_ERR_CUDA;
    const unsigned fg = (unsigned)((total + TISEG_THREADS - 1) / TISEG_THREADS);
    // remove_small_objects(inst == id, 5): 4-connected pieces of equal id
    TISEG_TRY(ccl_build(c, g, img_eq(d_inst, 0), 1, par));
    TISEG_TRY(ccl_areas(c, g, par, aux));
    TISEG_LAUNCH_AS(c, TISEG_ID_NAME(T, "k_fix_keep"), k_fix_keep<T>, fg, TISEG_THREADS, 0, (long long)total, (long long)g.P, d_inst, par,
                    aux, kept);
    // measure.label(mask): 8-connected pieces of equal id
    TISEG_TRY(ccl_build(c, g, img_eq((const T*)kept, 0), 2, par));
    TISEG_TRY(zero(c, cnt, (size_t)N * VM * sizeof(int)));
    TISEG_TRY(zero(c, vmax, (size_t)N * sizeof(int)));
    TISEG_LAUNCH_AS(c, TISEG_ID_NAME(T, "k_fix_root_slots"), k_fix_root_slots<T>, warp_grid(g), TISEG_THREADS, 0, g, kept, par, cnt, aux,
                    vmax, VM, c->d_err);
    TISEG_LAUNCH(c, k_fix_scan, N, 1024, 0, cnt, base, vmax, VM);
    TISEG_LAUNCH_AS(c, TISEG_ID_NAME(T, "k_fix_list"), k_fix_list<T>, warp_grid(g), TISEG_THREADS, 0, g, kept, par, base, aux, lst, VM);
    int* newid = ws<int>(c, total);
    if (!newid) return TISEG_ERR_CUDA;
    TISEG_LAUNCH_AS(c, TISEG_ID_NAME(T, "k_fix_newid"), k_fix_newid<T>, warp_grid(g), TISEG_THREADS, 0, g, kept, par, base, cnt, lst, newid,
                    VM);
    TISEG_TRY(apply_rank(c, g, par, newid, d_out));
    return call.finish();
}

}  // namespace tiseg

using namespace tiseg;

extern "C" {

int tiseg_gen_hv_map(tiseg_ctx* c, const int32_t* inst, int N, int H, int W, float* hv_out) {
    return gen_hv_map_any(c, inst, N, H, W, hv_out);
}

int tiseg_gen_hv_map_u16(tiseg_ctx* c, const uint16_t* inst, int N, int H, int W, float* hv_out) {
    return gen_hv_map_any(c, inst, N, H, W, hv_out);
}

int tiseg_instance_distance_map(tiseg_ctx* c, const int32_t* inst, int N, int H, int W, int inst_norm, float* dist_out) {
    if (!c || !inst || !dist_out) { set_error("tiseg_instance_distance_map: bad argument"); return TISEG_ERR_ARG; }
    Call call(c, "tiseg_instance_distance_map", N, H, W);
    const Geom& g = call.g;
    const size_t total = call.total;
    const int32_t* d_inst = call.in(inst, total);
    float* d_out = call.out(dist_out, total);
    TISEG_TRY(call.status());
    const int VM = g.P + 1 < (1 << 16) ? (1 << 16) : g.P + 1;
    int* col = ws<int>(c, total); int* dist = ws<int>(c, total);
    int* maxd = ws<int>(c, (size_t)N * VM);
    if (!col || !dist || !maxd) return TISEG_ERR_CUDA;
    TISEG_TRY(zero(c, maxd, (size_t)N * VM * sizeof(int)));
    TISEG_LAUNCH(c, k_idm_columns, dim3((g.W + TISEG_THREADS - 1) / TISEG_THREADS, N), TISEG_THREADS, 0, g, d_inst, col);
    TISEG_LAUNCH(c, k_idm_rows, dim3(g.H, N), TISEG_THREADS, 0, g, d_inst, col, dist, maxd, VM);
    TISEG_LAUNCH(c, k_idm_finish, warp_grid(g), TISEG_THREADS, 0, g, d_inst, dist, maxd, VM, inst_norm, d_out);
    return call.finish();
}

int tiseg_fix_inst(tiseg_ctx* c, const int32_t* inst, int N, int H, int W, int32_t* out) {
    return fix_inst_any(c, inst, N, H, W, out);
}

int tiseg_fix_inst_u16(tiseg_ctx* c, const uint16_t* inst, int N, int H, int W, int32_t* out) {
    return fix_inst_any(c, inst, N, H, W, out);
}

int tiseg_bound_label(tiseg_ctx* c, const uint8_t* sem, const int32_t* inst, int N, int H, int W, int edge_id,
                      int radius_dilate, int radius_erode, uint8_t* sem_out, uint8_t* sem_w_bound_out) {
    if (!c || !sem || !inst || !sem_w_bound_out || radius_dilate < 0 || radius_erode < 0 || radius_dilate > 64 ||
        radius_erode > 64 || edge_id < 0 || edge_id > 255) {
        set_error("tiseg_bound_label: bad argument");
        return TISEG_ERR_ARG;
    }
    Call call(c, "tiseg_bound_label", N, H, W);
    const uint8_t* d_sem = call.in(sem, call.total);
    const int32_t* d_inst = call.in(inst, call.total);
    uint8_t* d_so = call.out(sem_out, call.total);
    uint8_t* d_bo = call.out(sem_w_bound_out, call.total);
    TISEG_TRY(call.status());
    const Geom& g = call.g;
    TISEG_LAUNCH(c, k_bound_label, warp_grid(g), TISEG_THREADS, 0, g, d_sem, d_inst, edge_id, radius_dilate, radius_erode,
                 d_so, d_bo);
    return call.finish();
}

int tiseg_unet_weight_map(tiseg_ctx* c, const int32_t* inst, int N, int H, int W, double w0, double sigma,
                          int32_t* inner_out, double* wmap_out) {
    if (!c || !inst || !inner_out || !wmap_out || !(sigma > 0)) { set_error("tiseg_unet_weight_map: bad argument"); return TISEG_ERR_ARG; }
    Call call(c, "tiseg_unet_weight_map", N, H, W);
    const Geom& g = call.g;
    const size_t total = call.total;
    const int32_t* d_inst = call.in(inst, total);
    int32_t* d_inner = call.out(inner_out, total);
    double* d_w = call.out(wmap_out, total);
    TISEG_TRY(call.status());
    const int VM = g.P + 1 < (1 << 16) ? (1 << 16) : g.P + 1;
    uint8_t* seen = ws<uint8_t>(c, (size_t)N * VM);
    int* count = ws<int>(c, N);
    int4* col = ws<int4>(c, total);
    if (!seen || !count || !col) return TISEG_ERR_CUDA;
    TISEG_TRY(zero(c, seen, (size_t)N * VM));
    TISEG_TRY(zero(c, count, (size_t)N * sizeof(int)));
    TISEG_LAUNCH(c, k_unet_inner, warp_grid(g), TISEG_THREADS, 0, g, d_inst, d_inner, seen, VM, c->d_err);
    TISEG_LAUNCH(c, k_count_seen, dim3(32, N), 256, 0, seen, VM, count);
    TISEG_LAUNCH(c, k_unet_columns, dim3((g.W + TISEG_THREADS - 1) / TISEG_THREADS, N), TISEG_THREADS, 0, g, d_inner, col);
    TISEG_LAUNCH(c, k_unet_weight, dim3(g.H, N), TISEG_THREADS, 0, g, d_inner, col, count, w0, sigma, d_w);
    return call.finish();
}

}  // extern "C"
