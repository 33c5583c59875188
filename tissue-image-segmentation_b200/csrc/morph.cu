// K2 / K4 + the UNet-family postprocess (A2): fill holes, remove small objects, label dilation / erosion,
// and the per-class loop of unet.py:71-93 and its siblings, all batched over tiles.
#include "ccl.cuh"
#include "morph.cuh"

namespace tiseg {

// ---- fill holes: background components (4-connected) that do not reach the image border ------------
// scipy.ndimage.binary_fill_holes == complement of the border-seeded propagation through ~mask with the
// cross structure.  `par` is the flattened forest of the COMPLEMENT image (par >= 0 <=> background pixel).
__global__ void k_border_touch(Geom g, const int* __restrict__ par, uint8_t* touch) {
    // one thread per border pixel: 2W + 2H per tile
    int n = blockIdx.y;
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    int per = 2 * g.W + 2 * g.H;
    if (i >= per) return;
    int y, x;
    if (i < g.W) { y = 0; x = i; }
    else if (i < 2 * g.W) { y = g.H - 1; x = i - g.W; }
    else if (i < 2 * g.W + g.H) { y = i - 2 * g.W; x = 0; }
    else { y = i - 2 * g.W - g.H; x = g.W - 1; }
    long long base = (long long)n * g.P;
    int p = par[base + y * g.W + x];
    if (p >= 0) touch[base + p] = 1;
}

__global__ void __launch_bounds__(TISEG_THREADS)
k_fill_from_forest(long long P, const int* __restrict__ par, const uint8_t* __restrict__ touch, uint8_t* __restrict__ out,
                   bool vec) {
    const long long base = (long long)blockIdx.y * P, i = flat4_index();
    if (i >= P) return;
    Pack4<int> p = ld4(par + base, i, P, vec);
    Pack4<uint8_t> o;
#pragma unroll
    for (int k = 0; k < 4; ++k) o.v[k] = (uint8_t)((p.v[k] < 0) || (i + k < P && !touch[base + p.v[k]]));
    st4(out + base, i, P, vec, o);
}

int fill_from_complement_forest(tiseg_ctx* c, const Geom& g, const int* par, uint8_t* out) {
    size_t total = (size_t)g.N * g.P;
    uint8_t* touch = ws<uint8_t>(c, total);
    if (!touch) return TISEG_ERR_CUDA;
    TISEG_TRY(zero(c, touch, total));
    int per = 2 * g.W + 2 * g.H;
    TISEG_LAUNCH(c, k_border_touch, dim3((per + 255) / 256, g.N), 256, 0, g, par, touch);
    TISEG_LAUNCH(c, k_fill_from_forest, dim3(flat4_grid(g.P), g.N), TISEG_THREADS, 0, (long long)g.P, par, touch, out,
                 (g.P % 4 == 0) && aligned16(par) && (((uintptr_t)out) & 3) == 0);
    return TISEG_OK;
}

// ---- remove small objects ---------------------------------------------------------------------------
__global__ void __launch_bounds__(TISEG_THREADS)
k_keep_large(long long P, const int* __restrict__ par, const int* __restrict__ area, int min_size, uint8_t* __restrict__ out,
             bool vec) {
    const long long base = (long long)blockIdx.y * P, i = flat4_index();
    if (i >= P) return;
    Pack4<int> p = ld4(par + base, i, P, vec);
    Pack4<uint8_t> o;
#pragma unroll
    for (int k = 0; k < 4; ++k) o.v[k] = (uint8_t)(i + k < P && p.v[k] >= 0 && area[base + p.v[k]] >= min_size);
    st4(out + base, i, P, vec, o);
}

int remove_small_mask(tiseg_ctx* c, const Geom& g, const uint8_t* mask, int min_size, int conn, uint8_t* out) {
    size_t total = (size_t)g.N * g.P;
    int* par = ws<int>(c, total);
    int* area = ws<int>(c, total);
    if (!par || !area) return TISEG_ERR_CUDA;
    TISEG_TRY(ccl_build(c, g, ImgMaskU8{mask}, conn, par));
    TISEG_TRY(ccl_areas(c, g, par, area));
    TISEG_LAUNCH(c, k_keep_large, dim3(flat4_grid(g.P), g.N), TISEG_THREADS, 0, (long long)g.P, par, area, min_size, out,
                 (g.P % 4 == 0) && aligned16(par) && (((uintptr_t)out) & 3) == 0);
    return TISEG_OK;
}

// int input: the label values are the component ids (skimage: bincount of the labels themselves)
__global__ void __launch_bounds__(TISEG_THREADS)
k_label_hist(Geom g, const int32_t* __restrict__ lab, int* hist, int KS, int* bad, bool vec) {
    Quad q;
    if (!warp_quad(g, q)) return;
    int v[4];
    quad_load_i32(g, q, lab + q.base, 0, vec, v);
    if (!__any_sync(0xffffffffu, (v[0] | v[1] | v[2] | v[3]) != 0)) return;                      // (uniform)
    const QuadRuns r = quad_runs(v, 0, q.lane);
    FOR_QUAD_RUNS(r, k, len) {
        if (v[k] < 0 || v[k] >= KS) { *bad = 1; continue; }
        atomicAdd(&hist[(long long)q.n * KS + v[k]], (int)len);
    }
}
__global__ void k_drop_small_labels(Geom g, const int32_t* __restrict__ lab, const int* __restrict__ hist, int KS,
                                    int min_size, int32_t* __restrict__ out) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    int v = lab[px.base + px.idx];
    bool keep = v != 0 && (v < 0 || v >= KS || hist[(long long)px.n * KS + v] >= min_size);
    out[px.base + px.idx] = keep ? v : 0;
}

int remove_small_labels(tiseg_ctx* c, const Geom& g, const int32_t* lab, int min_size, int32_t* out) {
    int KS = g.P + 1;
    int* hist = ws<int>(c, (size_t)g.N * KS);
    int* bad = ws<int>(c, 1);
    if (!hist || !bad) return TISEG_ERR_CUDA;
    TISEG_TRY(zero(c, hist, (size_t)g.N * KS * sizeof(int)));
    TISEG_TRY(zero(c, bad, sizeof(int)));
    TISEG_LAUNCH(c, k_label_hist, quad_grid(g), TISEG_THREADS, 0, g, lab, hist, KS, bad, (g.W % 4 == 0) && aligned16(lab));
    TISEG_LAUNCH(c, k_drop_small_labels, warp_grid(g), TISEG_THREADS, 0, g, lab, hist, KS, min_size, out);
    return TISEG_OK;
}

// ---- label dilation / erosion (grey max / min filter over disk(r) or square(2r+1)) -------------------
template <bool DILATE>
__global__ void __launch_bounds__(TISEG_THREADS)
k_grey_morph(Geom g, const int32_t* __restrict__ lab, int footprint, int r, int32_t* __restrict__ out) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    const int32_t* t = lab + px.base;
    int v = t[px.idx];
    int r2 = r * r;
    for (int dy = -r; dy <= r; ++dy) {
        int yy = px.y + dy;
        if (yy < 0 || yy >= g.H) continue;
        for (int dx = -r; dx <= r; ++dx) {
            int xx = px.x + dx;
            if (xx < 0 || xx >= g.W) continue;
            if (footprint == 0 && dx * dx + dy * dy > r2) continue;
            int u = t[yy * g.W + xx];
            v = DILATE ? max(v, u) : min(v, u);
        }
    }
    out[px.base + px.idx] = v;
}

int grey_morph(tiseg_ctx* c, const Geom& g, const int32_t* lab, int footprint, int radius, bool dilate, int32_t* out) {
    if (dilate) TISEG_LAUNCH(c, k_grey_morph<true>, warp_grid(g), TISEG_THREADS, 0, g, lab, footprint, radius, out);
    else        TISEG_LAUNCH(c, k_grey_morph<false>, warp_grid(g), TISEG_THREADS, 0, g, lab, footprint, radius, out);
    return TISEG_OK;
}

// ---- UNet-family postprocess --------------------------------------------------------------------------
__global__ void k_zero_class(Geom g, uint8_t* cls, int edge_id, const uint8_t* __restrict__ kill) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    long long i = px.base + px.idx;
    if ((edge_id >= 0 && cls[i] == edge_id) || (kill && kill[i] > 0)) cls[i] = 0;
}

__global__ void __launch_bounds__(TISEG_THREADS)
k_class_presence(long long P, const uint8_t* __restrict__ cls, unsigned long long* present, bool vec) {
    const long long base = (long long)blockIdx.y * P;
    unsigned lo = 0, hi = 0;
    for (long long i = flat4_index(); i < P; i += (long long)gridDim.x * blockDim.x * 4) {
        Pack4<uint8_t> v = ld4(cls + base, i, P, vec);
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (i + k < P) { if (v.v[k] < 32) lo |= 1u << v.v[k]; else if (v.v[k] < 64) hi |= 1u << (v.v[k] - 32); }
    }
    lo = __reduce_or_sync(0xffffffffu, lo);
    hi = __reduce_or_sync(0xffffffffu, hi);
    if ((threadIdx.x & 31) == 0) {
        unsigned long long m = ((unsigned long long)hi << 32) | lo;
        if ((present[blockIdx.y] & m) != m) atomicOr(&present[blockIdx.y], m);
    }
}

// dilation(disk(r)) of the class's label image fused with the overwrite into inst / sem (unet.py:86-91).
// One thread = four adjacent pixels: every row of the footprint is read once (four centre values + r on each side)
// instead of once per tap, and threads whose whole window is background — most of them — write nothing.
template <int R>
__global__ void __launch_bounds__(TISEG_THREADS)
k_unet_compose(Geom g, const int32_t* __restrict__ lab, int cls_id, const int* __restrict__ cur, uint8_t* seen, int KS,
               int* haszero, uint8_t* __restrict__ sem, int32_t* __restrict__ inst, bool vec) {
    const int W4 = (g.W + 3) >> 2;
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = t < (long long)W4 * g.H;
    const int n = blockIdx.y;
    int v[4] = {0, 0, 0, 0};
    int y = 0, x = 0;
    if (live) {
        y = (int)(t / W4); x = (int)(t - (long long)y * W4) * 4;
        const int32_t* tl = lab + (long long)n * g.P;
#pragma unroll
        for (int dy = -R; dy <= R; ++dy) {
            const int yy = y + dy;
            if (yy < 0 || yy >= g.H) continue;
            const int32_t* row = tl + (long long)yy * g.W;
            int w[4 + 2 * R];                                   // columns x-R .. x+3+R
            if (vec) { const Pack4<int> c4 = *reinterpret_cast<const Pack4<int>*>(row + x); w[R] = c4.v[0]; w[R + 1] = c4.v[1]; w[R + 2] = c4.v[2]; w[R + 3] = c4.v[3]; }
            else {
#pragma unroll
                for (int k = 0; k < 4; ++k) w[R + k] = x + k < g.W ? row[x + k] : 0;
            }
#pragma unroll
            for (int k = 1; k <= R; ++k) { w[R - k] = x - k >= 0 ? row[x - k] : 0; w[R + 3 + k] = x + 3 + k < g.W ? row[x + 3 + k] : 0; }
#pragma unroll
            for (int k = 0; k < 4; ++k)
#pragma unroll
                for (int dx = -R; dx <= R; ++dx)
                    if (dx * dx + dy * dy <= R * R) v[k] = max(v[k], w[R + k + dx]);
        }
        const long long o = (long long)n * g.P + (long long)y * g.W + x;
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (x + k < g.W && v[k] > 0) {
                inst[o + k] = v[k] + cur[n];
                sem[o + k] = (uint8_t)cls_id;
                seen[(long long)n * KS + v[k]] = 1;
            }
    }
    bool z = false;
#pragma unroll
    for (int k = 0; k < 4; ++k) z |= live && x + k < g.W && v[k] == 0;
    if (__any_sync(0xffffffffu, z) && (threadIdx.x & 31) == 0 && !haszero[n]) haszero[n] = 1;
}

__global__ void k_zero_prefix_u8(uint8_t* a, int KS, const int* __restrict__ counts) {
    int n = blockIdx.y;
    int k = counts[n];
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i <= k; i += gridDim.x * blockDim.x) a[(long long)n * KS + i] = 0;
}

// cur += len(np.unique(dilated + cur)) = surviving labels + (1 if any zero pixel), only for classes present
__global__ void k_unet_advance(const uint8_t* __restrict__ seen, int KS, const int* __restrict__ counts,
                               int* haszero, const unsigned long long* __restrict__ present, int cls_id, int* cur) {
    int n = blockIdx.x;
    int k = counts[n];
    int s = 0;
    for (int i = 1 + threadIdx.x; i <= k; i += blockDim.x) s += seen[(long long)n * KS + i];
    for (int d = 16; d; d >>= 1) s += __shfl_down_sync(0xffffffffu, s, d);
    __shared__ int sh[8];
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
        for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += sh[i];
        if ((present[n] >> cls_id) & 1ull) cur[n] += t + (haszero[n] ? 1 : 0);
        haszero[n] = 0;
    }
}

int postproc_unet_dev(tiseg_ctx* c, const Geom& g, uint8_t* cls, int max_class, int radius, int edge_id,
                      const uint8_t* kill, uint8_t* sem, int32_t* inst) {
    int N = g.N, KS = g.P + 1;
    size_t total = (size_t)N * g.P;
    if (edge_id >= 0 || kill) TISEG_LAUNCH(c, k_zero_class, warp_grid(g), TISEG_THREADS, 0, g, cls, edge_id, kill);
    unsigned long long* present = ws<unsigned long long>(c, (size_t)N);
    int* cur = ws<int>(c, (size_t)N);
    int* haszero = ws<int>(c, (size_t)N);
    int* counts = ws<int>(c, (size_t)N);
    int* par = ws<int>(c, total);
    int* aux = ws<int>(c, total);           // areas, then ranks
    uint8_t* m1 = ws<uint8_t>(c, total);
    uint8_t* m2 = ws<uint8_t>(c, total);
    int32_t* lab = ws<int32_t>(c, total);
    uint8_t* seen = ws<uint8_t>(c, (size_t)N * KS);
    if (!present || !cur || !haszero || !counts || !par || !aux || !m1 || !m2 || !lab || !seen) return TISEG_ERR_CUDA;
    TISEG_TRY(zero(c, present, (size_t)N * sizeof(unsigned long long)));
    TISEG_TRY(zero(c, cur, (size_t)N * sizeof(int)));
    TISEG_TRY(zero(c, haszero, (size_t)N * sizeof(int)));
    TISEG_TRY(zero(c, sem, total));
    TISEG_TRY(zero(c, inst, total * sizeof(int32_t)));
    {
        unsigned gx = flat4_grid(g.P);
        gx = gx > 32 ? (gx + 15) / 16 : gx;                   // ~16 groups per thread
        TISEG_LAUNCH(c, k_class_presence, dim3(gx, N), TISEG_THREADS, 0, (long long)g.P, cls, present,
                     (g.P % 4 == 0) && (((uintptr_t)cls) & 3) == 0);
    }
    for (int id = 1; id <= max_class; ++id) {
        if (id == edge_id) continue;
        // binary_fill_holes(pred == id)
        TISEG_TRY(ccl_build(c, g, ImgNotClassU8{cls, id}, 1, par));
        TISEG_TRY(fill_from_complement_forest(c, g, par, m1));
        // remove_small_objects(., 5): bool input -> 4-connected components
        TISEG_TRY(ccl_build(c, g, ImgMaskU8{m1}, 1, par));
        TISEG_TRY(ccl_areas(c, g, par, aux));
        TISEG_LAUNCH(c, k_keep_large, dim3(flat4_grid(g.P), N), TISEG_THREADS, 0, (long long)g.P, par, aux, 5, m2,
                     (g.P % 4 == 0) && aligned16(par) && (((uintptr_t)m2) & 3) == 0);
        // measure.label (8-connected, raster ids)
        const unsigned* roots;
        TISEG_TRY(ccl_build(c, g, ImgMaskU8{m2}, 2, par, &roots));
        TISEG_TRY(rank_from_bits(c, g, roots, aux, counts));
        TISEG_TRY(apply_rank(c, g, par, aux, lab));
        // dilation(disk(radius)) + overwrite + cur bookkeeping
        TISEG_LAUNCH(c, k_zero_prefix_u8, dim3(8, N), 256, 0, seen, KS, counts);
        {
            const dim3 qg((unsigned)(((long long)((g.W + 3) / 4) * g.H + TISEG_THREADS - 1) / TISEG_THREADS), (unsigned)N);
            const bool v4 = (g.W % 4 == 0) && aligned16(lab);
            switch (radius) {
                case 0: TISEG_LAUNCH(c, k_unet_compose<0>, qg, TISEG_THREADS, 0, g, lab, id, cur, seen, KS, haszero, sem, inst, v4); break;
                case 1: TISEG_LAUNCH(c, k_unet_compose<1>, qg, TISEG_THREADS, 0, g, lab, id, cur, seen, KS, haszero, sem, inst, v4); break;
                case 2: TISEG_LAUNCH(c, k_unet_compose<2>, qg, TISEG_THREADS, 0, g, lab, id, cur, seen, KS, haszero, sem, inst, v4); break;
                default: TISEG_LAUNCH(c, k_unet_compose<3>, qg, TISEG_THREADS, 0, g, lab, id, cur, seen, KS, haszero, sem, inst, v4); break;
            }
        }
        TISEG_LAUNCH(c, k_unet_advance, N, 256, 0, seen, KS, counts, haszero, present, id, cur);
    }
    return TISEG_OK;
}

}  // namespace tiseg

using namespace tiseg;

extern "C" {

int tiseg_fill_holes(tiseg_ctx* c, const uint8_t* mask, int N, int H, int W, uint8_t* out) {
    if (!c || !mask || !out) { set_error("tiseg_fill_holes: bad argument"); return TISEG_ERR_ARG; }
    Call call(c, "tiseg_fill_holes", N, H, W);
    const uint8_t* d_in = call.in(mask, call.total);
    uint8_t* d_out = call.out(out, call.total);
    TISEG_TRY(call.status());
    int* par = ws<int>(c, call.total);
    if (!par) return TISEG_ERR_CUDA;
    TISEG_TRY(ccl_build(c, call.g, ImgNotMaskU8{d_in}, 1, par));
    TISEG_TRY(fill_from_complement_forest(c, call.g, par, d_out));
    return call.finish();
}

int tiseg_remove_small_objects(tiseg_ctx* c, const uint8_t* mask, int N, int H, int W, int min_size, int connectivity,
                               uint8_t* out) {
    if (!c || !mask || !out || (connectivity != 1 && connectivity != 2)) { set_error("tiseg_remove_small_objects: bad argument"); return TISEG_ERR_ARG; }
    Call call(c, "tiseg_remove_small_objects", N, H, W);
    const uint8_t* d_in = call.in(mask, call.total);
    uint8_t* d_out = call.out(out, call.total);
    TISEG_TRY(call.status());
    TISEG_TRY(remove_small_mask(c, call.g, d_in, min_size, connectivity, d_out));
    return call.finish();
}

int tiseg_remove_small_labels(tiseg_ctx* c, const int32_t* lab, int N, int H, int W, int min_size, int32_t* out) {
    if (!c || !lab || !out) { set_error("tiseg_remove_small_labels: bad argument"); return TISEG_ERR_ARG; }
    Call call(c, "tiseg_remove_small_labels", N, H, W);
    const int32_t* d_in = call.in(lab, call.total);
    int32_t* d_out = call.out(out, call.total);
    TISEG_TRY(call.status());
    TISEG_TRY(remove_small_labels(c, call.g, d_in, min_size, d_out));
    return call.finish();
}

static int morph_entry(tiseg_ctx* c, const int32_t* lab, int N, int H, int W, int footprint, int radius, bool dil,
                       int32_t* out) {
    if (!c || !lab || !out || footprint < 0 || footprint > 1 || radius < 0 || radius > 3) { set_error("label morphology: bad argument (radius <= 3)"); return TISEG_ERR_ARG; }
    Call call(c, dil ? "tiseg_dilate_labels" : "tiseg_erode_labels", N, H, W);
    const int32_t* d_in = call.in(lab, call.total);
    int32_t* d_out = call.out(out, call.total);
    TISEG_TRY(call.status());
    if (d_in == d_out) { set_error("label morphology cannot run in place"); return TISEG_ERR_ARG; }
    TISEG_TRY(grey_morph(c, call.g, d_in, footprint, radius, dil, d_out));
    return call.finish();
}
int tiseg_dilate_labels(tiseg_ctx* c, const int32_t* lab, int N, int H, int W, int footprint, int radius, int32_t* out) {
    return morph_entry(c, lab, N, H, W, footprint, radius, true, out);
}
int tiseg_erode_labels(tiseg_ctx* c, const int32_t* lab, int N, int H, int W, int footprint, int radius, int32_t* out) {
    return morph_entry(c, lab, N, H, W, footprint, radius, false, out);
}

int tiseg_postproc_unet(tiseg_ctx* c, uint8_t* cls, int N, int H, int W, int max_class, int radius, int edge_id,
                        const uint8_t* kill, uint8_t* sem_out, int32_t* inst_out) {
    if (!c || !cls || !sem_out || !inst_out || max_class < 1 || max_class > 63 || radius < 0 || radius > 3) {
        set_error("tiseg_postproc_unet: bad argument (1 <= max_class <= 63, radius <= 3)");
        return TISEG_ERR_ARG;
    }
    Call call(c, "tiseg_postproc_unet", N, H, W);
    const size_t total = call.total;
    const bool mutate = edge_id >= 0 || kill;          // then the class map is edited in place (and copied back from host)
    uint8_t* d_cls = mutate ? call.inout(cls, total) : const_cast<uint8_t*>(call.in(cls, total));
    const uint8_t* d_kill = call.in(kill, total);
    uint8_t* d_sem = call.out(sem_out, total);
    int32_t* d_inst = call.out(inst_out, total);
    TISEG_TRY(call.status());
    TISEG_TRY(postproc_unet_dev(c, call.g, d_cls, max_class, radius, edge_id, d_kill, d_sem, d_inst));
    return call.finish();
}

}  // extern "C"
