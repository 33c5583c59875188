// Train-time label generation, SURVEY §8f rank 4: DirectionLabelMake (tiseg/datasets/ops/direction_map.py:36-193) after its
// _fix_inst, for to_center = True (the default every config uses).
//   tiseg_direction_labels   dist_gt, point_gt, dir_gt, reg_dir_gt, loss_weight_map of a batch of fixed instance maps
// The reference loops over the instances of a tile on the host: per instance a numba search for the "centerness" point
// (center_calculation.py:8-54: eight binary searches of 24 steps per PIXEL), a distance-to-centre map, an 11x11 torch
// conv2d on the single-instance map, then whole-tile numpy.  Here every step is one pass over the pixels of the batch with
// per-instance state in tables dense by id:
//   k_dl_centerness   centerness of every instance pixel (float64, the numba arithmetic), atomicMax per instance
//   k_dl_center_pick  first raster pixel that reaches the maximum (the reference keeps the first: strict >)
//   k_dl_maxdist      largest distance to the centre per instance
//   k_dl_dist         (1 - d / (max + 1e-7)) in float64 -> float32 map; dist_gt = sqrt(map) * 10; the impulses of point_gt
//   k_dl_direction    the 11x11 correlation restricted to the pixel's own instance (the reference convolves the
//                     single-instance map), angle, direction class, regression angle
//   k_dl_gauss<AXIS>  scipy.ndimage.gaussian_filter(sigma = 2) of the impulses: two 1-D passes in scipy's own
//                     accumulation order (symmetric branch of NI_Correlate1D), float32 between the passes
//   k_dl_weight       loss_weight_map (num_angles == 8): dilation(dd * (10 - dist), disk(1)) * 2 + 1
// Integer / float64-derived outputs (centres, dist_gt, point_gt) reproduce the reference bit for bit; the gradient is a
// float32 sum of 121 products whose order in the reference is the convolution backend's, so the angle — and the class
// where the angle sits on a bin edge — is pinned to float tolerance (tests/test_gpu_ops.py).
#include <cmath>

#include "common.cuh"

namespace tiseg {

int ddm_dev(tiseg_ctx* c, const Geom& g, const uint8_t* dir_map, int T, float* dd);      // cdnet.cu

struct DlTab {
    unsigned long long* best;      // [N, VM] bits of the largest centerness (positive doubles order like integers)
    int* center;                   // [N, VM] flat index of the centre
    unsigned long long* maxd;      // [N, VM] bits of the largest distance to the centre
    int VM;
};
struct DlDirs { double s[8], c[8]; };      // (sin, cos)(2 pi / 8 * i), evaluated on the host like the reference does

__global__ void k_dl_init(DlTab t, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    t.best[i] = 0ull; t.center[i] = 0x7fffffff; t.maxd[i] = 0ull;
}

// center_calculation.py:27-53
__global__ void __launch_bounds__(TISEG_THREADS)
k_dl_centerness(Geom g, const int32_t* __restrict__ inst, DlDirs d, double* __restrict__ cent, DlTab t, int* bad) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    const int32_t* tile = inst + px.base;
    const int v = tile[px.idx];
    if (v == 0) return;
    if (v < 0 || v >= t.VM) { *bad = 1; return; }
    const int H = g.H, W = g.W;
    const double fi = (double)px.y, fj = (double)px.x;
    double max_d = 0.0, min_d = 10000000.0;
#pragma unroll 1
    for (int k = 0; k < 8; ++k) {
        double lo = 0.0, hi = 1000000.0;
        while (fabs(lo - hi) > 0.1) {
            const double mid = (lo + hi) / 2;
            const double xo = rint(__dadd_rn(fi, __dmul_rn(d.s[k], mid))), yo = rint(__dadd_rn(fj, __dmul_rn(d.c[k], mid)));
            bool in = xo >= 0.0 && yo < (double)W && yo >= 0.0 && xo < (double)H;
            if (in) in = tile[(int)xo * W + (int)yo] == v;
            if (in) lo = mid; else hi = mid;
        }
        max_d = fmax(max_d, hi);
        min_d = fmin(min_d, lo);
    }
    const double c = min_d / max_d;
    cent[px.base + px.idx] = c;
    atomicMax(&t.best[(long long)px.n * t.VM + v], (unsigned long long)__double_as_longlong(c));
}
__global__ void __launch_bounds__(TISEG_THREADS)
k_dl_center_pick(Geom g, const int32_t* __restrict__ inst, const double* __restrict__ cent, DlTab t) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    const int v = inst[px.base + px.idx];
    if (v <= 0 || v >= t.VM) return;
    const long long o = (long long)px.n * t.VM + v;
    if ((unsigned long long)__double_as_longlong(cent[px.base + px.idx]) == t.best[o]) atomicMin(&t.center[o], px.idx);
}
__device__ __forceinline__ double dl_dist_to(int idx, int W, int y, int x) {
    const int cy = idx / W, cx = idx - cy * W;
    const long long dy = y - cy, dx = x - cx;
    return sqrt((double)(dy * dy + dx * dx));           // scipy's EDT of a single point: the correctly rounded root
}
__global__ void __launch_bounds__(TISEG_THREADS)
k_dl_maxdist(Geom g, const int32_t* __restrict__ inst, DlTab t) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    const int v = inst[px.base + px.idx];
    if (v <= 0 || v >= t.VM) return;
    const long long o = (long long)px.n * t.VM + v;
    atomicMax(&t.maxd[o], (unsigned long long)__double_as_longlong(dl_dist_to(t.center[o], g.W, px.y, px.x)));
}
// direction_map.py:159-170, 147-151
__global__ void __launch_bounds__(TISEG_THREADS)
k_dl_dist(Geom g, const int32_t* __restrict__ inst, DlTab t, float* __restrict__ dmap, float* __restrict__ dist_out,
          float* __restrict__ impulse) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    const int v = inst[px.base + px.idx];
    float m = 0.f, pt = 0.f;
    if (v > 0 && v < t.VM) {
        const long long o = (long long)px.n * t.VM + v;
        const double dd = dl_dist_to(t.center[o], g.W, px.y, px.x);
        const double mx = __longlong_as_double((long long)t.maxd[o]);
        m = (float)(1.0 - dd / (mx + 0.0000001));       // (float32 map += float64 instance map)
        if (t.center[o] == px.idx) pt = 255.f;
    }
    dmap[px.base + px.idx] = m;
    dist_out[px.base + px.idx] = sqrtf(m) * 10.f;
    impulse[px.base + px.idx] = pt;
}

// gradient_calculation.py:8-50 + direction_map.py:101-123
__global__ void __launch_bounds__(TISEG_THREADS)
k_dl_direction(Geom g, const int32_t* __restrict__ inst, const float* __restrict__ dmap, int num_angles,
               uint8_t* __restrict__ dir_out, float* __restrict__ reg_out) {
    __shared__ float ker[2][121];
    for (int i = threadIdx.x; i < 121; i += blockDim.x) {
        const int j_ = i / 11 - 5, i_ = i % 11 - 5;
        const double den = (double)(i_ * i_ + j_ * j_);
        ker[0][i] = den > 0 ? (float)((double)j_ / den) : 0.f;       // channel 0: rows (sobel_y), channel 1: columns
        ker[1][i] = den > 0 ? (float)((double)i_ / den) : 0.f;
    }
    __syncthreads();
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    const int32_t* tile = inst + px.base;
    const float* dm = dmap + px.base;
    const int v = tile[px.idx];
    uint8_t dir = 0;
    float reg = 0.f;
    if (v > 0) {
        float g0 = 0.f, g1 = 0.f;
        for (int dy = -5; dy <= 5; ++dy) {
            const int yy = px.y + dy;
            if (yy < 0 || yy >= g.H) continue;
            for (int dx = -5; dx <= 5; ++dx) {
                const int xx = px.x + dx;
                if (xx < 0 || xx >= g.W) continue;
                const int q = yy * g.W + xx;
                if (tile[q] != v) continue;
                const float a = dm[q];
                g0 = __fadd_rn(g0, __fmul_rn(a, ker[0][(dy + 5) * 11 + dx + 5]));
                g1 = __fadd_rn(g1, __fmul_rn(a, ker[1][(dy + 5) * 11 + dx + 5]));
            }
        }
        const float angle = atan2f(g0, g1) * (180.0f / 3.14159274101257324f);       // np.degrees(np.arctan2(.)) in float32
        // align_angle (direction_calculation.py:60-73): bin 0 wraps around +-180, bin i is centred on -180 + step * i
        const float step = 360.f / (float)num_angles;
        int idx = 0;
        for (int i = 1; i < num_angles; ++i) {
            const float middle = -180.f + step * (float)i;
            if (angle > middle - step / 2 && angle <= middle + step / 2) idx = i;
        }
        dir = (uint8_t)(idx + 1);
        float r = angle;
        if (r < 0.f) r += 360.f;
        reg = r / 180.f * 3.14159274101257324f;
    }
    dir_out[px.base + px.idx] = dir;
    reg_out[px.base + px.idx] = reg;
}

// scipy.ndimage.gaussian_filter1d along one axis, mode 'reflect', float32 in / out, float64 accumulation in the order of
// NI_Correlate1D's symmetric branch: centre tap first, then the pairs from the outermost inwards
template <int AXIS>
__global__ void __launch_bounds__(TISEG_THREADS)
k_dl_gauss(Geom g, const float* __restrict__ in, const double* __restrict__ w, int radius, float* __restrict__ out) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    const float* tile = in + px.base;
    const int n = AXIS == 0 ? g.H : g.W, c = AXIS == 0 ? px.y : px.x, stride = AXIS == 0 ? g.W : 1;
    const int origin = px.idx - c * stride;
    auto at = [&](int i) {
        while (i < 0 || i >= n) i = i < 0 ? -i - 1 : 2 * n - 1 - i;       // reflect: d c b a | a b c d | d c b a
        return (double)tile[origin + i * stride];
    };
    double tmp = at(c) * w[radius];
    for (int ll = -radius; ll < 0; ++ll) tmp = __dadd_rn(tmp, __dmul_rn(__dadd_rn(at(c + ll), at(c - ll)), w[ll + radius]));
    out[px.base + px.idx] = (float)tmp;
}

// direction_map.py:89-98: dilation with disk(1) = the plus-shaped maximum (out-of-image neighbours do not take part)
__global__ void __launch_bounds__(TISEG_THREADS)
k_dl_weight(Geom g, const float* __restrict__ dd, const float* __restrict__ dist, float* __restrict__ wout) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    const float* D = dd + px.base;
    const float* S = dist + px.base;
    auto val = [&](int y, int x) { const int q = y * g.W + x; return D[q] * (10.f - S[q]); };
    float m = val(px.y, px.x);
    if (px.y > 0) m = fmaxf(m, val(px.y - 1, px.x));
    if (px.y + 1 < g.H) m = fmaxf(m, val(px.y + 1, px.x));
    if (px.x > 0) m = fmaxf(m, val(px.y, px.x - 1));
    if (px.x + 1 < g.W) m = fmaxf(m, val(px.y, px.x + 1));
    wout[px.base + px.idx] = m * 2.f + 1.0f;
}

}  // namespace tiseg

using namespace tiseg;

extern "C" int tiseg_direction_labels(tiseg_ctx* c, const int32_t* inst, int N, int H, int W, int num_angles,
                                      const double* gauss_weights, int gauss_radius, float* dist_out, float* point_out,
                                      uint8_t* dir_out, float* reg_dir_out, float* weight_out) {
    if (!c || !inst || !gauss_weights || gauss_radius < 0 || gauss_radius > 64 || !dist_out || !point_out || !dir_out ||
        !reg_dir_out || num_angles < 2 || num_angles > 64 || (weight_out && num_angles != 8)) {
        set_error("tiseg_direction_labels: bad argument (2 <= num_angles <= 64; the weight map exists for 8 angles only)");
        return TISEG_ERR_ARG;
    }
    Call call(c, "tiseg_direction_labels", N, H, W);
    const size_t total = call.total;
    const int32_t* d_inst = call.in(inst, total);
    float* d_dist = call.out(dist_out, total);
    float* d_point = call.out(point_out, total);
    uint8_t* d_dir = call.out(dir_out, total);
    float* d_reg = call.out(reg_dir_out, total);
    float* d_w = call.out(weight_out, total);
    TISEG_TRY(call.status());
    const Geom& g = call.g;
    const int VM = g.P + 1 < (1 << 16) ? (1 << 16) : g.P + 1;
    const size_t nt = (size_t)N * VM;
    DlTab t;
    t.VM = VM;
    t.best = ws<unsigned long long>(c, nt); t.center = ws<int>(c, nt); t.maxd = ws<unsigned long long>(c, nt);
    double* cent = ws<double>(c, total);
    float* dmap = ws<float>(c, total);
    float* impulse = ws<float>(c, total);
    float* tmp = ws<float>(c, total);
    double* d_gw = ws<double>(c, (size_t)2 * gauss_radius + 1);
    if (!t.best || !t.center || !t.maxd || !cent || !dmap || !impulse || !tmp || !d_gw) return TISEG_ERR_CUDA;
    // (the weights are host data: 2 * radius + 1 doubles, as scipy.ndimage._filters._gaussian_kernel1d returns them)
    TISEG_CHECK(cudaMemcpyAsync(d_gw, gauss_weights, ((size_t)2 * gauss_radius + 1) * sizeof(double), cudaMemcpyDefault, c->stream));
    DlDirs dirs;
    for (int i = 0; i < 8; ++i) { dirs.s[i] = sin(2 * M_PI / 8 * i); dirs.c[i] = cos(2 * M_PI / 8 * i); }   // center_calculation.py:23-24
    TISEG_LAUNCH(c, k_dl_init, (unsigned)((nt + 255) / 256), 256, 0, t, (long long)nt);
    TISEG_LAUNCH(c, k_dl_centerness, warp_grid(g), TISEG_THREADS, 0, g, d_inst, dirs, cent, t, c->d_err);
    TISEG_LAUNCH(c, k_dl_center_pick, warp_grid(g), TISEG_THREADS, 0, g, d_inst, cent, t);
    TISEG_LAUNCH(c, k_dl_maxdist, warp_grid(g), TISEG_THREADS, 0, g, d_inst, t);
    TISEG_LAUNCH(c, k_dl_dist, warp_grid(g), TISEG_THREADS, 0, g, d_inst, t, dmap, d_dist, impulse);
    TISEG_LAUNCH(c, k_dl_direction, warp_grid(g), TISEG_THREADS, 0, g, d_inst, dmap, num_angles, d_dir, d_reg);
    TISEG_LAUNCH(c, k_dl_gauss<0>, warp_grid(g), TISEG_THREADS, 0, g, impulse, d_gw, gauss_radius, tmp);
    TISEG_LAUNCH(c, k_dl_gauss<1>, warp_grid(g), TISEG_THREADS, 0, g, tmp, d_gw, gauss_radius, d_point);
    if (d_w) {
        float* dd = ws<float>(c, total);
        if (!dd) return TISEG_ERR_CUDA;
        TISEG_TRY(ddm_dev(c, g, d_dir, 1, dd));
        TISEG_LAUNCH(c, k_dl_weight, warp_grid(g), TISEG_THREADS, 0, g, dd, d_dist, d_w);
    }
    return call.finish();
}
