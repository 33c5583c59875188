// K11 — exact distance transforms of a binary mask: Euclidean (scipy.ndimage.distance_transform_edt) and chessboard
// (scipy.ndimage.distance_transform_cdt, the default metric).  Neither runs at test time in the reference; they
// build training targets — datasets/ops/distance_map.py:93 (cdt per instance box), datasets/ops/direction_map.py:167,179,
// datasets/ops/unet_map.py:72, datasets/utils/direction_calculation.py:164, models/losses/surface_loss.py:7 (edt) —
// and the synthetic inputs of the bench.
//
// Both metrics separate into a column pass and a row pass:
//   g(x, y)  = vertical distance from (x, y) to the nearest zero of column x            (two sweeps per column)
//   edt^2    = min over x' of (x - x')^2 + g(x', y)^2        cdt = min over x' of max(|x - x'|, g(x', y))
// The row pass widens the search outwards from x and stops as soon as the horizontal offset alone reaches the best
// value found, so its cost is the local object radius, not the row length.  All arithmetic is exact integer; the
// Euclidean result is sqrt of the exact squared distance in fp64, as scipy computes it.
#include "common.cuh"

namespace tiseg {

#define DT_INF 0x3fffffff

__global__ void __launch_bounds__(TISEG_THREADS)
k_dt_columns(Geom g, const uint8_t* __restrict__ mask, int* __restrict__ col, int* has_zero) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, n = blockIdx.y;
    if (x >= g.W) return;
    const uint8_t* m = mask + (long long)n * g.P + x;
    int* c = col + (long long)n * g.P + x;
    int d = DT_INF;
    bool any = false;
    for (int y = 0; y < g.H; ++y) {
        if (m[(long long)y * g.W] == 0) { d = 0; any = true; } else if (d != DT_INF) ++d;
        c[(long long)y * g.W] = d;
    }
    d = DT_INF;
    for (int y = g.H - 1; y >= 0; --y) {
        if (m[(long long)y * g.W] == 0) d = 0; else if (d != DT_INF) ++d;
        if (d < c[(long long)y * g.W]) c[(long long)y * g.W] = d;
    }
    if (any) has_zero[n] = 1;
}

// one block per row; the row of column distances lives in shared memory when it fits
template <bool EUCLID>
__global__ void __launch_bounds__(TISEG_THREADS)
k_dt_rows(Geom g, const int* __restrict__ col, const int* __restrict__ has_zero, double* __restrict__ edt,
          int32_t* __restrict__ cdt, int use_smem) {
    extern __shared__ int srow[];
    const int y = blockIdx.x, n = blockIdx.y;
    const int* grow = col + (long long)n * g.P + (long long)y * g.W;
    const int* row = grow;
    if (use_smem) {
        for (int x = threadIdx.x; x < g.W; x += blockDim.x) srow[x] = grow[x];
        __syncthreads();
        row = srow;
    }
    const bool some = has_zero[n] != 0;
    for (int x = threadIdx.x; x < g.W; x += blockDim.x) {
        long long o = (long long)n * g.P + (long long)y * g.W + x;
        if (!some) {
            // no zero anywhere: scipy's edt then measures from the point (-1, 0) (its feature transform is never
            // written); its cdt reports -1
            if (EUCLID) edt[o] = sqrt((double)((long long)(y + 1) * (y + 1) + (long long)x * x));
            else cdt[o] = -1;
            continue;
        }
        const int g0 = row[x];
        long long best = EUCLID ? (g0 == DT_INF ? (long long)DT_INF * 4 : (long long)g0 * g0) : g0;
        for (int d = 1; d < g.W; ++d) {
            if ((EUCLID ? (long long)d * d : (long long)d) >= best) break;
            if (x - d >= 0) {
                const int gv = row[x - d];
                if (gv != DT_INF) { long long v = EUCLID ? (long long)d * d + (long long)gv * gv : (long long)max(d, gv); if (v < best) best = v; }
            }
            if (x + d < g.W) {
                const int gv = row[x + d];
                if (gv != DT_INF) { long long v = EUCLID ? (long long)d * d + (long long)gv * gv : (long long)max(d, gv); if (v < best) best = v; }
            }
        }
        if (EUCLID) edt[o] = sqrt((double)best);
        else cdt[o] = (int32_t)best;
    }
}

int distance_transform_dev(tiseg_ctx* c, const Geom& g, const uint8_t* mask, int metric, double* edt, int32_t* cdt) {
    size_t total = (size_t)g.N * g.P;
    int* col = ws<int>(c, total);
    int* has_zero = ws<int>(c, (size_t)g.N);
    if (!col || !has_zero) return TISEG_ERR_CUDA;
    TISEG_TRY(zero(c, has_zero, (size_t)g.N * sizeof(int)));
    TISEG_LAUNCH(c, k_dt_columns, dim3((g.W + TISEG_THREADS - 1) / TISEG_THREADS, g.N), TISEG_THREADS, 0, g, mask, col, has_zero);
    const int use_smem = (size_t)g.W * sizeof(int) <= 48 * 1024;
    const size_t smem = use_smem ? (size_t)g.W * sizeof(int) : 0;
    if (metric == 0) TISEG_LAUNCH(c, k_dt_rows<true>, dim3(g.H, g.N), TISEG_THREADS, smem, g, col, has_zero, edt, cdt, use_smem);
    else             TISEG_LAUNCH(c, k_dt_rows<false>, dim3(g.H, g.N), TISEG_THREADS, smem, g, col, has_zero, edt, cdt, use_smem);
    return TISEG_OK;
}

}  // namespace tiseg

using namespace tiseg;

extern "C" {

int tiseg_distance_transform_edt(tiseg_ctx* c, const uint8_t* mask, int N, int H, int W, double* out) {
    if (!c || !mask || !out) { set_error("tiseg_distance_transform_edt: bad argument"); return TISEG_ERR_ARG; }
    Call call(c, "tiseg_distance_transform_edt", N, H, W);
    const uint8_t* d_mask = call.in(mask, call.total);
    double* d_out = call.out(out, call.total);
    TISEG_TRY(call.status());
    TISEG_TRY(distance_transform_dev(c, call.g, d_mask, 0, d_out, nullptr));
    return call.finish();
}

int tiseg_distance_transform_cdt(tiseg_ctx* c, const uint8_t* mask, int N, int H, int W, int32_t* out) {
    if (!c || !mask || !out) { set_error("tiseg_distance_transform_cdt: bad argument"); return TISEG_ERR_ARG; }
    Call call(c, "tiseg_distance_transform_cdt", N, H, W);
    const uint8_t* d_mask = call.in(mask, call.total);
    int32_t* d_out = call.out(out, call.total);
    TISEG_TRY(call.status());
    TISEG_TRY(distance_transform_dev(c, call.g, d_mask, 1, nullptr, d_out));
    return call.finish();
}

}  // extern "C"
