// K5b — grey-scale reconstruction by erosion (skimage.morphology.reconstruction(seed, mask, method='erosion'), 3x3
// footprint; dist.py:43-57 H_reconstruction_erosion).  At test time the reference calls it with lambda = 0.0
// (dist.py:281), where it is the identity, and with h = 1 inside find_maxima, which the DIST path replaces by the
// regional-minimum analysis of dist.cu; this kernel serves lambda > 0 (the paper's p1) and the stand-alone operator.
//
// R = greatest fixed point below the seed of  R <- max(erode3x3(R), mask).  The operator is monotone, so chaotic
// (asynchronous) iteration reaches the same fixed point: every CTA keeps a 32 x 32 tile plus a one-pixel halo in shared
// memory, relaxes it until nothing changes inside the tile, writes it back and raises a flag if it changed anything;
// the host repeats the sweep until a whole sweep raises no flag (out-of-image taps never lower a pixel).
#include "common.cuh"

namespace tiseg {

#define RC_T 32
__global__ void __launch_bounds__(256)
k_recon_erode_tile(Geom g, const uint8_t* __restrict__ mask, uint8_t* R, int* changed) {
    __shared__ uint8_t sr[(RC_T + 2) * (RC_T + 2)];
    __shared__ uint8_t sm[RC_T * RC_T];
    __shared__ int again, any;
    const int tilesX = (g.W + RC_T - 1) / RC_T;
    const int ty = blockIdx.x / tilesX, tx = blockIdx.x - ty * tilesX, n = blockIdx.y;
    const int x0 = tx * RC_T, y0 = ty * RC_T;
    const long long base = (long long)n * g.P;
    for (int i = threadIdx.x; i < (RC_T + 2) * (RC_T + 2); i += blockDim.x) {
        const int ly = i / (RC_T + 2), lx = i - ly * (RC_T + 2), y = y0 + ly - 1, x = x0 + lx - 1;
        sr[i] = (y >= 0 && y < g.H && x >= 0 && x < g.W) ? R[base + (long long)y * g.W + x] : (uint8_t)255;
    }
    for (int i = threadIdx.x; i < RC_T * RC_T; i += blockDim.x) {
        const int ly = i / RC_T, lx = i - ly * RC_T, y = y0 + ly, x = x0 + lx;
        sm[i] = (y < g.H && x < g.W) ? mask[base + (long long)y * g.W + x] : (uint8_t)255;
    }
    if (threadIdx.x == 0) any = 0;
    __syncthreads();
    for (int it = 0; it < 4 * RC_T; ++it) {
        if (threadIdx.x == 0) again = 0;
        __syncthreads();
        bool ch = false;
        for (int i = threadIdx.x; i < RC_T * RC_T; i += blockDim.x) {
            const int ly = i / RC_T, lx = i - ly * RC_T, c = (ly + 1) * (RC_T + 2) + lx + 1;
            int mn = 255;
#pragma unroll
            for (int dy = -1; dy <= 1; ++dy)
#pragma unroll
                for (int dx = -1; dx <= 1; ++dx) mn = min(mn, (int)sr[c + dy * (RC_T + 2) + dx]);
            const int v = max(mn, (int)sm[i]);
            if (v < sr[c]) { sr[c] = (uint8_t)v; ch = true; }       // in place: any order reaches the same fixed point
        }
        if (ch) again = 1;
        __syncthreads();
        if (!again) break;
        if (threadIdx.x == 0) any = 1;
        __syncthreads();
    }
    __syncthreads();
    if (!any) return;
    for (int i = threadIdx.x; i < RC_T * RC_T; i += blockDim.x) {
        const int ly = i / RC_T, lx = i - ly * RC_T, y = y0 + ly, x = x0 + lx;
        if (y < g.H && x < g.W) R[base + (long long)y * g.W + x] = sr[(ly + 1) * (RC_T + 2) + lx + 1];
    }
    if (threadIdx.x == 0) *changed = 1;
}

__global__ void __launch_bounds__(TISEG_THREADS)
k_recon_seed(long long total, const uint8_t* __restrict__ mask, const uint8_t* __restrict__ seed, int add, uint8_t* __restrict__ R) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    // seed given: clamp it from below by the mask (the library requires seed >= mask); else seed = min(255, mask + add)
    const int m = mask[i];
    R[i] = (uint8_t)(seed ? max((int)seed[i], m) : min(255, m + add));
}

// R <- reconstruction by erosion of `mask` from R (R >= mask on entry).  Synchronises with the host between sweeps.
int reconstruction_erosion_dev(tiseg_ctx* c, const Geom& g, const uint8_t* mask, uint8_t* R) {
    int* changed = ws<int>(c, 1);
    if (!changed) return TISEG_ERR_CUDA;
    const int tiles = ((g.W + RC_T - 1) / RC_T) * ((g.H + RC_T - 1) / RC_T);
    for (int sweep = 0; sweep < g.H + g.W + 8; ++sweep) {
        TISEG_TRY(zero(c, changed, sizeof(int)));
        for (int k = 0; k < 4; ++k) TISEG_LAUNCH(c, k_recon_erode_tile, dim3(tiles, g.N), 256, 0, g, mask, R, changed);
        int h = 0;
        TISEG_CHECK(cudaMemcpyAsync(&h, changed, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
        TISEG_CHECK(cudaStreamSynchronize(c->stream));
        if (!h) return TISEG_OK;
    }
    set_error("reconstruction did not converge");
    return TISEG_ERR_LIMIT;
}

int h_reconstruction_erosion_dev(tiseg_ctx* c, const Geom& g, const uint8_t* img, int h, uint8_t* out) {
    const long long total = (long long)g.N * g.P;
    TISEG_LAUNCH(c, k_recon_seed, flat_grid(total), TISEG_THREADS, 0, total, img, (const uint8_t*)nullptr, h, out);
    return reconstruction_erosion_dev(c, g, img, out);
}

}  // namespace tiseg

using namespace tiseg;

extern "C" int tiseg_reconstruction_erosion_u8(tiseg_ctx* c, const uint8_t* seed, const uint8_t* mask, int N, int H, int W,
                                               uint8_t* out) {
    if (!c || !seed || !mask || !out) { set_error("tiseg_reconstruction_erosion_u8: bad argument"); return TISEG_ERR_ARG; }
    Call call(c, "tiseg_reconstruction_erosion_u8", N, H, W);
    const long long total = (long long)call.total;
    const uint8_t* d_seed = call.in(seed, total);
    const uint8_t* d_mask = call.in(mask, total);
    uint8_t* d_out = call.out(out, total);
    TISEG_TRY(call.status());
    TISEG_LAUNCH(c, k_recon_seed, flat_grid(total), TISEG_THREADS, 0, total, d_mask, d_seed, 0, d_out);
    TISEG_TRY(reconstruction_erosion_dev(c, call.g, d_mask, d_out));
    return call.finish();
}
