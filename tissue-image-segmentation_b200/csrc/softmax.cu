// K1 — softmax over channels + TTA mean + argmax in one pass over the logits.
// Replaces tiseg/models/segmentors/base.py:321-339 (F.softmax per variant, sum/len) and the
// `argmax(dim=1)` + `.cpu().numpy()` that every segmentor does next (unet.py:62-64, dist.py:266).
//
// fp32 arithmetic in the same order as the reference expression: e = exp(x - max), s = e_0 + e_1 + ...,
// p = e / s, acc += p per variant, acc / T.  One thread per pixel, channel planes read coalesced.
// The logits may be fp32, fp16 or bf16 (TI = the element type); they are converted to fp32 as they are loaded.
#include "common.cuh"

namespace tiseg {

template <class TI, int CMAX>
__global__ void __launch_bounds__(TISEG_THREADS)
k_softmax_argmax(long long P, const TI* __restrict__ logits, int T, int C, float* __restrict__ prob,
                 uint8_t* __restrict__ cls, bool vec) {
    // one thread = 4 consecutive pixels of one tile (blockIdx.y): float4 per channel plane, uchar4 out
    const int n = blockIdx.y;
    const long long i = flat4_index();
    if (i >= P) return;
    float acc[CMAX][4];
    for (int t = 0; t < T; ++t) {
        const TI* src = logits + ((long long)n * T + t) * C * P;
        Pack4<float> x[CMAX];
        float m[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
        for (int c = 0; c < CMAX; ++c)
            if (c < C) {
                x[c] = ld4f(src + c * P, i, P, vec);
#pragma unroll
                for (int k = 0; k < 4; ++k) m[k] = fmaxf(m[k], x[c].v[k]);
            }
        float s[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int c = 0; c < CMAX; ++c)
            if (c < C) {
#pragma unroll
                for (int k = 0; k < 4; ++k) { x[c].v[k] = expf(x[c].v[k] - m[k]); s[k] = s[k] + x[c].v[k]; }
            }
#pragma unroll
        for (int c = 0; c < CMAX; ++c)
            if (c < C) {
#pragma unroll
                for (int k = 0; k < 4; ++k) acc[c][k] = (t == 0) ? x[c].v[k] / s[k] : acc[c][k] + x[c].v[k] / s[k];
            }
    }
    const float tf = (float)T;
    Pack4<uint8_t> best;
    float bv[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
    for (int k = 0; k < 4; ++k) best.v[k] = 0;
#pragma unroll
    for (int c = 0; c < CMAX; ++c)
        if (c < C) {
            Pack4<float> p;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                p.v[k] = acc[c][k] / tf;
                if (p.v[k] > bv[k]) { bv[k] = p.v[k]; best.v[k] = (uint8_t)c; }
            }
            if (prob) st4(prob + ((long long)n * C + c) * P, i, P, vec, p);
        }
    if (cls) st4(cls + (long long)n * P, i, P, vec, best);
}

// One variant and only the class map wanted.  softmax is increasing in the logit, so away from ties the class is the
// first maximum of the logits themselves (pure streaming, no exp).  It is NOT the same thing inside the tie band: the
// reference takes the first maximum of the fp32 PROBABILITIES (base.py:332-336, unet.py:62), and exp(x_c - max) rounds
// to exactly 1.0f for every logit within ~8e-8 of the maximum (and e / s can round to 1 / s a little further out), so
// an EARLIER class whose logit is a hair below the maximum wins there.  Bound: with max - x_c > 1e-6, e_c <= 1 - 7e-7
// under expf's 2-ulp error and two roundings of 6e-8 cannot close that gap, so the probabilities are strictly ordered
// like the logits.  Pixels with a runner-up inside 1e-6 (or a NaN) are re-evaluated with the exact arithmetic of
// k_softmax_argmax (same expf, same summation order, first maximum).
template <class TI, int CMAX>
__global__ void __launch_bounds__(TISEG_THREADS)
k_argmax_logits(long long P, const TI* __restrict__ logits, int C, uint8_t* __restrict__ cls, bool vec) {
    const int n = blockIdx.y;
    const long long i = flat4_index();
    if (i >= P) return;
    const TI* src = logits + (long long)n * C * P;
    Pack4<float> x[CMAX];
#pragma unroll
    for (int c = 0; c < CMAX; ++c) if (c < C) x[c] = ld4f(src + c * P, i, P, vec);
    Pack4<uint8_t> best;
    float bv[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) { best.v[k] = 0; bv[k] = x[0].v[k]; }
#pragma unroll
    for (int c = 1; c < CMAX; ++c)
        if (c < C) {
#pragma unroll
            for (int k = 0; k < 4; ++k) if (x[c].v[k] > bv[k]) { bv[k] = x[c].v[k]; best.v[k] = (uint8_t)c; }
        }
    // runner-up inside the tie band (or NaN)?  count the logits not clearly below the maximum; the maximum itself is one
    int near[4] = {0, 0, 0, 0};
#pragma unroll
    for (int c = 0; c < CMAX; ++c)
        if (c < C) {
#pragma unroll
            for (int k = 0; k < 4; ++k) near[k] += (bv[k] - x[c].v[k] > 1.0e-6f) ? 0 : 1;
        }
    if ((near[0] | near[1] | near[2] | near[3]) > 1) {            // rare: the exact arithmetic of k_softmax_argmax
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (near[k] <= 1) continue;
            float m = -INFINITY, e[CMAX], sum = 0.f;
#pragma unroll
            for (int c = 0; c < CMAX; ++c) if (c < C) m = fmaxf(m, x[c].v[k]);
#pragma unroll
            for (int c = 0; c < CMAX; ++c) if (c < C) { e[c] = expf(x[c].v[k] - m); sum = sum + e[c]; }
            int b = 0;
            float pv = -INFINITY;
#pragma unroll
            for (int c = 0; c < CMAX; ++c)
                if (c < C) {
                    const float p = (e[c] / sum) / 1.f;          // T = 1: the TTA mean divides by 1
                    if (p > pv) { pv = p; b = c; }
                }
            best.v[k] = (uint8_t)b;
        }
    }
    st4(cls + (long long)n * P, i, P, vec, best);
}

// The same for exactly two classes (every binary nuclei model), written for the instruction issue rate: 32-bit tile-local
// offsets from opaque tile bases, no class loop.  The generic kernel spends ~35 instructions per pixel on index arithmetic
// and dead class slots and ran at 60 % of the HBM rate; this one is bound by the two reads per pixel (4 B each in fp32).
template <class TI>
__global__ void __launch_bounds__(TISEG_THREADS)
k_argmax_logits2(int P, const TI* __restrict__ logits, uint8_t* __restrict__ cls, bool vec) {
    const int i = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i >= P) return;
    const TI* a = logits + (long long)blockIdx.y * 2 * P;
    uint8_t* o = cls + (long long)blockIdx.y * P;
    asm volatile("" : "+l"(a)); asm volatile("" : "+l"(o));
    __builtin_assume(__isGlobal(a)); __builtin_assume(__isGlobal(o));
    float x0[4], x1[4];
    if (vec) {
        ld4f_aligned(a + i, x0);
        ld4f_aligned(a + P + i, x1);
    } else {
#pragma unroll
        for (int k = 0; k < 4; ++k) { x0[k] = i + k < P ? to_f32(a[i + k]) : 0.f; x1[k] = i + k < P ? to_f32(a[P + i + k]) : 1.f; }
    }
    unsigned best = 0u;
    bool near = false;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        if (x1[k] > x0[k]) best |= 1u << (8 * k);
        near |= !(fabsf(x1[k] - x0[k]) > 1.0e-6f);               // runner-up inside the tie band, or a NaN
    }
    if (near) {                                                  // rare: the exact arithmetic of k_softmax_argmax
        best = 0u;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            unsigned b = x1[k] > x0[k] ? 1u : 0u;
            if (!(fabsf(x1[k] - x0[k]) > 1.0e-6f)) {
                const float m = fmaxf(fmaxf(-INFINITY, x0[k]), x1[k]);
                const float e0 = expf(x0[k] - m), e1 = expf(x1[k] - m);
                float sum = 0.f; sum = sum + e0; sum = sum + e1;
                const float p0 = (e0 / sum) / 1.f, p1 = (e1 / sum) / 1.f;        // T = 1: the TTA mean divides by 1
                int bb = 0; float pv = -INFINITY;
                if (p0 > pv) { pv = p0; bb = 0; }
                if (p1 > pv) { pv = p1; bb = 1; }
                b = (unsigned)bb;
            }
            best |= b << (8 * k);
        }
    }
    if (vec) *reinterpret_cast<unsigned*>(o + i) = best;
    else {
#pragma unroll
        for (int k = 0; k < 4; ++k) if (i + k < P) o[i + k] = (uint8_t)(best >> (8 * k));
    }
}

// (the fp32 launches keep their plain timing names; the half-precision ones carry the dtype, TISEG_IN_NAME)
template <class TI>
int softmax_argmax_dev(tiseg_ctx* c, const Geom& g, const TI* d_in, int T, int C, float* d_prob, uint8_t* d_cls) {
    const long long P = g.P;
    const bool vec = (P % 4 == 0) && aligned_x4<TI>(d_in) && aligned16(d_prob) && (((uintptr_t)d_cls) & 3) == 0;
    dim3 grid(flat4_grid(P), (unsigned)g.N);
    if (T == 1 && !d_prob) {
        if (C == 2) TISEG_LAUNCH_AS(c, TISEG_IN_NAME(TI, "k_argmax_logits2"), k_argmax_logits2<TI>, grid, TISEG_THREADS, 0, (int)P, d_in, d_cls, vec);
        else if (C <= 2) TISEG_LAUNCH_AS(c, TISEG_IN_NAME(TI, "k_argmax_logits<2>"), (k_argmax_logits<TI, 2>), grid, TISEG_THREADS, 0, P, d_in, C, d_cls, vec);
        else if (C <= 4) TISEG_LAUNCH_AS(c, TISEG_IN_NAME(TI, "k_argmax_logits<4>"), (k_argmax_logits<TI, 4>), grid, TISEG_THREADS, 0, P, d_in, C, d_cls, vec);
        else if (C <= 8) TISEG_LAUNCH_AS(c, TISEG_IN_NAME(TI, "k_argmax_logits<8>"), (k_argmax_logits<TI, 8>), grid, TISEG_THREADS, 0, P, d_in, C, d_cls, vec);
        else TISEG_LAUNCH_AS(c, TISEG_IN_NAME(TI, "k_argmax_logits<16>"), (k_argmax_logits<TI, 16>), grid, TISEG_THREADS, 0, P, d_in, C, d_cls, vec);
        return TISEG_OK;
    }
    if (C <= 4) TISEG_LAUNCH_AS(c, TISEG_IN_NAME(TI, "k_softmax_argmax<4>"), (k_softmax_argmax<TI, 4>), grid, TISEG_THREADS, 0, P, d_in, T, C, d_prob, d_cls, vec);
    else if (C <= 8) TISEG_LAUNCH_AS(c, TISEG_IN_NAME(TI, "k_softmax_argmax<8>"), (k_softmax_argmax<TI, 8>), grid, TISEG_THREADS, 0, P, d_in, T, C, d_prob, d_cls, vec);
    else TISEG_LAUNCH_AS(c, TISEG_IN_NAME(TI, "k_softmax_argmax<16>"), (k_softmax_argmax<TI, 16>), grid, TISEG_THREADS, 0, P, d_in, T, C, d_prob, d_cls, vec);
    return TISEG_OK;
}
template int softmax_argmax_dev<float>(tiseg_ctx*, const Geom&, const float*, int, int, float*, uint8_t*);
template int softmax_argmax_dev<__half>(tiseg_ctx*, const Geom&, const __half*, int, int, float*, uint8_t*);
template int softmax_argmax_dev<__nv_bfloat16>(tiseg_ctx*, const Geom&, const __nv_bfloat16*, int, int, float*, uint8_t*);

// ---- the step before K1, fused into its load indexing (SURVEY §8f rank 2) ------------------------------------------
// The reference stitches the half-overlap window outputs of every TTA variant into a canvas (base.py:255-295), undoes
// the variant's rotation / flip (base.py:365-381), applies softmax and averages (base.py:321-336).  Those are pure
// re-indexings, so this kernel reads every logit ONCE, straight from the window tensors:
//   original pixel (y, x)  ->  pixel of the variant's (transformed) image, by the inverse of reverse_tta_transform
//                          ->  window (my, mx) whose kept centre region holds it, and the position inside the window.
// window == 0 means "whole" inference: the variant tensor is the full transformed image.
struct TtaPlan {
    int T;
    int rot[16];                // rotate_degree // 90 of the forward transform (0..3)
    int flip[16];               // 0 none, 1 horizontal, 2 vertical, 3 diagonal
    long long off[16];          // element offset of variant t inside one tile's block of the input
    long long tile_stride;      // elements per tile
    int window, overlap;
};

__device__ __forceinline__ void tta_source(const TtaPlan& p, int t, int H, int W, int y, int x, int& sy, int& sx, int& Ht,
                                           int& Wt) {
    // Y = rot90(flip(X), k), k = (4 - rot) % 4, with torch.rot90 counter-clockwise: rot90(Z, 1)[i, j] = Z[j, Wz - 1 - i]
    const int k = (4 - p.rot[t]) & 3;
    Ht = (k & 1) ? W : H; Wt = (k & 1) ? H : W;       // shape of Z (and of X)
    int a, b;
    if (k == 0) { a = y; b = x; }
    else if (k == 1) { a = x; b = Wt - 1 - y; }
    else if (k == 2) { a = Ht - 1 - y; b = Wt - 1 - x; }
    else { a = Ht - 1 - x; b = y; }
    const int f = p.flip[t];
    sy = (f & 2) ? Ht - 1 - a : a;
    sx = (f & 1) ? Wt - 1 - b : b;
}

// element index (without the channel term) of pixel (sy, sx) of a variant image of shape (Ht, Wt): whole tensor or windows
__device__ __forceinline__ long long window_source(const TtaPlan& p, int C, int Ht, int Wt, int sy, int sx, long long& cstride) {
    if (p.window == 0) { cstride = (long long)Ht * Wt; return (long long)sy * Wt + sx; }
    const int win = p.window, ov = p.overlap, st = win - ov;
    const int pad_h = Ht - win > 0 ? st - (Ht - win) % st : win - Ht;          // base.py:264-273
    const int pad_w = Wt - win > 0 ? st - (Wt - win) % st : win - Wt;
    const int H1 = Ht + pad_h, W1 = Wt + pad_w;
    const int My = (H1 - win) / st + 1, Mx = (W1 - win) / st + 1;
    const int Y = sy + (H1 - Ht) / 2, X = sx + (W1 - Wt) / 2;                    // crop of base.py:294
    int my = (Y - ov / 2) / st; my = my < 0 ? 0 : (my > My - 1 ? My - 1 : my);
    int mx = (X - ov / 2) / st; mx = mx < 0 ? 0 : (mx > Mx - 1 ? Mx - 1 : mx);
    if (Y < ov / 2) my = 0;
    if (X < ov / 2) mx = 0;
    cstride = (long long)win * win;
    return ((long long)(my * Mx + mx) * C) * win * win + (long long)(Y - my * st) * win + (X - mx * st);
}

// SOFTMAX = false: the plain mean of the reverse-transformed variants, what the reference does with its regression heads
// (`sum(dist_logit_list) / len(dist_logit_list)`, dist.py:398-410; hovernet.py:406 keeps variant 0 only, i.e. T = 1)
template <class TI, int CMAX, bool SOFTMAX>
__global__ void __launch_bounds__(TISEG_THREADS)
k_softmax_argmax_tta(Geom g, const TI* __restrict__ in, TtaPlan plan, int C, float* __restrict__ prob,
                     uint8_t* __restrict__ cls) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    float acc[CMAX];
    for (int t = 0; t < plan.T; ++t) {
        int sy, sx, Ht, Wt;
        tta_source(plan, t, g.H, g.W, px.y, px.x, sy, sx, Ht, Wt);
        long long cs;
        const TI* src = in + (long long)px.n * plan.tile_stride + plan.off[t] + window_source(plan, C, Ht, Wt, sy, sx, cs);
        float xv[CMAX], m = -INFINITY;
#pragma unroll
        for (int c = 0; c < CMAX; ++c) if (c < C) { xv[c] = to_f32(src[c * cs]); m = fmaxf(m, xv[c]); }
        if (SOFTMAX) {
            float sum = 0.f;
#pragma unroll
            for (int c = 0; c < CMAX; ++c) if (c < C) { xv[c] = expf(xv[c] - m); sum = sum + xv[c]; }
#pragma unroll
            for (int c = 0; c < CMAX; ++c) if (c < C) acc[c] = (t == 0) ? xv[c] / sum : acc[c] + xv[c] / sum;
        } else {
#pragma unroll
            for (int c = 0; c < CMAX; ++c) if (c < C) acc[c] = (t == 0) ? xv[c] : acc[c] + xv[c];
        }
    }
    const float tf = (float)plan.T;
    int best = 0;
    float bv = -INFINITY;
#pragma unroll
    for (int c = 0; c < CMAX; ++c)
        if (c < C) {
            const float pv = acc[c] / tf;
            if (pv > bv) { bv = pv; best = c; }
            if (prob) prob[((long long)px.n * C + c) * g.P + px.idx] = pv;
        }
    if (cls) cls[px.base + px.idx] = (uint8_t)best;
}

}  // namespace tiseg

using namespace tiseg;

// elements of one variant: the whole transformed image, or all its windows
static long long tta_variant_elems(int C, int Ht, int Wt, int window, int overlap) {
    if (window == 0) return (long long)C * Ht * Wt;
    const int st = window - overlap;
    const int pad_h = Ht - window > 0 ? st - (Ht - window) % st : window - Ht;
    const int pad_w = Wt - window > 0 ? st - (Wt - window) % st : window - Wt;
    const int My = (Ht + pad_h - window) / st + 1, Mx = (Wt + pad_w - window) / st + 1;
    return (long long)My * Mx * C * window * window;
}

extern "C" long long tiseg_tta_input_elems(int T, int C, int H, int W, const int* rotate_degrees, int window, int overlap) {
    long long n = 0;
    for (int t = 0; t < T; ++t) {
        const bool odd = ((rotate_degrees[t] / 90) & 1) != 0;
        n += tta_variant_elems(C, odd ? W : H, odd ? H : W, window, overlap);
    }
    return n;
}

template <class TI>
static int tta_launch(tiseg_ctx* c, const Geom& g, const TI* d_in, const TtaPlan& plan, int C, float* d_prob, uint8_t* d_cls,
                      bool softmax) {
    if (softmax) {
        if (C <= 4) TISEG_LAUNCH_AS(c, TISEG_IN_NAME(TI, "(k_softmax_argmax_tta<4, true>)"), (k_softmax_argmax_tta<TI, 4, true>), warp_grid(g), TISEG_THREADS, 0, g, d_in, plan, C, d_prob, d_cls);
        else if (C <= 8) TISEG_LAUNCH_AS(c, TISEG_IN_NAME(TI, "(k_softmax_argmax_tta<8, true>)"), (k_softmax_argmax_tta<TI, 8, true>), warp_grid(g), TISEG_THREADS, 0, g, d_in, plan, C, d_prob, d_cls);
        else TISEG_LAUNCH_AS(c, TISEG_IN_NAME(TI, "(k_softmax_argmax_tta<16, true>)"), (k_softmax_argmax_tta<TI, 16, true>), warp_grid(g), TISEG_THREADS, 0, g, d_in, plan, C, d_prob, d_cls);
    } else {
        if (C <= 4) TISEG_LAUNCH_AS(c, TISEG_IN_NAME(TI, "(k_softmax_argmax_tta<4, false>)"), (k_softmax_argmax_tta<TI, 4, false>), warp_grid(g), TISEG_THREADS, 0, g, d_in, plan, C, d_prob, d_cls);
        else if (C <= 8) TISEG_LAUNCH_AS(c, TISEG_IN_NAME(TI, "(k_softmax_argmax_tta<8, false>)"), (k_softmax_argmax_tta<TI, 8, false>), warp_grid(g), TISEG_THREADS, 0, g, d_in, plan, C, d_prob, d_cls);
        else TISEG_LAUNCH_AS(c, TISEG_IN_NAME(TI, "(k_softmax_argmax_tta<16, false>)"), (k_softmax_argmax_tta<TI, 16, false>), warp_grid(g), TISEG_THREADS, 0, g, d_in, plan, C, d_prob, d_cls);
    }
    return TISEG_OK;
}

static int tta_entry(tiseg_ctx* c, int dtype, const void* logits, int N, int T, int C, int H, int W, const int* rotate_degrees,
                     const int* flips, int window, int overlap, float* prob, uint8_t* cls, bool softmax) {
    if (!c || !logits || !rotate_degrees || !flips || T <= 0 || T > 16 || C <= 0 || C > 16 || (!prob && !cls) ||
        window < 0 || (window > 0 && (overlap < 0 || overlap >= window))) {
        set_error("tiseg_softmax_argmax_tta_typed: bad argument (1 <= T, C <= 16, 0 <= overlap < window)");
        return TISEG_ERR_ARG;
    }
    TISEG_TRY(check_geom(N, H, W));
    TtaPlan plan;
    plan.T = T; plan.window = window; plan.overlap = overlap;
    long long off = 0;
    for (int t = 0; t < T; ++t) {
        if (rotate_degrees[t] % 90 != 0 || flips[t] < 0 || flips[t] > 3) { set_error("tiseg_softmax_argmax_tta_typed: bad transform"); return TISEG_ERR_ARG; }
        plan.rot[t] = ((rotate_degrees[t] / 90) % 4 + 4) % 4;
        plan.flip[t] = flips[t];
        plan.off[t] = off;
        const bool odd = (plan.rot[t] & 1) != 0;
        off += tta_variant_elems(C, odd ? W : H, odd ? H : W, window, overlap);
    }
    plan.tile_stride = off;
    begin_call(c);
    Geom g = make_geom(N, H, W);
    size_t total = (size_t)N * g.P;
    const void* d_in = in_ptr(c, logits, (size_t)N * (size_t)off * dtype_bytes(dtype));
    float* d_prob = prob ? tiseg::out(c, prob, total * C) : nullptr;
    uint8_t* d_cls = cls ? tiseg::out(c, cls, total) : nullptr;
    if (!d_in) return TISEG_ERR_CUDA;
    TISEG_TRY(with_dtype(dtype, [&](auto z) { return tta_launch(c, g, (const decltype(z)*)d_in, plan, C, d_prob, d_cls, softmax); }));
    return end_call(c);
}

extern "C" int tiseg_softmax_argmax_tta_typed(tiseg_ctx* c, int dtype, const void* logits, int N, int T, int C, int H, int W,
                                              const int* rotate_degrees, const int* flips, int window, int overlap,
                                              float* prob, uint8_t* cls) {
    TISEG_TRY(check_dtype(dtype, "tiseg_softmax_argmax_tta_typed"));
    return tta_entry(c, dtype, logits, N, T, C, H, W, rotate_degrees, flips, window, overlap, prob, cls, true);
}

extern "C" int tiseg_tta_mean_typed(tiseg_ctx* c, int dtype, const void* maps, int N, int T, int C, int H, int W,
                                    const int* rotate_degrees, const int* flips, int window, int overlap, float* mean_out) {
    TISEG_TRY(check_dtype(dtype, "tiseg_tta_mean_typed"));
    if (!mean_out) { set_error("tiseg_tta_mean_typed: null output"); return TISEG_ERR_ARG; }
    return tta_entry(c, dtype, maps, N, T, C, H, W, rotate_degrees, flips, window, overlap, mean_out, nullptr, false);
}

extern "C" int tiseg_softmax_argmax_typed(tiseg_ctx* c, int dtype, const void* logits, int N, int T, int C, int H, int W,
                                          float* prob, uint8_t* cls) {
    TISEG_TRY(check_dtype(dtype, "tiseg_softmax_argmax_typed"));
    if (!c || !logits || T <= 0 || C <= 0 || C > 16 || (!prob && !cls)) {
        set_error("tiseg_softmax_argmax_typed: bad argument (1 <= C <= 16)");
        return TISEG_ERR_ARG;
    }
    TISEG_TRY(check_geom(N, H, W));
    begin_call(c);
    Geom g = make_geom(N, H, W);
    size_t total = (size_t)N * g.P;
    const void* d_in = in_ptr(c, logits, total * T * C * dtype_bytes(dtype));
    float* d_prob = prob ? tiseg::out(c, prob, total * C) : nullptr;
    uint8_t* d_cls = cls ? tiseg::out(c, cls, total) : nullptr;
    if (!d_in) return TISEG_ERR_CUDA;
    TISEG_TRY(with_dtype(dtype, [&](auto z) { return softmax_argmax_dev(c, g, (const decltype(z)*)d_in, T, C, d_prob, d_cls); }));
    return end_call(c);
}
