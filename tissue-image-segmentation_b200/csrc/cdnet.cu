// K9 — CDNet direction-guided refinement.
//   tiseg_ddm           generate_direction_differential_map (tiseg/models/utils/direct_diff_map.py:95-167), 9 classes
//   tiseg_cdnet_refine_typed
//                       the tail of CDNet.inference after the CNN (tiseg/models/segmentors/cdnet.py:183-217):
//                       softmax + TTA mean of the semantic head, TTA mean of the point head, per variant
//                       dir[:,0] *= sem[:,0] -> argmax -> DDM, mean DDM, _ddm_enhencement (cdnet.py:354-367), argmax.
// The reference does this with ~60 ATen launches per TTA variant (8 torch.roll temporaries); here the DDM is one
// wrap-around 3x3 stencil on the uint8 direction map plus a per-tile max/min reduction.
// The head outputs may be fp32, fp16 or bf16 (TI): the kernels that read them convert at the load; the probabilities,
// DDM and point mean the library makes from them are fp32.
#include <cfloat>

#include "common.cuh"

namespace tiseg {

template <class TI>
int softmax_argmax_dev(tiseg_ctx* c, const Geom& g, const TI* d_in, int T, int C, float* d_prob, uint8_t* d_cls);   // softmax.cu

// label -> (vertical, horizontal) unit-step vector, direct_diff_map.py:7
__constant__ float c_dir9[9][2] = {{0, 0}, {0, -1}, {-1, -1}, {-1, 0}, {-1, 1}, {0, 1}, {1, 1}, {1, 0}, {1, -1}};

// level = 1 - round(min over the 8 circularly shifted neighbours of cos(anchor, neighbour)), background -> 0.
// The cosine only depends on the two direction labels, so every block first evaluates the reference's fp32
// expression for the 81 label pairs (same operations, same rounding) into a shared table of LEVELS
// (1 - rint(cos); rint is monotone, so 1 - rint(min cos) = max of the pair levels); a pixel is then eight byte loads,
// eight table lookups and a max.
__global__ void __launch_bounds__(TISEG_THREADS)
k_ddm_levels(Geom g, const uint8_t* __restrict__ dir, uint8_t* __restrict__ lv, int* mm) {
    __shared__ int s_lvl[81];
    if (threadIdx.x < 81) {
        const int d = threadIdx.x / 9, e = threadIdx.x - d * 9;
        const float a0 = c_dir9[d][0], a1 = c_dir9[d][1], f0 = c_dir9[e][0], f1 = c_dir9[e][1];
        const float na = sqrtf(a0 * a0 + a1 * a1);
        const float num = a0 * f0 + a1 * f1;
        const float den = na * sqrtf(f0 * f0 + f1 * f1) + 0.000001f;
        s_lvl[threadIdx.x] = d == 0 ? 0 : (int)(1.f - rintf(num / den));      // torch.round: half to even; background -> 1 -> level 0
    }
    __syncthreads();
    Pix px;
    if (!warp_pixel(g, px)) return;
    int level = -1;
    if (px.ok) {
        const uint8_t* t = dir + px.base;
        int d = t[px.idx];
        if (d > 8) d = 0;
        // torch.roll(shifts=(sv, sh)): feature[y, x] = anchor[y - sv, x - sh] (wrap-around); the 8 shifts of
        // direct_diff_map.py:116-131 cover all 8 neighbours, so the extremum does not depend on their order
        level = 0;
        if (d != 0) {
            level = -8;
#pragma unroll
            for (int sv = -1; sv <= 1; ++sv) {
                int yy = px.y - sv; yy = yy < 0 ? yy + g.H : (yy >= g.H ? yy - g.H : yy);
#pragma unroll
                for (int sh = -1; sh <= 1; ++sh) {
                    if (sv == 0 && sh == 0) continue;
                    int xx = px.x - sh; xx = xx < 0 ? xx + g.W : (xx >= g.W ? xx - g.W : xx);
                    int e = t[yy * g.W + xx];
                    if (e > 8) e = 0;
                    level = max(level, s_lvl[d * 9 + e]);
                }
            }
        }
        lv[px.base + px.idx] = (uint8_t)level;
    }
    int hi = level, lo = level < 0 ? 255 : level;
    for (int s = 16; s; s >>= 1) { hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, s)); lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, s)); }
    if (px.lane == 0) {
        if (hi > mm[2 * px.n]) atomicMax(&mm[2 * px.n], hi);
        if (lo < mm[2 * px.n + 1]) atomicMin(&mm[2 * px.n + 1], lo);
    }
}

__global__ void k_ddm_mm_init(int* mm, int n) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { mm[2 * i] = 0; mm[2 * i + 1] = 255; }
}

__device__ __forceinline__ float ddm_normalise(int level, int mx, int mn) {
    float v = (float)level;
    if (mx == 0) return v;                                    // all-zero map is returned as is (:162-163)
    return (v - (float)mn) / ((float)mx - (float)mn);
}

// dd[n] = (sum over the T variants of the normalised DDM) / T   (cdnet.py:201-212), T = 1 for tiseg_ddm
__global__ void __launch_bounds__(TISEG_THREADS)
k_ddm_mean(Geom g, const uint8_t* __restrict__ lv, const int* __restrict__ mm, int T, float* __restrict__ dd) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    float acc = 0.f;
    for (int t = 0; t < T; ++t) {
        long long tile = (long long)px.n * T + t;
        float v = ddm_normalise(lv[tile * g.P + px.idx], mm[2 * tile], mm[2 * tile + 1]);
        acc = t == 0 ? v : acc + v;
    }
    dd[px.base + px.idx] = acc / (float)T;
}

// per variant: softmax over the D direction channels, channel 0 scaled by the mean background probability,
// argmax (first maximum).  Four pixels per thread, every logit read once (128-bit loads), exp evaluated once.
template <class TI, int DMAX>
__global__ void __launch_bounds__(TISEG_THREADS)
k_dir_map(long long P, const TI* __restrict__ dir_logits, const float* __restrict__ sem_prob, int T, int D, int C,
          uint8_t* __restrict__ dir_map, bool vec) {
    const int n = blockIdx.y;
    const long long i = flat4_index();
    if (i >= P) return;
    const Pack4<float> s0 = ld4(sem_prob + ((long long)n * C) * P, i, P, vec);
    for (int t = 0; t < T; ++t) {
        const TI* src = dir_logits + ((long long)n * T + t) * D * P;
        Pack4<float> x[DMAX];
        float m[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
        for (int d = 0; d < DMAX; ++d)
            if (d < D) {
                x[d] = ld4f(src + d * P, i, P, vec);
#pragma unroll
                for (int k = 0; k < 4; ++k) m[k] = fmaxf(m[k], x[d].v[k]);
            }
        float s[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int d = 0; d < DMAX; ++d)
            if (d < D) {
#pragma unroll
                for (int k = 0; k < 4; ++k) { x[d].v[k] = expf(x[d].v[k] - m[k]); s[k] = s[k] + x[d].v[k]; }
            }
        Pack4<uint8_t> best;
        float bv[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
        for (int k = 0; k < 4; ++k) best.v[k] = 0;
#pragma unroll
        for (int d = 0; d < DMAX; ++d)
            if (d < D) {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    float p = x[d].v[k] / s[k];
                    if (d == 0) p = p * s0.v[k];
                    if (p > bv[k]) { bv[k] = p; best.v[k] = (uint8_t)d; }
                }
            }
        st4(dir_map + ((long long)n * T + t) * P, i, P, vec, best);
    }
}

__device__ __forceinline__ int float_order_key(float f) {   // monotone float -> int map for atomicMax
    int b = __float_as_int(f);
    return b >= 0 ? b : b ^ 0x7fffffff;
}
__device__ __forceinline__ float float_from_key(int k) { return __int_as_float(k >= 0 ? k : k ^ 0x7fffffff); }

__global__ void k_key_init(int* k, int n) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) k[i] = float_order_key(-INFINITY);
}

// point = sum_t point_t / T and its per-tile maximum
template <class TI>
__global__ void __launch_bounds__(TISEG_THREADS)
k_point_mean(Geom g, const TI* __restrict__ point_logits, int T, float* __restrict__ pmean, int* pmax_key) {
    Pix px;
    if (!warp_pixel(g, px)) return;
    float acc = -INFINITY;
    if (px.ok) {
        for (int t = 0; t < T; ++t) {
            float v = to_f32(point_logits[((long long)px.n * T + t) * g.P + px.idx]);
            acc = t == 0 ? v : acc + v;
        }
        acc = acc / (float)T;
        pmean[px.base + px.idx] = acc;
    }
    int k = float_order_key(acc);
    for (int s = 16; s; s >>= 1) k = max(k, __shfl_xor_sync(0xffffffffu, k, s));
    if (px.lane == 0 && k > pmax_key[px.n]) atomicMax(&pmax_key[px.n], k);
}

// _ddm_enhencement + argmax.
//   mode 0 (cdnet.py:354-367):            p[-1] = (p[-1] + dd') * (1 + dd'),  dd' = dd - dd * (point / max(point) > 0.2)
//   mode 1 (multi_task_cdnet.py:548-564): f = ((point + 0.2) / max(point + 0.2))^2,  dd' = dd - dd * (f > 0.6),
//                                         p[-1] = p[-1] * (1 + dd') * (1 - f), values >= 1 become 0.95
//         (its last line, `sem_logit[:, -2][foreground_map == 0.8] = 1`, compares a bool map with 0.8 and never fires)
// fp32 throughout, operations in the reference's order; max(point + 0.2) = fl(max(point) + 0.2f) because fp32 addition is
// monotone.
__global__ void __launch_bounds__(TISEG_THREADS)
k_ddm_enhance(Geom g, float* __restrict__ sem_prob, int C, const float* __restrict__ dd, const float* __restrict__ pmean,
              const int* __restrict__ pmax_key, int if_ddm, int mode, uint8_t* __restrict__ cls) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    const long long P = g.P;
    float* sp = sem_prob + (long long)px.n * C * P + px.idx;
    if (if_ddm) {
        const float pm = float_from_key(pmax_key[px.n]);
        const float d = dd[px.base + px.idx];
        if (mode == 0) {
            const float pmap = (pmean[px.base + px.idx] / pm) > 0.2f ? 1.f : 0.f;
            const float d2 = d - d * pmap;
            sp[(C - 1) * P] = (sp[(C - 1) * P] + d2) * (1.f + d2);
        } else {
            const float t = (pmean[px.base + px.idx] + 0.2f) / (pm + 0.2f);
            const float f = t * t;
            const float d2 = d - d * (f > 0.6f ? 1.f : 0.f);
            float e = (sp[(C - 1) * P] * (1.f + d2)) * (1.f - f);
            if (e >= 1.f) e = 0.95f;
            sp[(C - 1) * P] = e;
        }
    }
    if (cls) {
        int best = 0;
        float bv = -INFINITY;
        for (int ch = 0; ch < C; ++ch) { float p = sp[ch * P]; if (p > bv) { bv = p; best = ch; } }
        cls[px.base + px.idx] = (uint8_t)best;
    }
}

int ddm_dev(tiseg_ctx* c, const Geom& g, const uint8_t* dir_map, int T, float* dd) {
    // dir_map: [N*T, H, W]; dd: [N, H, W]
    Geom gt = make_geom(g.N * T, g.H, g.W);
    uint8_t* lv = ws<uint8_t>(c, (size_t)gt.N * gt.P);
    int* mm = ws<int>(c, 2 * (size_t)gt.N);
    if (!lv || !mm) return TISEG_ERR_CUDA;
    TISEG_LAUNCH(c, k_ddm_mm_init, (gt.N + 255) / 256, 256, 0, mm, gt.N);
    TISEG_LAUNCH(c, k_ddm_levels, warp_grid(gt), TISEG_THREADS, 0, gt, dir_map, lv, mm);
    TISEG_LAUNCH(c, k_ddm_mean, warp_grid(g), TISEG_THREADS, 0, g, lv, mm, T, dd);
    return TISEG_OK;
}

}  // namespace tiseg

using namespace tiseg;

extern "C" {

int tiseg_ddm(tiseg_ctx* c, const uint8_t* dir_map, int N, int H, int W, float* dd) {
    if (!c || !dir_map || !dd) { set_error("tiseg_ddm: bad argument"); return TISEG_ERR_ARG; }
    TISEG_TRY(check_geom(N, H, W));
    begin_call(c);
    Geom g = make_geom(N, H, W);
    size_t total = (size_t)N * g.P;
    const uint8_t* d_dir = in(c, dir_map, total);
    float* d_dd = tiseg::out(c, dd, total);
    if (!d_dir || !d_dd) return TISEG_ERR_CUDA;
    TISEG_TRY(ddm_dev(c, g, d_dir, 1, d_dd));
    return end_call(c);
}

}  // extern "C"

// the refinement after the front kernels: per-variant direction maps from dir_all on, TI = element type of the heads
template <class TI>
static int cdnet_refine_run(tiseg_ctx* c, const Geom& g, const TI* d_sem, const TI* d_dir, const TI* d_pt, int T, int C, int D,
                            int if_ddm, float* d_prob, uint8_t* d_cls, float* d_dd, uint8_t* dir_all, float* pmean, int* pmax) {
    const int N = g.N;
    // softmax + TTA mean of the semantic head: the K1 kernel
    TISEG_TRY(softmax_argmax_dev(c, g, d_sem, T, C, d_prob, nullptr));
    {
        const bool v4 = (g.P % 4 == 0) && aligned_x4<TI>(d_dir) && aligned16(d_prob) && (((uintptr_t)dir_all) & 3) == 0;
        const dim3 fg(flat4_grid(g.P), (unsigned)N);
        TISEG_LAUNCH_AS(c, TISEG_IN_NAME(TI, "k_dir_map<9>"), (k_dir_map<TI, 9>), fg, TISEG_THREADS, 0, (long long)g.P, d_dir, d_prob, T, D, C,
                        dir_all, v4);     // D == 9 is checked by the caller
    }
    TISEG_TRY(ddm_dev(c, g, dir_all, T, d_dd));
    TISEG_LAUNCH(c, k_key_init, (N + 255) / 256, 256, 0, pmax, N);
    TISEG_LAUNCH_AS(c, TISEG_IN_NAME(TI, "k_point_mean"), k_point_mean<TI>, warp_grid(g), TISEG_THREADS, 0, g, d_pt, T, pmean, pmax);
    TISEG_LAUNCH(c, k_ddm_enhance, warp_grid(g), TISEG_THREADS, 0, g, d_prob, C, d_dd, pmean, pmax, if_ddm, 0, d_cls);
    return TISEG_OK;
}

extern "C" {

int tiseg_cdnet_refine_typed(tiseg_ctx* c, int dtype, const void* sem_logits, const void* dir_logits, const void* point_logits,
                             int N, int T, int C, int D, int H, int W, int if_ddm, float* sem_prob_out, uint8_t* cls_out,
                             uint8_t* dir_map_out, float* dd_out) {
    TISEG_TRY(check_dtype(dtype, "tiseg_cdnet_refine_typed"));
    if (!c || !sem_logits || !dir_logits || !point_logits || T <= 0 || C < 2 || C > 16 || D != 9) {
        set_error("tiseg_cdnet_refine_typed: bad argument (2 <= C <= 16, D == 9)");
        return TISEG_ERR_ARG;
    }
    TISEG_TRY(check_geom(N * T, H, W));
    begin_call(c);
    Geom g = make_geom(N, H, W);
    size_t total = (size_t)N * g.P;
    const size_t eb = dtype_bytes(dtype);
    const void* d_sem = in_ptr(c, sem_logits, total * T * C * eb);
    const void* d_dir = in_ptr(c, dir_logits, total * T * D * eb);
    const void* d_pt = in_ptr(c, point_logits, total * T * eb);
    float* d_prob = sem_prob_out ? tiseg::out(c, sem_prob_out, total * C) : ws<float>(c, total * C);
    uint8_t* d_cls = cls_out ? tiseg::out(c, cls_out, total) : nullptr;
    float* d_dd = dd_out ? tiseg::out(c, dd_out, total) : ws<float>(c, total);
    uint8_t* dir_all = ws<uint8_t>(c, total * T);
    float* pmean = ws<float>(c, total);
    int* pmax = ws<int>(c, (size_t)N);
    if (!d_sem || !d_dir || !d_pt || !d_prob || !d_dd || !dir_all || !pmean || !pmax) return TISEG_ERR_CUDA;
    TISEG_TRY(with_dtype(dtype, [&](auto z) {
        using TI = decltype(z);
        return cdnet_refine_run(c, g, (const TI*)d_sem, (const TI*)d_dir, (const TI*)d_pt, T, C, D, if_ddm, d_prob, d_cls, d_dd,
                                dir_all, pmean, pmax);
    }));
    if (dir_map_out) {
        // dir_map_list[0] of every tile (cdnet.py:217)
        uint8_t* d_dm = tiseg::out(c, dir_map_out, total);
        if (!d_dm) return TISEG_ERR_CUDA;
        TISEG_CHECK(cudaMemcpy2DAsync(d_dm, g.P, dir_all, (size_t)T * g.P, g.P, N, cudaMemcpyDeviceToDevice, c->stream));
    }
    return end_call(c);
}

int tiseg_ddm_enhance(tiseg_ctx* c, float* sem_prob, const float* dd, const float* point, int N, int C, int H, int W, int mode) {
    if (!c || !sem_prob || !dd || !point || C < 2 || C > 16 || (mode != 0 && mode != 1)) {
        set_error("tiseg_ddm_enhance: bad argument (2 <= C <= 16, mode 0 | 1)");
        return TISEG_ERR_ARG;
    }
    TISEG_TRY(check_geom(N, H, W));
    begin_call(c);
    Geom g = make_geom(N, H, W);
    const size_t total = (size_t)N * g.P;
    float* d_prob = (float*)inout_ptr(c, sem_prob, total * C * sizeof(float));
    const float* d_dd = in(c, dd, total);
    const float* d_pt = in(c, point, total);
    float* pmean = ws<float>(c, total);
    int* pmax = ws<int>(c, (size_t)N);
    if (!d_prob || !d_dd || !d_pt || !pmean || !pmax) return TISEG_ERR_CUDA;
    TISEG_LAUNCH(c, k_key_init, (N + 255) / 256, 256, 0, pmax, N);
    TISEG_LAUNCH_AS(c, "k_point_mean", k_point_mean<float>, warp_grid(g), TISEG_THREADS, 0, g, d_pt, 1, pmean, pmax);
    TISEG_LAUNCH(c, k_ddm_enhance, warp_grid(g), TISEG_THREADS, 0, g, d_prob, C, d_dd, pmean, pmax, 1, mode, (uint8_t*)nullptr);
    return end_call(c);
}

}  // extern "C"

namespace tiseg {
// use_regression (multi_task_cdnet.py:304-315): the direction head is ONE channel, an angle in radians.  Per variant:
// clamp to [0, 2 pi], degrees, (180, 360] -> (-180, 0], class = 1 + bin of align_angle with eight angles
// (direction_calculation.py:60-73); background (first maximum of the mean three-class probabilities is class 0) -> 0.
template <class TI>
__global__ void __launch_bounds__(TISEG_THREADS)
k_reg_dir_map(Geom g, const TI* __restrict__ reg, const float* __restrict__ tc_prob, int T, int C, uint8_t* __restrict__ dir_map) {
    Pix px;
    if (!warp_pixel(g, px) || !px.ok) return;
    const float* tp = tc_prob + (long long)px.n * C * g.P + px.idx;
    float best = tp[0];
    bool bg = true;
    for (int k = 1; k < C; ++k) if (tp[(long long)k * g.P] > best) { best = tp[(long long)k * g.P]; bg = false; }
    for (int t = 0; t < T; ++t) {
        const long long tile = (long long)px.n * T + t;
        float a = to_f32(reg[tile * g.P + px.idx]);
        if (a < 0.f) a = 0.f;
        if (a > 6.28318548202514648f) a = 6.28318548202514648f;
        float deg = (a * 180.f) / 3.14159274101257324f;
        if (deg > 180.f) deg -= 360.f;
        int idx = 0;
        for (int i = 1; i < 8; ++i) {
            const float middle = -180.f + 45.f * (float)i;
            if (deg > middle - 22.5f && deg <= middle + 22.5f) idx = i;
        }
        dir_map[tile * g.P + px.idx] = bg ? (uint8_t)0 : (uint8_t)(idx + 1);
    }
}
}  // namespace tiseg

// the refinement after the staging, TI = element type of the heads
template <class TI>
static int mtcdnet_refine_run(tiseg_ctx* c, const Geom& g, const TI* d_tc, const TI* d_sem, const TI* d_dir, const TI* d_pt, int T,
                              int Ctc, int Csem, int D, int if_ddm, float* d_tcp, uint8_t* d_tcc, float* d_semp, uint8_t* d_semc,
                              float* d_dd, uint8_t* dir_all, float* pmean, int* pmax) {
    const int N = g.N;
    const size_t total = (size_t)N * g.P;
    // softmax + TTA mean of the three-class and of the semantic head (multi_task_cdnet.py:283-294)
    TISEG_TRY(softmax_argmax_dev(c, g, d_tc, T, Ctc, d_tcp, nullptr));
    if (d_semp || d_semc) {
        float* sp = d_semp;
        if (!sp && T > 1) { sp = ws<float>(c, total * Csem); if (!sp) return TISEG_ERR_CUDA; }      // (T == 1: streaming argmax)
        TISEG_TRY(softmax_argmax_dev(c, g, d_sem, T, Csem, sp, d_semc));
    }
    if (D == 1) {   // use_regression: the angle head -> classes (:304-315)
        TISEG_LAUNCH_AS(c, TISEG_IN_NAME(TI, "k_reg_dir_map"), k_reg_dir_map<TI>, warp_grid(g), TISEG_THREADS, 0, g, d_dir, d_tcp, T, Ctc, dir_all);
    } else {   // per variant: dir[:, 0] *= tc[:, 0]; argmax; DDM (:318-322)
        const bool v4 = (g.P % 4 == 0) && aligned_x4<TI>(d_dir) && aligned16(d_tcp) && (((uintptr_t)dir_all) & 3) == 0;
        TISEG_LAUNCH_AS(c, TISEG_IN_NAME(TI, "k_dir_map<9>"), (k_dir_map<TI, 9>), dim3(flat4_grid(g.P), (unsigned)N), TISEG_THREADS, 0,
                        (long long)g.P, d_dir, d_tcp, T, D, Ctc, dir_all, v4);
    }
    TISEG_TRY(ddm_dev(c, g, dir_all, T, d_dd));
    TISEG_LAUNCH(c, k_key_init, (N + 255) / 256, 256, 0, pmax, N);
    TISEG_LAUNCH_AS(c, TISEG_IN_NAME(TI, "k_point_mean"), k_point_mean<TI>, warp_grid(g), TISEG_THREADS, 0, g, d_pt, T, pmean, pmax);
    TISEG_LAUNCH(c, k_ddm_enhance, warp_grid(g), TISEG_THREADS, 0, g, d_tcp, Ctc, d_dd, pmean, pmax, if_ddm, 1, d_tcc);
    return TISEG_OK;
}

extern "C" {

int tiseg_mtcdnet_refine_typed(tiseg_ctx* c, int dtype, const void* tc_logits, const void* sem_logits, const void* dir_logits,
                               const void* point_logits, int N, int T, int Ctc, int Csem, int D, int H, int W, int if_ddm,
                               float* tc_prob_out, uint8_t* tc_cls_out, float* sem_prob_out, uint8_t* sem_cls_out,
                               uint8_t* dir_map_out, float* dd_out) {
    TISEG_TRY(check_dtype(dtype, "tiseg_mtcdnet_refine_typed"));
    if (!c || !tc_logits || !sem_logits || !dir_logits || !point_logits || T <= 0 || Ctc < 2 || Ctc > 16 || Csem < 1 ||
        Csem > 16 || (D != 9 && D != 1)) {
        set_error("tiseg_mtcdnet_refine_typed: bad argument (2 <= Ctc <= 16, 1 <= Csem <= 16, D == 9, or D == 1: the regression head)");
        return TISEG_ERR_ARG;
    }
    TISEG_TRY(check_geom(N * T, H, W));
    begin_call(c);
    Geom g = make_geom(N, H, W);
    const size_t total = (size_t)N * g.P;
    const size_t eb = dtype_bytes(dtype);
    const void* d_tc = in_ptr(c, tc_logits, total * T * Ctc * eb);
    const void* d_sem = in_ptr(c, sem_logits, total * T * Csem * eb);
    const void* d_dir = in_ptr(c, dir_logits, total * T * D * eb);
    const void* d_pt = in_ptr(c, point_logits, total * T * eb);
    float* d_tcp = tc_prob_out ? tiseg::out(c, tc_prob_out, total * Ctc) : ws<float>(c, total * Ctc);
    uint8_t* d_tcc = tc_cls_out ? tiseg::out(c, tc_cls_out, total) : nullptr;
    float* d_semp = sem_prob_out ? tiseg::out(c, sem_prob_out, total * Csem) : nullptr;
    uint8_t* d_semc = sem_cls_out ? tiseg::out(c, sem_cls_out, total) : nullptr;
    float* d_dd = dd_out ? tiseg::out(c, dd_out, total) : ws<float>(c, total);
    uint8_t* dir_all = ws<uint8_t>(c, total * T);
    float* pmean = ws<float>(c, total);
    int* pmax = ws<int>(c, (size_t)N);
    if (!d_tc || !d_sem || !d_dir || !d_pt || !d_tcp || !d_dd || !dir_all || !pmean || !pmax) return TISEG_ERR_CUDA;
    TISEG_TRY(with_dtype(dtype, [&](auto z) {
        using TI = decltype(z);
        return mtcdnet_refine_run(c, g, (const TI*)d_tc, (const TI*)d_sem, (const TI*)d_dir, (const TI*)d_pt, T, Ctc, Csem, D, if_ddm,
                                  d_tcp, d_tcc, d_semp, d_semc, d_dd, dir_all, pmean, pmax);
    }));
    if (dir_map_out) {
        uint8_t* d_dm = tiseg::out(c, dir_map_out, total);
        if (!d_dm) return TISEG_ERR_CUDA;
        TISEG_CHECK(cudaMemcpy2DAsync(d_dm, g.P, dir_all, (size_t)T * g.P, g.P, N, cudaMemcpyDeviceToDevice, c->stream));
    }
    return end_call(c);
}

}  // extern "C"
