// The step before the softmax / mean of the TTA variants, as load indexing (SURVEY §8f rank 2): window stitch
// (base.py:255-295) and reverse_tta_transform (base.py:365-381).  Shared by the softmax / mean kernels (softmax.cu) and the
// direction / point fronts of the CDNet tails (cdnet.cu).
#pragma once
#include "common.cuh"

namespace tiseg {

// The reference stitches the half-overlap window outputs of every TTA variant into a canvas (base.py:255-295), undoes
// the variant's rotation / flip (base.py:365-381), applies softmax and averages (base.py:321-336).  Those are pure
// re-indexings, so the kernels read every logit ONCE, straight from the window tensors:
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

// the plan of one head of C channels: checks the transforms (rotate_degrees multiples of 90, flips 0..3), 1 <= T <= 16 and
// 0 <= overlap < window; `where` names the entry in the error message (softmax.cu)
int tta_plan(TtaPlan& p, int T, int C, int H, int W, const int* rotate_degrees, const int* flips, int window, int overlap,
             const char* where);

// softmax (or plain) TTA mean + argmax of one head through its plan, k_softmax_argmax_tta (softmax.cu)
template <class TI>
int tta_launch(tiseg_ctx* c, const Geom& g, const TI* d_in, const TtaPlan& plan, int C, float* d_prob, uint8_t* d_cls,
               bool softmax);

#ifdef __CUDACC__
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
#endif

}  // namespace tiseg
