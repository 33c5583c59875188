// K6 — ordered marker-controlled watershed (skimage.segmentation.watershed, connectivity 1, compactness 0,
// no lines; dist.py:124, hovernet.py:361).
//
// The library's flood is a sequential priority queue ordered by (value, age): every marker pixel enters with
// age 0 (raster order), the minimum is popped, and each still-unlabelled in-mask 4-neighbour (up, left,
// right, down) is labelled AT PUSH TIME with the popped pixel's label and pushed with the next age.  A
// level-synchronous flood is not equivalent (plateau ties are decided by age), so the order is reproduced
// exactly — but per BLOB: 4-connected components of the mask never interact, and the restriction of the
// global order to one blob is the order of that blob flooded alone.  One warp owns one blob at a time
// (dynamic work queue per tile), so parallelism comes from the ~10^3 blobs per 1000^2 tile times the tiles
// of the batch.
//   uint8 images (DIST):   k_ws_flood_par stages each blob in shared memory, and one warp floods it from one
//                          array queue per level, popping up to 32 entries of the current level per step with
//                          the sequential result.  A blob too large for shared memory is flooded in global
//                          memory by one lane (flood_blob_global: 256 FIFO buckets, links in a global `next`).
//   fp64 images (HoVer):   k_rank_blobs replaces each blob's values by their dense ranks, then k_ws_flood_ranked
//                          floods the staged blob from FIFO buckets in shared memory, one lane per blob.  A blob
//                          too large to rank or stage is flooded by k_ws_flood_f64: a binary heap keyed
//                          (value, age) in a global arena slice sized by the blob's area.
#pragma once
#include "bitccl.cuh"
#include "ccl.cuh"

namespace tiseg {

struct BlobInfo {
    int* root;   // [N, KS] flat index of the blob's first pixel (its ymin = root / W)
    int* ymax;   // [N, KS]
    int* xmin;   // [N, KS]
    int* xmax;   // [N, KS]
    int* area;   // [N, KS]
    int* off;    // [N, KS] exclusive prefix of areas (fp64 heap slices)
    const int* count;  // [N] number of blobs
    int KS;
    // run-based blobs (DIST): smallest and largest marker label seen on the blob's pixels; NULL on the forest path.
    // A blob whose seeds all carry ONE label (lmin == lmax) is simply filled with it and never enters the flood; the
    // flood's work lists only take blobs with lmin < lmax.  (Counted over the marker PIXELS, not the marker roots: a
    // marker plateau is 8-connected and can reach into a second 4-connected blob through a diagonal.)
    int* lmin;   // [N, KS]
    int* lmax;   // [N, KS]
    // optional by-product for a caller that renumbers the flood's regions in raster order (DIST's arrange_label):
    // first[n, label] = lowest flat index of a pixel carrying `label` (initialised to INT_MAX by the caller).  The fill
    // of single-marker blobs and the flood's write-back keep it up to date; NULL = not wanted.
    int* first;  // [N, KS]
};

// How the flood decides which cells of a staged bounding box belong to the blob.
//   forest: a flattened per-pixel forest of the mask (tiseg_watershed_*, HoVer-Net): in the blob <=> tp[pixel] == root.
//   mask:   no per-pixel forest exists (DIST, blobs from bit planes).  Every in-mask cell of the box is staged; cells of
//           OTHER blobs are never reached (blobs are 4-connected components and the flood moves by 4-neighbours), stay
//           unlabelled and are not written back.  Only the seeds must be the blob's own: the kernel that wrote the
//           seeds also wrote, at the same pixels, the id of the blob each of them lies in.
struct BlobMember {
    const int* par;           // forest mode: flattened per-pixel forest; mask mode: unused
    const uint8_t* mask_img;  // mask mode: pixel is in the mask <=> mask_img[pixel] < 255; NULL selects forest mode
    const int* seed_blob;     // mask mode: id of the blob every SEED pixel lies in (written where the seeds were written)
    const unsigned* seed_bits;// mask mode: bitmap of the seed pixels [N, H, SEG] (the flood rewrites the label map while
                              // other blobs are still being staged, so "label != 0" cannot tell a seed there)
    const unsigned* mask_bits;// mask mode: F plane of the mask and the blob forest / ids over its runs (blob_id_at): used to
    const int* bpar;          // clean the label map under the rare blobs that are flooded in global memory
    const int* brank;
};

// label map of the tiles list[0 .. *count): zero wherever the bit plane `keep` is clear (empty blocks when *count == 0)
int label_clean_listed(tiseg_ctx* c, const Geom& g, const int* list, const int* count, const unsigned* keep, int32_t* lab);

// mask functor -> flattened blob forest `par`, blob ids `rank` (at roots), BlobInfo
template <class MaskImg>
int blobs_build(tiseg_ctx* c, const Geom& g, MaskImg mask, int* par, int* rank, BlobInfo& b, bool want_offsets,
                int conn = 1);

int watershed_u8_dev(tiseg_ctx* c, const Geom& g, const uint8_t* image, const int* par, const int* rank,
                     const BlobInfo& b, int32_t* out);
// the same flood with blobs described by bit planes + run forest (mask mode of BlobMember)
int watershed_u8_masked_dev(tiseg_ctx* c, const Geom& g, const uint8_t* image, const BlobMember& mb, const BlobInfo& b, int32_t* out);
// blob table from the planes of the mask, in two steps with the seed scatter of the caller in between:
//   blobs_ccl     forest over runs, ids, roots; lmin / lmax / first-pixel tables initialised
//   (caller)      writes the seeds and, through blob_id_at, reports every seed run to its blob (lmin / lmax, seed_blob)
//   blobs_boxes_fill   boxes + areas of the blobs with two or more marker labels; the others are filled
int blobs_ccl(tiseg_ctx* c, const Geom& g, const BitPlanes& planes, int* par, int* rank, int* first, BlobInfo& b);
// bounding boxes + areas of the blobs that hold two or more marker labels (those are flooded); the pixels of all other
// blobs take their label at once: the single marker's, or 0
int blobs_boxes_fill(tiseg_ctx* c, const Geom& g, const BitPlanes& planes, const int* par, const int* rank, const BlobInfo& b,
                     int32_t* out);
int watershed_f64_dev(tiseg_ctx* c, const Geom& g, const double* image, const int* par, const int* rank,
                      const BlobInfo& b, int32_t* out);

// out = markers where the mask forest has a pixel, else 0 (skimage drops markers outside the mask)
int ws_seed(tiseg_ctx* c, const Geom& g, const int32_t* markers, const int* par, int32_t* out);
// root / bbox / area (/ offsets) of every blob of a flattened + ranked forest
int blobs_describe(tiseg_ctx* c, const Geom& g, const int* par, const int* rank, const unsigned* root_bits, BlobInfo& b,
                   bool want_offsets);

#ifdef __CUDACC__
// id of the blob that holds mask pixel (y, x)
__device__ __forceinline__ int blob_id_at(const BitPlanes& p, const Geom& g, int n, const int* __restrict__ par,
                                          const int* __restrict__ rank, int y, int x) {
    const long long base = (long long)n * g.P;
    return rank[base + find_ro(par + base, bit_node_of(p, g, (long long)n * g.H * g.SEG, y, x))];
}

template <class MaskImg>
int blobs_build(tiseg_ctx* c, const Geom& g, MaskImg mask, int* par, int* rank, BlobInfo& b, bool want_offsets,
                int conn) {
    int N = g.N, KS = g.P + 1;
    size_t ks = (size_t)N * KS;
    int* count = ws<int>(c, (size_t)N);
    b.root = ws<int>(c, ks); b.ymax = ws<int>(c, ks); b.xmin = ws<int>(c, ks); b.xmax = ws<int>(c, ks);
    b.area = ws<int>(c, ks); b.off = want_offsets ? ws<int>(c, ks) : nullptr;
    b.KS = KS; b.count = count; b.lmin = nullptr; b.lmax = nullptr; b.first = nullptr;
    if (!count || !b.root || !b.ymax || !b.xmin || !b.xmax || !b.area || (want_offsets && !b.off)) return TISEG_ERR_CUDA;
    const unsigned* roots;
    TISEG_TRY(ccl_build(c, g, mask, conn, par, &roots));
    TISEG_TRY(rank_from_bits(c, g, roots, rank, count));
    return blobs_describe(c, g, par, rank, roots, b, want_offsets);
}
#endif

}  // namespace tiseg
