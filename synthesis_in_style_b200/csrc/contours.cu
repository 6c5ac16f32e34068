// Contour stage on the device (SURVEY.md §8(f) row 1): class masks -> colour label image + drop decision, per batch.
// Replaces the host loop of BlackWhiteHandwrittenPrintedTextDatasetSegmenter.create_segmentation_image
//   scf/segmentation/black_white_handwritten_printed_text_segmenter.py:42-99
//   scf/segmentation/base_cluster_based_dataset_segmenter.py:148-450   (contours, overlap, merge, classify, render)
//   scf/segmentation/base_dataset_segmenter.py:52-57                   (3x3 cross dilation)
// which works on cv2 polygons.  Nothing here traces a polygon; the same results come from label maps:
//
//   * drawContours(FILLED) of an external contour of an 8-connected component = the component plus everything it
//     encloses = one 8-connected component of the complement of the OUTSIDE background (background 4-connected to the
//     image border).  Two union-find labellings per plane (background/4, then filled foreground/8) give every filled
//     shape; its root is its smallest linear index = the first point findContours reports.
//   * contourArea (Green's formula over the chain) = pixels - L/2 - 1, where L = number of chain points = boundary
//     cracks minus convex corners, both local 3x3 counts (Pick's theorem; a single pixel gives L = 0, area 0).
//   * boundingRect = min / max of the shape's pixels.
//   * merge_contours' result SET does not depend on its merge order: "strict bounding-box test and a common pixel" only
//     becomes true as shapes grow, so the set is the closure of that relation.  It is computed as a fixpoint: pixel-wise
//     pair detection -> union-find over shapes -> group bounding boxes -> for every merged group the holes of its union
//     (flood fill of the group's bounding-box window held as a bitmask in shared memory: the reference re-traces the
//     union's outer contour, which fills them) -> repeat while anything changed.
//   * classification = per-pixel overlap histogram (fine group, region class), rendering = per-pixel lookup.
//
// The ORDER of the merged contours (which the reference's drop rule reads: width and height of the FIRST contour of a
// class, segmentation_utils.py:60-64 + black_white...:61-75) is not reproduced.  The kernel decides the drop flag when it
// does not depend on the order (no contour of the class exceeds the limit, or all of them do) and otherwise marks the
// image for the host path (flag 2), as it does when a capacity is exceeded.  tests/test_contours_gpu.py compares label
// images and flags with synthesis_in_style_b200/contours.py (the polygon implementation pinned by the reference's goldens).
#include <limits.h>
#include <stdlib.h>
#include "common.cuh"

namespace sis {

constexpr int CT_MAX_PLANE_TYPES = 32;
constexpr int CT_MAX_KEYS = 4;
constexpr int CT_MAX_CLASSES = 7;
enum { CTR_SHAPES = 0, CTR_OVERFLOW = 1, CTR_NUM = 8 };
// The merge fixpoint is controlled ON THE DEVICE: the host enqueues CT_ROUNDS rounds of {pairs, boxes, pairs again, boxes,
// list, fill small, fill big} without ever reading a result back; every kernel of a round first looks at the control
// words the earlier kernels left and returns at once when it has nothing to do.  A batch whose fixpoint is still moving
// after the last round is handed to the host path (flag 2 on every image).
constexpr int CT_ROUNDS = 6;
enum { CTL_CHANGED1 = 0, CTL_DEFERRED1 = 1, CTL_CHANGED2 = 2, CTL_GLIST = 3, CTL_GLIST_BIG = 4, CTL_FILL_NEW = 5, CTL_STRIDE = 8 };

struct CtGeom {
    int B, S, n_cls, n_det, n_fine, fine_cls, px;
    int only_keep_overlapping, limit;
    double min_area2;                                   // 2 * min_class_contour_area
    const uint8_t* planes[CT_MAX_PLANE_TYPES];          // [B, S, S] each: det (key k, class c) at k*n_cls+c, then fine key k
    uint8_t colors[(CT_MAX_CLASSES + 1) * 3];           // background, then the classes
    int render_rank[CT_MAX_CLASSES];                    // later rank overwrites earlier (mask-dict order of the last fine key)
    __host__ __device__ int n_plane_types() const { return n_cls * n_det + n_fine; }
    __host__ __device__ int n_seg_types() const { return n_cls + 1; }
    // segment type st: 0..n_cls-1 = class-determination shapes of class st, n_cls = fine-grained shapes of fine_cls
    __host__ __device__ int keys_of(int st) const { return st < n_cls ? n_det : n_fine; }
    __host__ __device__ int plane_type(int st, int k) const { return st < n_cls ? k * n_cls + st : n_cls * n_det + k; }
};

struct CtWs {
    int32_t *lab, *aux, *fillmap, *key_count;
    uint8_t *fmask, *touch;
    int cap;
    int32_t *sh_seg, *sh_cnt, *sh_L, *sh_x0, *sh_y0, *sh_x1, *sh_y1, *parent;
    int32_t *g_x0, *g_y0, *g_x1, *g_y1, *g_members, *g_filled, *g_cnt, *g_L, *g_kept, *g_cls, *score, *glist;
    int32_t *ctr, *ctl, *img_kept, *img_huge;
    uint32_t* scratch;          // per-block bitmask slices of the big-window fill kernel (image sizes above ~830), or null
    int scratch_words;
};

// round o does something iff it is the first one or the round before it left new coverage / unfinished merging behind
__device__ __forceinline__ bool ct_round_active(const CtWs& W, int o) {
    if (o == 0) return true;
    const volatile int32_t* c = W.ctl + (o - 1) * CTL_STRIDE;
    return c[CTL_FILL_NEW] != 0 || c[CTL_CHANGED2] != 0;
}


// ------------------------------------------------------------------------------------------------ union-find
__device__ __forceinline__ int uf_find(const int32_t* parent, int i) {
    while (true) {
        const int p = ((const volatile int32_t*)parent)[i];
        if (p == i) return i;
        i = p;
    }
}
// find with path halving: every visited node is re-pointed at its grandparent (always an ancestor, so concurrent finds and
// unions stay correct).  Rows of one big region link into chains as long as the region is tall; without this every
// later find walks them again (measured on the pipeline's masks: outside test 179 -> 110 us, border marking 31 -> 15 us).
__device__ __forceinline__ int uf_find_halve(int32_t* parent, int i) {
    while (true) {
        const int p = ((volatile int32_t*)parent)[i];
        if (p == i) return i;
        const int gp = ((volatile int32_t*)parent)[p];
        if (gp != p) ((volatile int32_t*)parent)[i] = gp;
        i = gp;
    }
}
// links the larger root under the smaller one; true when this call joined two sets
__device__ __forceinline__ bool uf_unite(int32_t* parent, int a, int b) {
    while (true) {
        a = uf_find_halve(parent, a);
        b = uf_find_halve(parent, b);
        if (a == b) return false;
        if (a > b) { const int t = a; a = b; b = t; }
        const int old = atomicMin(&parent[b], a);
        if (old == b) return true;
        b = old;
    }
}

// ------------------------------------------------------------------------------------------------ shapes of a plane
// Union-find labelling with run starts: a pixel's first parent is the start of its horizontal run inside its 32-pixel
// warp segment (one ballot, no atomics), and the merge kernels only join where a run meets something new (the segment
// seam, and the first pixel of every contact with the row above).  A plane that is one big background region costs a few
// joins per row instead of two atomics per pixel (measured: 1.63 -> 0.2 ms for the background pass of 192 planes).
__device__ __forceinline__ int ct_run_start(bool in, bool row_start, int lane) {
    // lane of the first pixel of this lane's run: runs do not cross pixels outside the set nor a row start
    const unsigned inb = __ballot_sync(0xffffffffu, in), rs = __ballot_sync(0xffffffffu, in && row_start);
    const unsigned below = lane == 31 ? 0xffffffffu : ((2u << lane) - 1u);              // lanes <= lane
    const unsigned stop_in = rs & below, stop_out = ~inb & (below >> 1);                 // lanes < lane outside the set
    const int c1 = stop_in ? 31 - __clz(stop_in) : 0, c2 = stop_out ? 32 - __clz(stop_out) : 0;
    return c1 > c2 ? c1 : c2;
}

// pass 1: dilated mask; background pixels point at their run start, foreground = -1
__global__ void __launch_bounds__(256) ct_bg_init_kernel(const __grid_constant__ CtGeom G, const __grid_constant__ CtWs W) {
    const int total = G.n_plane_types() * G.B * G.px, rounded = (total + 31) / 32 * 32;     // < 2^31 (checked on the host)
    const int lane = threadIdx.x & 31;
    for (int i = blockIdx.x * 256 + threadIdx.x; i < rounded; i += gridDim.x * 256) {
        const bool valid = i < total;
        const int plane = valid ? i / G.px : 0, p = valid ? i - plane * G.px : 0;
        const int y = p / G.S, x = p - y * G.S;
        bool d = true;
        if (valid) {
            const int t = plane / G.B, b = plane - t * G.B;
            const uint8_t* m = G.planes[t] + (int64_t)b * G.px;
            d = m[p] != 0;                                          // 3x3 cross (base_dataset_segmenter.py:52-57)
            if (!d && y > 0) d = m[p - G.S] != 0;
            if (!d && y < G.S - 1) d = m[p + G.S] != 0;
            if (!d && x > 0) d = m[p - 1] != 0;
            if (!d && x < G.S - 1) d = m[p + 1] != 0;
        }
        const int start = ct_run_start(valid && !d, x == 0, lane);
        if (valid) {
            W.aux[i] = d ? -1 : p - (lane - start);
            W.touch[i] = 0;
        }
    }
}
// background, 4-connectivity
__global__ void __launch_bounds__(256) ct_bg_merge_kernel(const __grid_constant__ CtGeom G, const __grid_constant__ CtWs W) {
    const int total = G.n_plane_types() * G.B * G.px;
    const int lane = threadIdx.x & 31;
    for (int i = blockIdx.x * 256 + threadIdx.x; i < total; i += gridDim.x * 256) {
        const int plane = i / G.px, p = i - plane * G.px;
        int32_t* par = W.aux + (int64_t)plane * G.px;
        if (par[p] < 0) continue;
        const int y = p / G.S, x = p - y * G.S;
        const bool w = x > 0 && par[p - 1] >= 0;
        if (w && lane == 0) uf_unite(par, p, p - 1);                // the run continues across the segment seam
        if (y > 0 && par[p - G.S] >= 0 && !(w && par[p - G.S - 1] >= 0)) uf_unite(par, p, p - G.S);
    }
}
// background sets that reach the image border are the outside (marked at their roots, once the sets are final)
__global__ void __launch_bounds__(256) ct_bg_touch_kernel(const __grid_constant__ CtGeom G, const __grid_constant__ CtWs W) {
    const int total = G.n_plane_types() * G.B * 4 * G.S;
    for (int i = blockIdx.x * 256 + threadIdx.x; i < total; i += gridDim.x * 256) {
        const int plane = i / (4 * G.S), j = i - plane * 4 * G.S, side = j / G.S, t = j - side * G.S;
        const int p = side == 0 ? t : side == 1 ? (G.S - 1) * G.S + t : side == 2 ? t * G.S : t * G.S + G.S - 1;
        int32_t* par = W.aux + (int64_t)plane * G.px;
        if (par[p] >= 0) W.touch[(int64_t)plane * G.px + uf_find_halve(par, p)] = 1;
    }
}
// pass 2: filled foreground = dilated mask + background that does not reach the border; pixels point at their run start
__global__ void __launch_bounds__(256) ct_fg_init_kernel(const __grid_constant__ CtGeom G, const __grid_constant__ CtWs W) {
    const int total = G.n_plane_types() * G.B * G.px, rounded = (total + 31) / 32 * 32;     // < 2^31 (checked on the host)
    const int lane = threadIdx.x & 31;
    for (int i = blockIdx.x * 256 + threadIdx.x; i < rounded; i += gridDim.x * 256) {
        const bool valid = i < total;
        const int plane = valid ? i / G.px : 0, p = valid ? i - plane * G.px : 0;
        const int x = p % G.S;
        bool f = false;
        if (valid) {
            int32_t* par = W.aux + (int64_t)plane * G.px;
            f = par[p] < 0 || W.touch[(int64_t)plane * G.px + uf_find_halve(par, p)] == 0;
        }
        const int start = ct_run_start(f, x == 0, lane);
        if (valid) {
            W.fmask[i] = f ? 1 : 0;
            W.lab[i] = f ? p - (lane - start) : -1;
        }
    }
}
// filled foreground, 8-connectivity: W at the segment seam; N at the first pixel of a contact; NW / NE only when neither N
// nor the run neighbour on that side already carries the link
__global__ void __launch_bounds__(256) ct_fg_merge_kernel(const __grid_constant__ CtGeom G, const __grid_constant__ CtWs W) {
    const int total = G.n_plane_types() * G.B * G.px;
    const int lane = threadIdx.x & 31;
    for (int i = blockIdx.x * 256 + threadIdx.x; i < total; i += gridDim.x * 256) {
        if (!W.fmask[i]) continue;
        const int plane = i / G.px, p = i - plane * G.px;
        int32_t* lab = W.lab + (int64_t)plane * G.px;
        const uint8_t* f = W.fmask + (int64_t)plane * G.px;
        const int S = G.S, y = p / S, x = p - y * S;
        const bool w = x > 0 && f[p - 1];
        if (w && lane == 0) uf_unite(lab, p, p - 1);
        if (y == 0) continue;
        const bool n = f[p - S], nw = x > 0 && f[p - S - 1];
        if (n) {
            if (!(w && nw)) uf_unite(lab, p, p - S);
        } else {
            if (nw && !w) uf_unite(lab, p, p - S - 1);
            if (x < S - 1 && f[p - S + 1] && !f[p + 1]) uf_unite(lab, p, p - S + 1);
        }
    }
}
// roots get a compact shape id (aux[root]); every pixel's label becomes its root
__global__ void __launch_bounds__(256) ct_fg_ids_kernel(const __grid_constant__ CtGeom G, const __grid_constant__ CtWs W) {
    const int total = G.n_plane_types() * G.B * G.px;
    for (int i = blockIdx.x * 256 + threadIdx.x; i < total; i += gridDim.x * 256) {
        if (!W.fmask[i]) continue;
        const int plane = i / G.px, p = i - plane * G.px;
        int32_t* lab = W.lab + (int64_t)plane * G.px;
        // plain find: every store of this kernel is a final root.  (A halving find here could land its grandparent store
        // AFTER another thread's root store and leave a pixel pointing at an inner node, which the next kernel would read.)
        const int r = uf_find(lab, p);
        if (r != p) { lab[p] = r; continue; }
        const int id = atomicAdd(&W.ctr[CTR_SHAPES], 1);
        if (id >= W.cap) { W.ctr[CTR_OVERFLOW] = 1; W.aux[i] = -1; continue; }
        W.aux[i] = id;
        const int t = plane / G.B, b = plane - t * G.B;
        const int st = t < G.n_cls * G.n_det ? t % G.n_cls : G.n_cls;
        W.sh_seg[id] = st * G.B + b;
        W.sh_cnt[id] = 0; W.sh_L[id] = 0;
        W.sh_x0[id] = INT_MAX; W.sh_y0[id] = INT_MAX; W.sh_x1[id] = -1; W.sh_y1[id] = -1;
        W.parent[id] = id;
        W.g_filled[id] = 0; W.g_kept[id] = 0; W.g_cls[id] = -1;
        for (int c = 0; c < G.n_cls; ++c) W.score[(int64_t)id * G.n_cls + c] = 0;
        atomicAdd(&W.key_count[plane], 1);
    }
}
// per-shape pixel count, chain length (cracks - convex corners) and bounding box; labels become shape ids
__global__ void __launch_bounds__(256) ct_shape_stats_kernel(const __grid_constant__ CtGeom G, const __grid_constant__ CtWs W) {
    const int total = G.n_plane_types() * G.B * G.px;
    const int lane = threadIdx.x & 31;
    for (int i = blockIdx.x * 256 + threadIdx.x; i < total; i += gridDim.x * 256) {
        if (!W.fmask[i]) continue;
        const int plane = i / G.px, p = i - plane * G.px;
        const int64_t base = (int64_t)plane * G.px;
        const int id = W.aux[base + W.lab[i]];
        W.lab[i] = id;
        if (id < 0) continue;
        const uint8_t* f = W.fmask + base;
        const int S = G.S, y = p / S, x = p - y * S;
        const bool up = y == 0 || !f[p - S], dn = y == S - 1 || !f[p + S], lf = x == 0 || !f[p - 1], rt = x == S - 1 || !f[p + 1];
        int L = (int)up + dn + lf + rt;
        if (L) {
            // a convex corner: both sides outside and the diagonal not part of the shape (a diagonal pixel would be a pinch)
            if (up && lf && !(y > 0 && x > 0 && f[p - S - 1])) --L;
            if (up && rt && !(y > 0 && x < S - 1 && f[p - S + 1])) --L;
            if (dn && lf && !(y < S - 1 && x > 0 && f[p + S - 1])) --L;
            if (dn && rt && !(y < S - 1 && x < S - 1 && f[p + S + 1])) --L;
            if (L) atomicAdd(&W.sh_L[id], L);
            if (lf) atomicMin(&W.sh_x0[id], x);
            if (rt) atomicMax(&W.sh_x1[id], x);
            if (up) atomicMin(&W.sh_y0[id], y);
            if (dn) atomicMax(&W.sh_y1[id], y);
        }
        // one add per shape and warp: neighbouring lanes mostly sit in the same shape
        const unsigned same = __match_any_sync(__activemask(), id);
        if (lane == __ffs(same) - 1) atomicAdd(&W.sh_cnt[id], __popc(same));
    }
}

// ------------------------------------------------------------------------------------------------ merge fixpoint
__device__ __forceinline__ bool ct_strict(const CtWs& W, int a, int b) {
    // BBox.is_overlapping_with (segmentation_utils.py:50-54): touching boxes do not overlap
    return W.g_x0[a] < W.g_x1[b] && W.g_x1[a] > W.g_x0[b] && W.g_y0[a] < W.g_y1[b] && W.g_y1[a] > W.g_y0[b];
}
// the groups whose filled shape covers pixel p of segment (st, b): one per key plus the hole fill
__device__ __forceinline__ int ct_cover(const CtGeom& G, const CtWs& W, int st, int b, int p, int* out) {
    int n = 0;
    const int nk = G.keys_of(st);
    for (int k = 0; k <= nk; ++k) {
        const int id = k < nk ? W.lab[((int64_t)G.plane_type(st, k) * G.B + b) * G.px + p]
                              : W.fillmap[((int64_t)st * G.B + b) * G.px + p];
        if (id < 0) continue;
        const int r = uf_find(W.parent, id);
        bool seen = false;
        for (int j = 0; j < n; ++j) seen |= out[j] == r;
        if (!seen) out[n++] = r;
    }
    return n;
}
__global__ void __launch_bounds__(256) ct_pairs_kernel(const __grid_constant__ CtGeom G, const __grid_constant__ CtWs W, int round, int pass) {
    int32_t* ctl = W.ctl + round * CTL_STRIDE;
    // pass 0: whenever the round is active; pass 1: only when pass 0 both joined groups (boxes grew) and held a pair back
    if (!ct_round_active(W, round)) return;
    if (pass == 1 && !(((volatile int32_t*)ctl)[CTL_CHANGED1] && ((volatile int32_t*)ctl)[CTL_DEFERRED1])) return;
    const int total = G.n_seg_types() * G.B * G.px;
    for (int i = blockIdx.x * 256 + threadIdx.x; i < total; i += gridDim.x * 256) {
        const int seg = i / G.px, p = i - seg * G.px;
        const int st = seg / G.B, b = seg - st * G.B, nk = G.keys_of(st);
        if (nk < 2) continue;                            // a single key is never merged (base_cluster_based...:209)
        int covered = W.fillmap[i] >= 0;
        for (int k = 0; k < nk; ++k) covered += W.lab[((int64_t)G.plane_type(st, k) * G.B + b) * G.px + p] >= 0;
        if (covered < 2) continue;                       // most pixels: nothing to pair, no find
        int g[CT_MAX_KEYS + 1];
        const int n = ct_cover(G, W, st, b, p, g);
        for (int a = 0; a < n; ++a)
            for (int c = a + 1; c < n; ++c) {
                if (!ct_strict(W, g[a], g[c])) { if (pass == 0) ctl[CTL_DEFERRED1] = 1; }    // may pass once the boxes have grown
                else if (uf_unite(W.parent, g[a], g[c])) ctl[pass == 0 ? CTL_CHANGED1 : CTL_CHANGED2] = 1;
            }
    }
}
// does the box pass after pairs pass `pass` of `round` have anything to do?  (round < 0: unconditional)
__device__ __forceinline__ bool ct_boxes_needed(const CtWs& W, int round, int pass) {
    if (round < 0) return true;
    if (!ct_round_active(W, round)) return false;
    const volatile int32_t* ctl = W.ctl + round * CTL_STRIDE;
    return pass == 0 ? ctl[CTL_CHANGED1] != 0 : (ctl[CTL_CHANGED1] != 0 && ctl[CTL_DEFERRED1] != 0);
}
__global__ void __launch_bounds__(256) ct_group_reset_kernel(const __grid_constant__ CtWs W, int round, int pass) {
    if (!ct_boxes_needed(W, round, pass)) return;
    const int n = min(W.ctr[CTR_SHAPES], W.cap);
    for (int i = blockIdx.x * 256 + threadIdx.x; i < n; i += gridDim.x * 256) {
        W.g_x0[i] = INT_MAX; W.g_y0[i] = INT_MAX; W.g_x1[i] = -1; W.g_y1[i] = -1; W.g_members[i] = 0;
    }
}
__global__ void __launch_bounds__(256) ct_group_accum_kernel(const __grid_constant__ CtWs W, int round, int pass) {
    if (!ct_boxes_needed(W, round, pass)) return;
    const int n = min(W.ctr[CTR_SHAPES], W.cap);
    for (int i = blockIdx.x * 256 + threadIdx.x; i < n; i += gridDim.x * 256) {
        const int r = uf_find(W.parent, i);
        if (r != i) W.parent[i] = r;
        atomicMin(&W.g_x0[r], W.sh_x0[i]); atomicMin(&W.g_y0[r], W.sh_y0[i]);
        atomicMax(&W.g_x1[r], W.sh_x1[i]); atomicMax(&W.g_y1[r], W.sh_y1[i]);
        atomicAdd(&W.g_members[r], 1);
    }
}
// merged groups whose hole fill is out of date: small windows from the front of the list, large ones from its end (they
// get bigger blocks)
constexpr int CT_BIG_WINDOW = 96 * 96;
__global__ void __launch_bounds__(256) ct_list_groups_kernel(const __grid_constant__ CtWs W, int round) {
    if (!ct_round_active(W, round)) return;
    int32_t* ctl = W.ctl + round * CTL_STRIDE;
    if (round > 0 && !((volatile int32_t*)ctl)[CTL_CHANGED1]) return;      // no group changed: every fill is up to date
    const int n = min(W.ctr[CTR_SHAPES], W.cap);
    for (int i = blockIdx.x * 256 + threadIdx.x; i < n; i += gridDim.x * 256)
        if (W.parent[i] == i && W.g_members[i] > 1 && W.g_filled[i] != W.g_members[i]) {
            const bool big = (W.g_x1[i] - W.g_x0[i] + 3) * (W.g_y1[i] - W.g_y0[i] + 3) > CT_BIG_WINDOW;
            if (big) W.glist[W.cap - 1 - atomicAdd(&ctl[CTL_GLIST_BIG], 1)] = i;
            else W.glist[atomicAdd(&ctl[CTL_GLIST], 1)] = i;
        }
}

// occluded fill inside a word: bits of `s` spread through the runs of `f` (Kogge-Stone, both directions)
__device__ __forceinline__ uint32_t ct_spread(uint32_t s, uint32_t f) {
    uint32_t g = s, p = f;
    g |= p & (g << 1); p &= p << 1;
    g |= p & (g << 2); p &= p << 2;
    g |= p & (g << 4); p &= p << 4;
    g |= p & (g << 8); p &= p << 8;
    g |= p & (g << 16);
    uint32_t h = s; p = f;
    h |= p & (h >> 1); p &= p >> 1;
    h |= p & (h >> 2); p &= p >> 2;
    h |= p & (h >> 4); p &= p >> 4;
    h |= p & (h >> 8); p &= p >> 8;
    h |= p & (h >> 16);
    return g | h;
}

// One block per merged group: the union U of its members over the bounding box grown by one pixel, as a bitmask in shared
// memory; flood of the free pixels from the window's rim; what the flood does not reach and U does not cover is hole.
// Writes the holes to the fill map and the filled group's pixel count and chain length.
// Windows whose two bitmasks exceed the shared memory of the launch (image sizes above ~830: only the few groups that span
// most of such an image) keep them in a per-block slice of the workspace instead (W.scratch; the sweeps then run out of
// L2).  A window wider than 1024 pixels (32 word columns, one per lane) drops its left / right rim columns and seeds the
// free pixels of its first / last column instead: a reached rim column next to them is all the rim ever contributes.
template <int NT, bool BIG>
__global__ void __launch_bounds__(NT) ct_group_fill_kernel(const __grid_constant__ CtGeom G, const __grid_constant__ CtWs W, int round, int smem_words) {
    extern __shared__ uint32_t ct_sm[];
    __shared__ int red[3];
    constexpr int NW = NT / 32;
    int32_t* ctl = W.ctl + round * CTL_STRIDE;
    const int n_list = ((volatile int32_t*)ctl)[BIG ? CTL_GLIST_BIG : CTL_GLIST], tid = threadIdx.x;
    for (int gi = blockIdx.x; gi < n_list; gi += gridDim.x) {
    __syncthreads();                                     // the previous group's bitmasks and sums are no longer read
    const int g = W.glist[BIG ? W.cap - 1 - gi : gi];
    const int seg = W.sh_seg[g], st = seg / G.B, b = seg - st * G.B, nk = G.keys_of(st);
    const int rimx = (W.g_x1[g] - W.g_x0[g] + 3 > 1024) ? 0 : 1;
    const int x0 = W.g_x0[g] - rimx, y0 = W.g_y0[g] - 1;
    const int ww = W.g_x1[g] - W.g_x0[g] + 1 + 2 * rimx, hh = W.g_y1[g] - W.g_y0[g] + 3, wpr = (ww + 31) >> 5, words = hh * wpr;
    uint32_t* U = (BIG && 2 * words > smem_words) ? W.scratch + (size_t)blockIdx.x * W.scratch_words : ct_sm;
    uint32_t* R = U + words;
    if (tid < 3) red[tid] = 0;
    // U: one word per warp step, lane = pixel (coalesced label reads of every key, one ballot per word)
    for (int w0 = tid >> 5; w0 < words; w0 += 2 * NW) {
        uint32_t ub[2];
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int w = w0 + j * NW;
            bool in = false;
            if (w < words) {
                const int row = w / wpr, wc = w - row * wpr, xw = wc * 32 + (tid & 31);
                if (row > 0 && row < hh - 1 && xw >= rimx && xw < ww - rimx) {
                    const int p = (y0 + row) * G.S + x0 + xw;
                    int ids[CT_MAX_KEYS];
#pragma unroll
                    for (int k = 0; k < CT_MAX_KEYS; ++k)
                        ids[k] = k < nk ? W.lab[((int64_t)G.plane_type(st, k) * G.B + b) * G.px + p] : -1;
#pragma unroll
                    for (int k = 0; k < CT_MAX_KEYS; ++k) in |= ids[k] >= 0 && uf_find(W.parent, ids[k]) == g;
                }
            }
            ub[j] = __ballot_sync(0xffffffffu, in);
        }
        if ((tid & 31) == 0) {
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int w = w0 + j * NW;
                if (w >= words) continue;
                const int row = w / wpr, wc = w - row * wpr;
                const int nbits = min(32, ww - wc * 32);
                const uint32_t valid = nbits == 32 ? 0xffffffffu : ((1u << nbits) - 1u);
                uint32_t r = 0;
                if (row == 0 || row == hh - 1) r = valid;      // the rim is free and reached
                else {
                    if (wc == 0) r |= 1u;
                    if (wc == wpr - 1) r |= 1u << ((ww - 1) & 31);
                    if (!rimx) r &= ~ub[j];                    // no rim columns: the free pixels of the edge columns are the seeds
                }
                U[w] = ub[j];
                R[w] = r;
            }
        }
    }
    __syncthreads();
    // Flood, lane = word column (wpr <= 32), one band of rows per warp: a sweep walks the band's rows in order, each row
    // taking the reach of the row before it and closing it sideways (inside the words by ct_spread, across words by
    // shuffles), so reach travels the whole band per sweep however often it turns sideways; every warp sweeps its band
    // down and up, then the bands exchange their rim rows through the barrier, until nothing changes.  (Row-parallel
    // iterations move reach one row per block-wide barrier: 1.7 ms for a window of 258^2.)
    {
        const int lane = tid & 31, warp = tid >> 5;
        const bool act = lane < wpr;
        const int nbits = act ? min(32, ww - lane * 32) : 0;
        const uint32_t valid = nbits == 32 ? 0xffffffffu : (nbits > 0 ? (1u << nbits) - 1u : 0u);
        const int band = (hh + NW - 1) / NW, r0 = warp * band, r1 = min(hh, r0 + band);       // rows [r0, r1)
        int again;
        do {
            bool mine = false;
            for (int dir = 0; dir < 2 && r0 < r1; ++dir) {
                const int step = dir ? -1 : 1, first = dir ? r1 - 1 : r0, before = first - step;
                uint32_t prev = (act && before >= 0 && before < hh) ? ((volatile uint32_t*)R)[before * wpr + lane] : 0u;
                for (int row = first; row >= r0 && row < r1; row += step) {
                    const uint32_t f = act ? (~U[row * wpr + lane] & valid) : 0u, r = act ? R[row * wpr + lane] : 0u;
                    uint32_t sres = (r | prev) & f;
                    while (true) {
                        sres = ct_spread(sres, f);
                        const uint32_t fl = __shfl_up_sync(0xffffffffu, sres, 1), fr = __shfl_down_sync(0xffffffffu, sres, 1);
                        uint32_t t = sres;
                        if (lane > 0) t |= (fl >> 31) & f;
                        if (lane < 31) t |= (fr << 31) & f;
                        const bool grew = t != sres;
                        sres = t;
                        if (!__any_sync(0xffffffffu, grew)) break;
                    }
                    if (sres != r) { R[row * wpr + lane] = sres; mine = true; }
                    prev = sres;
                }
            }
            again = __syncthreads_or(mine ? 1 : 0);
        } while (again);
    }
    // filled shape F = everything the flood did not reach
    int cnt = 0, L = 0, fresh = 0;
    int32_t* fm = W.fillmap + (int64_t)seg * G.px;
    auto Fw = [&](int row, int wc) -> uint32_t {
        if (row < 0 || row >= hh || wc < 0 || wc >= wpr) return 0u;
        const int nbits = min(32, ww - wc * 32);
        const uint32_t valid = nbits == 32 ? 0xffffffffu : ((1u << nbits) - 1u);
        return ~R[row * wpr + wc] & valid;
    };
    for (int w = tid; w < words; w += NT) {
        const int row = w / wpr, wc = w - row * wpr;
        const uint32_t F = Fw(row, wc);
        if (!F) continue;
        const uint32_t up = Fw(row - 1, wc), dn = Fw(row + 1, wc);
        const uint32_t lf = (F << 1) | (Fw(row, wc - 1) >> 31), rt = (F >> 1) | (Fw(row, wc + 1) << 31);
        const uint32_t ul = (up << 1) | (Fw(row - 1, wc - 1) >> 31), ur = (up >> 1) | (Fw(row - 1, wc + 1) << 31);
        const uint32_t dl = (dn << 1) | (Fw(row + 1, wc - 1) >> 31), dr = (dn >> 1) | (Fw(row + 1, wc + 1) << 31);
        cnt += __popc(F);
        L += __popc(F & ~up) + __popc(F & ~dn) + __popc(F & ~lf) + __popc(F & ~rt);
        L -= __popc(F & ~up & ~lf & ~ul) + __popc(F & ~up & ~rt & ~ur) + __popc(F & ~dn & ~lf & ~dl) + __popc(F & ~dn & ~rt & ~dr);
        uint32_t hole = F & ~U[w];
        while (hole) {
            const int i = __ffs(hole) - 1;
            hole &= hole - 1;
            const int p = (y0 + row) * G.S + x0 + wc * 32 + i;
            const int old = fm[p];
            if (old < 0 || uf_find(W.parent, old) != g) ++fresh;
            fm[p] = g;
        }
    }
    atomicAdd(&red[0], cnt); atomicAdd(&red[1], L); atomicAdd(&red[2], fresh);
    __syncthreads();
    if (tid == 0) {
        W.g_cnt[g] = red[0]; W.g_L[g] = red[1]; W.g_filled[g] = W.g_members[g];
        if (red[2]) ctl[CTL_FILL_NEW] = 1;
    }
    }
}

// ------------------------------------------------------------------------------------------------ decisions
// which groups survive merge_contours_of_same_class_from_different_images + drop_too_small_contours
__global__ void __launch_bounds__(256) ct_finalize_kernel(const __grid_constant__ CtGeom G, const __grid_constant__ CtWs W) {
    const int n = min(W.ctr[CTR_SHAPES], W.cap);
    for (int i = blockIdx.x * 256 + threadIdx.x; i < n; i += gridDim.x * 256) {
        if (W.parent[i] != i) continue;
        const int seg = W.sh_seg[i], st = seg / G.B, b = seg - st * G.B, nk = G.keys_of(st);
        bool valid = true;                                // a class with no contour in one of the keys is dropped (:241-245)
        for (int k = 0; k < nk; ++k) valid &= W.key_count[G.plane_type(st, k) * G.B + b] > 0;
        const int members = W.g_members[i];
        if (members == 1) { W.g_cnt[i] = W.sh_cnt[i]; W.g_L[i] = W.sh_L[i]; }
        const bool keep_overlap = st < G.n_cls ? G.only_keep_overlapping != 0 : true;     // fine-grained: always (:334-349)
        const bool merged_ok = nk == 1 || members > 1 || !keep_overlap;
        const bool big = (double)(2 * (int64_t)W.g_cnt[i] - W.g_L[i] - 2) >= G.min_area2;
        W.g_kept[i] = st < G.n_cls ? (valid && merged_ok && big) : (valid && merged_ok);
    }
}
// classify_fine_grained_contours' overlap sums: score[fine group][class] += 1 per common pixel with a kept region of the
// class whose bounding box strictly overlaps the fine group's
__global__ void __launch_bounds__(256) ct_classify_kernel(const __grid_constant__ CtGeom G, const __grid_constant__ CtWs W) {
    const int total = G.B * G.px;
    for (int i = blockIdx.x * 256 + threadIdx.x; i < total; i += gridDim.x * 256) {
        const int b = i / G.px, p = i - b * G.px;
        int fg[CT_MAX_KEYS + 1], rg[CT_MAX_KEYS + 1];
        const int nf = ct_cover(G, W, G.n_cls, b, p, fg);
        if (!nf) continue;
        for (int c = 0; c < G.n_cls; ++c) {
            const int nr = ct_cover(G, W, c, b, p, rg);
            for (int a = 0; a < nf; ++a) {
                if (!W.g_kept[fg[a]]) continue;
                for (int r = 0; r < nr; ++r)
                    if (W.g_kept[rg[r]] && ct_strict(W, fg[a], rg[r])) {
                        // neighbouring pixels mostly add to the same (group, class): one atomic per warp and target
                        const int key = fg[a] * G.n_cls + c;
                        const unsigned same = __match_any_sync(__activemask(), key);
                        if ((threadIdx.x & 31) == __ffs(same) - 1) atomicAdd(&W.score[key], __popc(same));
                    }
            }
        }
    }
}
__global__ void __launch_bounds__(256) ct_assign_kernel(const __grid_constant__ CtGeom G, const __grid_constant__ CtWs W) {
    const int n = min(W.ctr[CTR_SHAPES], W.cap);
    for (int i = blockIdx.x * 256 + threadIdx.x; i < n; i += gridDim.x * 256) {
        if (W.parent[i] != i || !W.g_kept[i]) continue;
        const int seg = W.sh_seg[i], st = seg / G.B, b = seg - st * G.B;
        if (st != G.n_cls) continue;
        int best = -1, best_score = 0;                    // strict >: the first maximum in colour-map order wins (:371-384)
        for (int c = 0; c < G.n_cls; ++c) {
            const int s = W.score[(int64_t)i * G.n_cls + c];
            if (s > best_score) { best = c; best_score = s; }
        }
        const bool big = (double)(2 * (int64_t)W.g_cnt[i] - W.g_L[i] - 2) >= G.min_area2;
        if (best < 0 || !big) continue;
        W.g_cls[i] = best;
        atomicAdd(&W.img_kept[b * G.n_cls + best], 1);
        if (W.g_x1[i] - W.g_x0[i] + 1 > G.limit && W.g_y1[i] - W.g_y0[i] + 1 > G.limit) atomicAdd(&W.img_huge[b * G.n_cls + best], 1);
    }
}
// render_segmentation_image + determine_images_to_drop
__global__ void __launch_bounds__(256) ct_render_kernel(const __grid_constant__ CtGeom G, const __grid_constant__ CtWs W, uint8_t* __restrict__ out, int32_t* __restrict__ flags) {
    const int total = G.B * G.px;
    const uint8_t* ink_plane = G.planes[G.n_cls * G.n_det + G.n_fine - 1];
    for (int i = blockIdx.x * 256 + threadIdx.x; i < total; i += gridDim.x * 256) {
        const int b = i / G.px, p = i - b * G.px;
        int cls = -1;
        if (ink_plane[i]) {
            int fg[CT_MAX_KEYS + 1];
            const int nf = ct_cover(G, W, G.n_cls, b, p, fg);
            for (int a = 0; a < nf; ++a) {
                const int c = W.g_cls[fg[a]];
                if (c >= 0 && (cls < 0 || G.render_rank[c] > G.render_rank[cls])) cls = c;
            }
        }
        const uint8_t* col = G.colors + 3 * (cls + 1);
        out[3 * i] = col[0]; out[3 * i + 1] = col[1]; out[3 * i + 2] = col[2];
        if (p == 0) {
            // the reference looks at the FIRST contour of each class: decided here when every contour of the class agrees
            bool certain = false, undecided = false;
            for (int c = 0; c < G.n_cls; ++c) {
                const int huge = W.img_huge[b * G.n_cls + c], kept = W.img_kept[b * G.n_cls + c];
                certain |= huge > 0 && huge == kept;
                undecided |= huge > 0 && huge != kept;
            }
            const bool settled = !ct_round_active(W, CT_ROUNDS) && !W.ctr[CTR_OVERFLOW];
            flags[b] = !settled ? 2 : certain ? 1 : undecided ? 2 : 0;       // a certain drop in one class decides the image
        }
    }
}
// [shapes, rounds that did something, why the batch was handed to the host (0: it was not, 1: capacity, 3: fixpoint still moving)]
__global__ void ct_info_kernel(const __grid_constant__ CtWs W, int32_t* info) {
    int rounds = 0;
    for (int o = 0; o < CT_ROUNDS; ++o) rounds += ct_round_active(W, o) && (o == 0 || W.ctl[o * CTL_STRIDE + CTL_CHANGED1] || W.ctl[(o - 1) * CTL_STRIDE + CTL_FILL_NEW]);
    info[0] = W.ctr[CTR_SHAPES];
    info[1] = rounds;
    info[2] = W.ctr[CTR_OVERFLOW] ? 1 : ct_round_active(W, CT_ROUNDS) ? 3 : 0;
}
constexpr int CT_FILL_SMEM_MAX = 200 * 1024;
struct CtLayout {
    int64_t lab, aux, fillmap, key_count, fmask, touch, shapes, ctr, img, scratch, total;
    int scratch_words;
    int cap;
};
static CtLayout ct_layout(int B, int S, int n_cls, int n_det, int n_fine) {
    CtLayout L;
    const int64_t px = (int64_t)S * S, np = (int64_t)(n_cls * n_det + n_fine) * B, ns = (int64_t)(n_cls + 1) * B;
    auto up = [](int64_t v) { return (v + 255) / 256 * 256; };
    int64_t off = 0;
    L.lab = off; off += up(np * px * 4);
    L.aux = off; off += up(np * px * 4);
    L.fillmap = off; off += up(ns * px * 4);
    L.fmask = off; off += up(np * px);
    L.touch = off; off += up(np * px);
    L.key_count = off; off += up(np * 4);
    // two shapes of a plane are never 8-adjacent, so a plane holds at most S^2/4; 16 k per plane is far above what masks
    // produce (overflow marks the whole batch for the host path)
    const int64_t per_plane = px / 4 < 16384 ? px / 4 : 16384;
    L.cap = (int)(np * per_plane);
    L.shapes = off; off += up((int64_t)L.cap * 4) * (20 + n_cls);
    L.ctr = off; off += up((CTR_NUM + (CT_ROUNDS + 1) * CTL_STRIDE) * 4);
    L.img = off; off += up((int64_t)B * n_cls * 4) * 2;
    // big-window bitmasks that do not fit in shared memory: one slice per block of the (one block per SM) big-window launch
    const int64_t wmax = S + 2, mask_words = 2 * wmax * ((wmax + 31) / 32);
    L.scratch_words = mask_words * 4 > CT_FILL_SMEM_MAX ? (int)mask_words : 0;
    L.scratch = off; off += up((int64_t)L.scratch_words * 4) * kNumSMs;
    L.total = off;
    return L;
}

}  // namespace sis

using namespace sis;

extern "C" int sis_contour_stage_workspace_bytes(int batch, int size, int n_classes, int n_det_keys, int n_fine_keys, int64_t* bytes) {
    SIS_REQUIRE(bytes != nullptr, "contour stage: null output");
    SIS_REQUIRE(batch > 0 && size > 0 && n_classes > 0 && n_det_keys > 0 && n_fine_keys > 0, "contour stage: sizes must be positive");
    *bytes = ct_layout(batch, size, n_classes, n_det_keys, n_fine_keys).total;
    return SIS_OK;
}

extern "C" int sis_contour_stage(const uint8_t* const* d_det_masks, const uint8_t* const* d_fine_masks, int batch, int size,
                                 int n_classes, int n_det_keys, int n_fine_keys, int fine_class, int only_keep_overlapping,
                                 double min_class_contour_area, const uint8_t* colors_rgb, const int* render_rank,
                                 void* d_workspace, int64_t workspace_bytes, uint8_t* d_label_rgb, int32_t* d_flags,
                                 int32_t* d_info, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    SIS_REQUIRE(batch > 0 && size > 0, "contour stage: batch and image size must be positive");
    SIS_REQUIRE(n_classes >= 1 && n_classes <= CT_MAX_CLASSES, "contour stage: 1..%d classes besides the background (got %d)", CT_MAX_CLASSES, n_classes);
    SIS_REQUIRE(n_det_keys >= 1 && n_det_keys <= CT_MAX_KEYS && n_fine_keys >= 1 && n_fine_keys <= CT_MAX_KEYS,
                "contour stage: 1..%d keys per stage", CT_MAX_KEYS);
    SIS_REQUIRE(n_classes * n_det_keys + n_fine_keys <= CT_MAX_PLANE_TYPES, "contour stage: too many mask planes");
    SIS_REQUIRE(fine_class >= 0 && fine_class < n_classes, "contour stage: fine-grained class index out of range");
    SIS_REQUIRE(d_det_masks && d_fine_masks && colors_rgb && render_rank && d_workspace && d_label_rgb && d_flags,
                "contour stage: masks, outputs and workspace must be CUDA tensors (null pointer)");
    const CtLayout L = ct_layout(batch, size, n_classes, n_det_keys, n_fine_keys);
    SIS_REQUIRE(workspace_bytes >= L.total, "contour stage: workspace of %lld bytes, %lld needed", (long long)workspace_bytes, (long long)L.total);
    CtGeom G;
    G.B = batch; G.S = size; G.n_cls = n_classes; G.n_det = n_det_keys; G.n_fine = n_fine_keys; G.fine_cls = fine_class;
    G.px = size * size; G.only_keep_overlapping = only_keep_overlapping; G.limit = (int)(size * 0.95);
    G.min_area2 = 2.0 * min_class_contour_area;
    for (int t = 0; t < n_classes * n_det_keys; ++t) {
        SIS_REQUIRE(d_det_masks[t] != nullptr, "contour stage: null class-determination mask plane %d", t);
        G.planes[t] = d_det_masks[t];
    }
    for (int k = 0; k < n_fine_keys; ++k) {
        SIS_REQUIRE(d_fine_masks[k] != nullptr, "contour stage: null fine-grained mask plane %d", k);
        G.planes[n_classes * n_det_keys + k] = d_fine_masks[k];
    }
    for (int i = 0; i < (n_classes + 1) * 3; ++i) G.colors[i] = colors_rgb[i];
    for (int c = 0; c < n_classes; ++c) G.render_rank[c] = render_rank[c];

    char* base = (char*)d_workspace;
    CtWs W;
    W.lab = (int32_t*)(base + L.lab); W.aux = (int32_t*)(base + L.aux); W.fillmap = (int32_t*)(base + L.fillmap);
    W.fmask = (uint8_t*)(base + L.fmask); W.touch = (uint8_t*)(base + L.touch); W.key_count = (int32_t*)(base + L.key_count);
    W.cap = L.cap;
    const int64_t stride = ((int64_t)L.cap * 4 + 255) / 256 * 256;
    int32_t** fields[] = {&W.sh_seg, &W.sh_cnt, &W.sh_L, &W.sh_x0, &W.sh_y0, &W.sh_x1, &W.sh_y1, &W.parent, &W.g_x0, &W.g_y0,
                          &W.g_x1, &W.g_y1, &W.g_members, &W.g_filled, &W.g_cnt, &W.g_L, &W.g_kept, &W.g_cls, &W.glist, &W.score};
    for (int i = 0; i < 20; ++i) *fields[i] = (int32_t*)(base + L.shapes + stride * i);      // score takes slots 19 .. 19+n_cls
    W.ctr = (int32_t*)(base + L.ctr);
    W.ctl = W.ctr + CTR_NUM;
    W.scratch = L.scratch_words ? (uint32_t*)(base + L.scratch) : nullptr;
    W.scratch_words = (int)(((int64_t)L.scratch_words * 4 + 255) / 256 * 64);
    W.img_kept = (int32_t*)(base + L.img);
    W.img_huge = W.img_kept + ((int64_t)batch * n_classes * 4 + 255) / 256 * 64;

    const int64_t np = (int64_t)G.n_plane_types() * batch, ns = (int64_t)G.n_seg_types() * batch;
    const int wmax = size + 2, fill_full = 2 * wmax * ((wmax + 31) / 32) * 4;
    const int fill_smem = fill_full <= CT_FILL_SMEM_MAX ? fill_full : 96 * 1024;          // larger windows go to W.scratch
    const int fill_smem_small = min(fill_smem, 2 * 4 * (CT_BIG_WINDOW / 32 + wmax + 8));    // words <= area/32 + rows
    SIS_REQUIRE(size <= 1024, "contour stage: image size %d not supported (a window row must fit 32 word columns: <= 1024)", size);
    SIS_REQUIRE((int64_t)(n_classes * n_det_keys + n_fine_keys) * batch * size * size < (int64_t)1 << 31,
                "contour stage: %d planes of %d^2 pixels exceed the 32-bit pixel index; split the batch", (n_classes * n_det_keys + n_fine_keys) * batch, size);
    static int fill_smem_set = 0;
    if (fill_smem > fill_smem_set) {
        SIS_CHECK_CUDA(cudaFuncSetAttribute(ct_group_fill_kernel<1024, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, fill_smem));
        fill_smem_set = fill_smem;
    }
    SIS_CHECK_CUDA(cudaMemsetAsync(W.fillmap, 0xff, ns * G.px * 4, stream));
    SIS_CHECK_CUDA(cudaMemsetAsync(W.key_count, 0, np * 4, stream));
    SIS_CHECK_CUDA(cudaMemsetAsync(W.ctr, 0, (char*)(base + L.scratch) - (char*)W.ctr, stream));    // counters, control words, per-image sums
    const int grid_px = (int)min((int64_t)kNumSMs * 16, ceil_div64(np * G.px, 256));
    const int grid_seg = (int)min((int64_t)kNumSMs * 16, ceil_div64(ns * G.px, 256));
    const int grid_img = (int)min((int64_t)kNumSMs * 16, ceil_div64((int64_t)batch * G.px, 256));
    const int grid_sh = kNumSMs * 4;       // the shape-table kernels size their loops from the device counter
    ct_bg_init_kernel<<<grid_px, 256, 0, stream>>>(G, W); SIS_CHECK_LAUNCH();
    ct_bg_merge_kernel<<<grid_px, 256, 0, stream>>>(G, W); SIS_CHECK_LAUNCH();
    ct_bg_touch_kernel<<<(int)min((int64_t)kNumSMs * 8, ceil_div64(np * 4 * size, 256)), 256, 0, stream>>>(G, W); SIS_CHECK_LAUNCH();
    ct_fg_init_kernel<<<grid_px, 256, 0, stream>>>(G, W); SIS_CHECK_LAUNCH();
    ct_fg_merge_kernel<<<grid_px, 256, 0, stream>>>(G, W); SIS_CHECK_LAUNCH();
    ct_fg_ids_kernel<<<grid_px, 256, 0, stream>>>(G, W); SIS_CHECK_LAUNCH();
    ct_shape_stats_kernel<<<grid_px, 256, 0, stream>>>(G, W); SIS_CHECK_LAUNCH();
    ct_group_reset_kernel<<<grid_sh, 256, 0, stream>>>(W, -1, 0); SIS_CHECK_LAUNCH();
    ct_group_accum_kernel<<<grid_sh, 256, 0, stream>>>(W, -1, 0); SIS_CHECK_LAUNCH();
    if (n_det_keys > 1 || n_fine_keys > 1) {
        // No host round trip: CT_ROUNDS rounds are enqueued, each kernel decides on the device whether it still has work
        // (a round whose predecessor changed nothing returns in a few microseconds).
        for (int o = 0; o < CT_ROUNDS; ++o) {
            for (int pass = 0; pass < 2; ++pass) {
                ct_pairs_kernel<<<grid_seg, 256, 0, stream>>>(G, W, o, pass); SIS_CHECK_LAUNCH();
                ct_group_reset_kernel<<<grid_sh, 256, 0, stream>>>(W, o, pass); SIS_CHECK_LAUNCH();
                ct_group_accum_kernel<<<grid_sh, 256, 0, stream>>>(W, o, pass); SIS_CHECK_LAUNCH();
            }
            ct_list_groups_kernel<<<grid_sh, 256, 0, stream>>>(W, o); SIS_CHECK_LAUNCH();
            ct_group_fill_kernel<128, false><<<kNumSMs * 8, 128, fill_smem_small, stream>>>(G, W, o, fill_smem_small / 4); SIS_CHECK_LAUNCH();
            ct_group_fill_kernel<1024, true><<<kNumSMs, 1024, fill_smem, stream>>>(G, W, o, fill_smem / 4); SIS_CHECK_LAUNCH();
        }
    }
    ct_finalize_kernel<<<grid_sh, 256, 0, stream>>>(G, W); SIS_CHECK_LAUNCH();
    ct_classify_kernel<<<grid_img, 256, 0, stream>>>(G, W); SIS_CHECK_LAUNCH();
    ct_assign_kernel<<<grid_sh, 256, 0, stream>>>(G, W); SIS_CHECK_LAUNCH();
    ct_render_kernel<<<grid_img, 256, 0, stream>>>(G, W, d_label_rgb, d_flags); SIS_CHECK_LAUNCH();
    if (d_info) { ct_info_kernel<<<1, 1, 0, stream>>>(W, d_info); SIS_CHECK_LAUNCH(); }
    return SIS_OK;
}
