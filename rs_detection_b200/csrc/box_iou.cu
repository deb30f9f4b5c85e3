// box_iou.cu -- pairwise rotated IoU matrix + MaxIoU assignment (compile with -fmad=false).
//
// Replaces box_iou_rotated_cuda_kernel (python/jdet/ops/box_iou_rotated.py:413-461, v1 copy
// box_iou_rotated_v1.py:418-466) and the Python body of MaxIoUAssigner.assign_wrt_overlaps
// (python/jdet/models/boxes/assigner.py:111-170).  Also the horizontal BboxOverlaps2D matrix and the RPN's anchor
// assignment fused with it (rsdet_assign_hbb), which never stores the (num_gts, n) matrix.
//
// Kernel plan (FP32-ALU bound; no tensor cores -- nothing here is a contraction):
//   prep  : one thread per box -> RBox (double sin/cos once per box, not once per pair)
//   tiles : 64x64 IoU tile per CTA iteration, 128 threads.  Stage 1 runs the bounding-circle test on
//           all 4096 pairs (coalesced zero stores for the rejects; hits in a register bit mask, compacted
//           once per tile); stage 2 runs the separating-axis test densely on the survivors; stage 3 hands
//           ONE remaining pair to each thread, so the heavy clipper runs on dense warps instead of the
//           reference's 1-in-10 active lanes.
#include "common.cuh"
#include "rotated_iou.cuh"

namespace rsdet {

constexpr int kTile = 64;
constexpr int kIouThreads = 128;

__global__ void prep_rbox_kernel(const float* __restrict__ boxes, int n, int version, int zero_tiny, RBox* __restrict__ out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* b = boxes + (size_t)i * 5;
    RBox r = prep_rbox(b, version);
    // box_iou_rotated_v1.py:515-522: boxes with a side < 1e-3 give IoU 0 with everything
    if (zero_tiny && fminf(b[2], b[3]) < 0.001f) r.r = -1e30f;
    out[i] = r;
}

__global__ void __launch_bounds__(kIouThreads)
box_iou_tiles_kernel(const RBox* __restrict__ rows, int n1, const RBox* __restrict__ cols, int n2, float* __restrict__ out) {
    __shared__ RBox s_row[kTile];
    __shared__ RBox s_col[kTile];
    __shared__ unsigned short s_queue[kTile * kTile];
    constexpr int kQ2 = 1024;
    __shared__ unsigned short s_queue2[kQ2];
    __shared__ float2 s_pts[24 * kIouThreads];
    __shared__ int s_wsum[kIouThreads / 32];
    __shared__ int s_count;
    __shared__ int s_count2;

    const int tiles_x = ceil_div(n2, kTile);
    const int tiles_y = ceil_div(n1, kTile);
    const long long total = (long long)tiles_x * tiles_y;
    const int tid = threadIdx.x, lane = tid & 31;

    for (long long t = blockIdx.x; t < total; t += gridDim.x) {
        const int r0 = (int)(t / tiles_x) * kTile, c0 = (int)(t % tiles_x) * kTile;
        const int nr = min(kTile, n1 - r0), nc = min(kTile, n2 - c0);
        __syncthreads();  // previous iteration done with smem
        if (tid < kTile) {
            if (tid < nr) s_row[tid] = rows[r0 + tid];
        } else {
            int c = tid - kTile;
            if (c < nc) {
                s_col[c] = cols[c0 + c];
            }
        }
        __syncthreads();

        // stage 1: bounding circles on all 4096 pairs.  Thread = (column, row parity); hits go to a register
        // bit mask, the rejects get their zeros (a warp covers 32 consecutive columns of one row: coalesced),
        // and the hits are compacted once per tile (a ballot + atomic per 32 pairs costs more than the test).
        {
            const int c = tid & 63, rhalf = tid >> 6;
            unsigned hits = 0u;
            if (c < nc) {
                const float cx = s_col[c].x, cy = s_col[c].y, cr = s_col[c].r;
#pragma unroll 8
                for (int k = 0; k < 32; k++) {
                    const int r = 2 * k + rhalf;
                    if (r < nr) {
                        const float rs = s_row[r].r + cr, dx = s_row[r].x - cx, dy = s_row[r].y - cy;
                        const bool cand = (rs >= 0.f) && !(dx * dx + dy * dy > rs * rs);  // == rbox_may_overlap
                        hits |= (cand ? 1u : 0u) << k;
                        if (!cand) out[(size_t)(r0 + r) * n2 + c0 + c] = 0.f;
                    }
                }
            }
            const int mine = __popc(hits);
            int incl = mine;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int y = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += y;
            }
            if (lane == 31) s_wsum[tid >> 5] = incl;
            __syncthreads();
            int pos = incl - mine;
            for (int w = 0; w < (tid >> 5); w++) pos += s_wsum[w];
            if (tid == kIouThreads - 1) s_count = pos + mine;
            while (hits) {
                const int k = __ffs(hits) - 1;
                hits &= hits - 1;
                s_queue[pos++] = (unsigned short)(((2 * k + rhalf) << 6) | c);
            }
        }
        __syncthreads();

        // stage 2 (dense over the circle survivors): separating axes in both box frames -> exact zeros;
        // stage 3: one surviving pair per thread through the exact clipper
        const int cnt = s_count;
        for (int q0 = 0; q0 < cnt; q0 += kQ2) {
            const int qn = min(kQ2, cnt - q0);
            if (tid == 0) s_count2 = 0;
            __syncthreads();
            for (int qi = tid; qi < ((qn + 31) & ~31); qi += kIouThreads) {
                int p = 0;
                bool live = qi < qn;
                if (live) {
                    p = s_queue[q0 + qi];
                    live = rbox_inter_upper_bound(s_row[p >> 6], s_col[p & 63]) > 0.f;
                    if (!live) out[(size_t)(r0 + (p >> 6)) * n2 + c0 + (p & 63)] = 0.f;
                }
                const unsigned m = __ballot_sync(0xffffffffu, live);
                if (m) {
                    int base = 0;
                    if (lane == 0) base = atomicAdd(&s_count2, __popc(m));
                    base = __shfl_sync(0xffffffffu, base, 0);
                    if (live) s_queue2[base + __popc(m & ((1u << lane) - 1))] = (unsigned short)p;
                }
            }
            __syncthreads();
            const int cnt2 = s_count2;
            for (int qi = tid; qi < cnt2; qi += kIouThreads) {
                const int p = s_queue2[qi];
                const int r = p >> 6, c = p & 63;
                out[(size_t)(r0 + r) * n2 + c0 + c] = rotated_iou_pair<kIouThreads>(s_row[r], s_col[c], s_pts + tid);
            }
            __syncthreads();
        }
    }
}

// ------------------------------------------------------------------ assignment
// row pass: per-gt max / argmax over proposals (one warp per gt)
__global__ void assign_row_max_kernel(const float* __restrict__ ov, int G, int n, float* __restrict__ gt_max, int* __restrict__ gt_argmax) {
    int g = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (g >= G) return;
    float best = -INFINITY;
    int bi = 0x7fffffff;
    for (int j = lane; j < n; j += 32) {
        float v = ov[(size_t)g * n + j];
        if (v > best) { best = v; bi = j; }
    }
    for (int o = 16; o; o >>= 1) {
        float ob = __shfl_xor_sync(0xffffffffu, best, o);
        int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (ob > best || (ob == best && oi < bi)) { best = ob; bi = oi; }
    }
    if (lane == 0) { gt_max[g] = best; gt_argmax[g] = bi == 0x7fffffff ? 0 : bi; }
}

// column pass: assigner.py:124-168
__global__ void assign_col_kernel(const float* __restrict__ ov, int G, int n, float pos_thr, float neg_lo, float neg_hi,
                                  float min_pos_iou, int match_low_quality, int assign_all,
                                  const float* __restrict__ gt_max, const int* __restrict__ gt_argmax,
                                  const int32_t* __restrict__ gt_labels, int32_t labels_fill,
                                  int32_t* __restrict__ gt_inds, float* __restrict__ max_ov, int32_t* __restrict__ labels) {
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    float best = -INFINITY;
    int bi = 0;
    int lowq = 0;
    for (int g = 0; g < G; g++) {
        float v = ov[(size_t)g * n + j];
        if (v > best) { best = v; bi = g; }
        if (match_low_quality) {
            float gm = gt_max[g];
            if (gm >= min_pos_iou && (assign_all ? (v == gm) : (gt_argmax[g] == j))) lowq = g + 1;
        }
    }
    int a = -1;
    if (best >= neg_lo && best < neg_hi) a = 0;
    if (best >= pos_thr) a = bi + 1;
    if (lowq) a = lowq;
    gt_inds[j] = a;
    if (max_ov) max_ov[j] = best;
    if (labels) labels[j] = (a > 0 && gt_labels) ? gt_labels[a - 1] : labels_fill;
}

// ------------------------------------------------------------------ horizontal IoU + fused anchor assignment
// BboxOverlaps2D, mode='iou', not aligned: the mmdet 2.x bbox_overlaps that JDet's models/boxes/iou_calculator.py copies.
// fp32, no "+1", every operation rounded on its own (this unit is built with -fmad=false).  NOT pinned by a fixture
// (DESIGN.md section 3): both kernels below call this one function so that a fixture can correct it in one place.
// A disjoint or touching pair gives +0.0 (never -0.0), so every finite IoU is >= +0.0; the fused assignment relies on it.
__device__ __forceinline__ float hbb_iou(float ax1, float ay1, float ax2, float ay2, float bx1, float by1, float bx2, float by2) {
    const float area_a = (ax2 - ax1) * (ay2 - ay1);
    const float area_b = (bx2 - bx1) * (by2 - by1);
    const float dw = fminf(ax2, bx2) - fmaxf(ax1, bx1);
    const float dh = fminf(ay2, by2) - fmaxf(ay1, by1);
    const float w = dw > 0.f ? dw : 0.f;
    const float h = dh > 0.f ? dh : 0.f;
    const float overlap = w * h;
    const float uni = fmaxf((area_a + area_b) - overlap, 1e-6f);
    return overlap / uni;
}

__device__ __forceinline__ float hbb_iou(float4 a, float4 b) { return hbb_iou(a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w); }

constexpr int kOvRows = 8;  // rows of the (n1, n2) matrix per CTA pass: one column box in registers serves 8 rows

__global__ void __launch_bounds__(256)
bbox_overlaps_kernel(const float* __restrict__ b1, int n1, const float* __restrict__ b2, int n2, float* __restrict__ out) {
    const int j = blockIdx.x * 256 + threadIdx.x;
    if (j >= n2) return;
    const float bx1 = b2[4 * (size_t)j], by1 = b2[4 * (size_t)j + 1], bx2 = b2[4 * (size_t)j + 2], by2 = b2[4 * (size_t)j + 3];
    for (int r0 = blockIdx.y * kOvRows; r0 < n1; r0 += gridDim.y * kOvRows) {
        const int r1 = min(r0 + kOvRows, n1);
        for (int r = r0; r < r1; r++) {
            const float* a = b1 + 4 * (size_t)r;
            out[(size_t)r * n2 + j] = hbb_iou(a[0], a[1], a[2], a[3], bx1, by1, bx2, by2);
        }
    }
}

// The fused MaxIoU assignment (rsdet_assign_hbb).  A CTA owns 256 consecutive anchors.  The anchors of one pyramid level
// are stored in (h, w, a) order, so a CTA's anchors form a thin strip of the image, and most GTs miss it.  A GT "misses"
// the strip when one of its edges lies beyond the strip's hull on the far side:
//     gx1 >= max(ax2) || gx2 <= min(ax1) || gy1 >= max(ay2) || gy2 <= min(ay1)
// Then for every anchor of the strip min(ax2, gx2) <= max(ax1, gx1) (or likewise on y), the difference is <= 0 in fp32
// too, and the IoU is exactly +0.0.  Skipping such a GT changes no decision of the CTA's anchors:
//   * column max / argmax: all IoUs are >= +0.0 and the first maximal GT wins, so starting from (+0.0, GT 0) instead of
//     (-inf, -) gives the same pair, also for a column whose GTs are all skipped (max +0.0, argmax 0);
//   * low-quality pass: a GT with gt_max > 0 matches only anchors with IoU == gt_max > 0 (its argmax anchor among them),
//     none of which is in a strip it misses.  A GT with gt_max == 0 >= min_pos_iou matches IoU-0 anchors, so such a GT
//     is never skipped.
// NaN coordinates widen the hull to +-inf and fail every comparison, so a GT is never skipped because of one.
constexpr int kHbbThreads = 256;
constexpr int kHbbChunk = 1024;  // GTs staged in shared memory per chunk

struct StripHull {
    float x1, y1, x2, y2;  // min x1, min y1, max x2, max y2 over the CTA's valid anchors
    int any;               // the CTA has a valid anchor
};

__device__ __forceinline__ float nan_to(float v, float to) { return v == v ? v : to; }

// Block-wide hull of the valid anchors; every thread gets the result.
__device__ StripHull strip_hull(bool live, float x1, float y1, float x2, float y2) {
    __shared__ float s_h[4][kHbbThreads / 32];
    __shared__ int s_any[kHbbThreads / 32];
    float a = live ? nan_to(x1, -INFINITY) : INFINITY, b = live ? nan_to(y1, -INFINITY) : INFINITY;
    float c = live ? nan_to(x2, INFINITY) : -INFINITY, d = live ? nan_to(y2, INFINITY) : -INFINITY;
    for (int o = 16; o; o >>= 1) {
        a = fminf(a, __shfl_xor_sync(0xffffffffu, a, o));
        b = fminf(b, __shfl_xor_sync(0xffffffffu, b, o));
        c = fmaxf(c, __shfl_xor_sync(0xffffffffu, c, o));
        d = fmaxf(d, __shfl_xor_sync(0xffffffffu, d, o));
    }
    const int anyw = __any_sync(0xffffffffu, live);
    const int w = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) { s_h[0][w] = a; s_h[1][w] = b; s_h[2][w] = c; s_h[3][w] = d; s_any[w] = anyw; }
    __syncthreads();
    StripHull h{INFINITY, INFINITY, -INFINITY, -INFINITY, 0};
    for (int k = 0; k < kHbbThreads / 32; k++) {
        h.x1 = fminf(h.x1, s_h[0][k]); h.y1 = fminf(h.y1, s_h[1][k]);
        h.x2 = fmaxf(h.x2, s_h[2][k]); h.y2 = fmaxf(h.y2, s_h[3][k]);
        h.any |= s_any[k];
    }
    return h;
}

__device__ __forceinline__ bool misses(const StripHull& h, float4 g) {
    return g.x >= h.x2 || g.z <= h.x1 || g.y >= h.y2 || g.w <= h.y1;
}

__device__ __forceinline__ float4 load_box(const float* __restrict__ p, size_t i) {
    return make_float4(p[4 * i], p[4 * i + 1], p[4 * i + 2], p[4 * i + 3]);
}

// gt_key[g] = max over valid anchors of (IoU bits << 32 | ~anchor): the largest IoU, then the first anchor.  Only IoUs
// > 0 are posted, so a key of 0 means gt_max = +0.0 with the first valid anchor as argmax.
__device__ __forceinline__ void decode_gt_key(unsigned long long key, unsigned first_valid, float& gm, int& ga) {
    const unsigned hi = (unsigned)(key >> 32);
    gm = __uint_as_float(hi);
    ga = hi ? (int)~(unsigned)key : (int)first_valid;
}

__global__ void assign_hbb_init_kernel(unsigned long long* __restrict__ gt_key, int G, unsigned* __restrict__ first_valid) {
    for (int g = blockIdx.x * blockDim.x + threadIdx.x; g < G; g += gridDim.x * blockDim.x) gt_key[g] = 0ull;
    if (blockIdx.x == 0 && threadIdx.x == 0) *first_valid = 0xffffffffu;
}

// Row pass (match_low_quality only): per-GT max / first argmax over the valid anchors.  The CTA stages its valid anchors
// in order; each thread takes whole GTs of the compacted non-missing list and scans the strip, so ties keep the first
// anchor without any reduction; one 64-bit atomicMax per (GT, CTA) with a positive maximum.
__global__ void __launch_bounds__(kHbbThreads)
assign_hbb_gt_max_kernel(const float* __restrict__ gts, int G, const float* __restrict__ anchors, int n,
                         const uint8_t* __restrict__ valid, unsigned long long* __restrict__ gt_key,
                         unsigned* __restrict__ first_valid) {
    __shared__ float4 s_anc[kHbbThreads];
    __shared__ int s_aidx[kHbbThreads];
    __shared__ int s_wcnt[kHbbThreads / 32];
    __shared__ float4 s_gt[kHbbChunk];
    __shared__ int s_gidx[kHbbChunk];
    __shared__ int s_ng;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int j = blockIdx.x * kHbbThreads + tid;
    const bool live = j < n && (!valid || valid[j]);
    const float4 a = j < n ? load_box(anchors, j) : make_float4(0.f, 0.f, 0.f, 0.f);
    const StripHull hull = strip_hull(live, a.x, a.y, a.z, a.w);
    if (!hull.any) return;

    // order-preserving compaction of the valid anchors
    const unsigned m = __ballot_sync(0xffffffffu, live);
    if (lane == 0) s_wcnt[wid] = __popc(m);
    __syncthreads();
    int base = 0, na = 0;
    for (int k = 0; k < kHbbThreads / 32; k++) {
        base += k < wid ? s_wcnt[k] : 0;
        na += s_wcnt[k];
    }
    const int pos = base + __popc(m & ((1u << lane) - 1));
    if (live) { s_anc[pos] = a; s_aidx[pos] = j; }
    if (live && pos == 0) atomicMin(first_valid, (unsigned)j);

    for (int c0 = 0; c0 < G; c0 += kHbbChunk) {
        const int cn = min(kHbbChunk, G - c0);
        if (tid == 0) s_ng = 0;
        __syncthreads();  // s_anc written
        for (int k = tid; k < cn; k += kHbbThreads) {
            const float4 g = load_box(gts, (size_t)(c0 + k));
            if (!misses(hull, g)) {
                const int p = atomicAdd(&s_ng, 1);  // the per-GT maxima do not depend on the list's order
                s_gt[p] = g;
                s_gidx[p] = c0 + k;
            }
        }
        __syncthreads();
        const int ng = s_ng;
        for (int k = tid; k < ng; k += kHbbThreads) {
            const float4 g = s_gt[k];
            float best = 0.f;
            int bi = -1;
            for (int q = 0; q < na; q++) {
                const float v = hbb_iou(g, s_anc[q]);
                if (v > best) { best = v; bi = q; }
            }
            if (bi >= 0)
                atomicMax(gt_key + s_gidx[k], ((unsigned long long)__float_as_uint(best) << 32) | (unsigned)~(unsigned)s_aidx[bi]);
        }
        __syncthreads();  // the list and s_ng fully read before the next chunk resets them
    }
}

// Column pass: one thread per anchor over the GTs that do not miss the CTA's strip, staged in chunks and in GT order
// (the first maximal GT wins the argmax, the last low-quality match wins).  The decisions are assign_col_kernel's.
__global__ void __launch_bounds__(kHbbThreads)
assign_hbb_col_kernel(const float* __restrict__ gts, int G, const float* __restrict__ anchors, int n,
                      const uint8_t* __restrict__ valid, float pos_thr, float neg_lo, float neg_hi, float min_pos_iou,
                      int match_low_quality, int assign_all, const unsigned long long* __restrict__ gt_key,
                      const unsigned* __restrict__ first_valid, const int32_t* __restrict__ gt_labels,
                      int32_t labels_fill, int32_t* __restrict__ gt_inds, float* __restrict__ max_ov,
                      int32_t* __restrict__ labels) {
    __shared__ float4 s_gt[kHbbChunk];
    __shared__ int s_gidx[kHbbChunk];
    __shared__ float s_gm[kHbbChunk];
    __shared__ int s_ga[kHbbChunk];
    __shared__ int s_wcnt[kHbbThreads / 32];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int j = blockIdx.x * kHbbThreads + tid;
    const bool live = j < n && (!valid || valid[j]);
    const float4 a = j < n ? load_box(anchors, j) : make_float4(0.f, 0.f, 0.f, 0.f);
    const StripHull hull = strip_hull(live, a.x, a.y, a.z, a.w);

    float best = 0.f;
    int bi = 0, lowq = 0;
    if (hull.any) {
        const unsigned fv = match_low_quality ? *first_valid : 0u;
        for (int c0 = 0; c0 < G; c0 += kHbbChunk) {
            const int cn = min(kHbbChunk, G - c0);
            int base = 0;
            for (int r0 = 0; r0 < cn; r0 += kHbbThreads) {
                const int k = r0 + tid;
                float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
                float gm = 0.f;
                int ga = 0;
                bool keep = false;
                if (k < cn) {
                    g = load_box(gts, (size_t)(c0 + k));
                    keep = !misses(hull, g);
                    if (match_low_quality) {
                        decode_gt_key(gt_key[c0 + k], fv, gm, ga);
                        keep |= gm == 0.f && gm >= min_pos_iou;
                    }
                }
                const unsigned m = __ballot_sync(0xffffffffu, keep);
                __syncthreads();  // s_wcnt free (and, on the first round, the previous chunk's list fully read)
                if (lane == 0) s_wcnt[wid] = __popc(m);
                __syncthreads();
                int pos = base, tot = 0;
                for (int w = 0; w < kHbbThreads / 32; w++) {
                    pos += w < wid ? s_wcnt[w] : 0;
                    tot += s_wcnt[w];
                }
                pos += __popc(m & ((1u << lane) - 1));
                if (keep) { s_gt[pos] = g; s_gidx[pos] = c0 + k; s_gm[pos] = gm; s_ga[pos] = ga; }
                base += tot;
            }
            __syncthreads();
            if (live) {
                for (int q = 0; q < base; q++) {
                    const float v = hbb_iou(s_gt[q], a);
                    const int g = s_gidx[q];
                    if (v > best) { best = v; bi = g; }
                    if (match_low_quality) {
                        const float gm = s_gm[q];
                        if (gm >= min_pos_iou && (assign_all ? (v == gm) : (s_ga[q] == j))) lowq = g + 1;
                    }
                }
            }
        }
    }
    if (j >= n) return;
    int r = -1;
    if (live) {
        if (best >= neg_lo && best < neg_hi) r = 0;
        if (best >= pos_thr) r = bi + 1;
        if (lowq) r = lowq;
    }
    gt_inds[j] = r;
    if (max_ov) max_ov[j] = best;
    if (labels) labels[j] = (r > 0 && gt_labels) ? gt_labels[r - 1] : labels_fill;
}

}  // namespace rsdet

using namespace rsdet;

extern "C" size_t rsdet_box_iou_rotated_workspace_bytes(int n1, int n2) {
    return ws_bytes<RBox>(n1 > 0 ? n1 : 0) + ws_bytes<RBox>(n2 > 0 ? n2 : 0);
}

extern "C" int rsdet_box_iou_rotated(const float* boxes1, int n1, const float* boxes2, int n2, int version,
                                        int zero_tiny, float* ious, void* workspace, size_t workspace_bytes, void* stream) {
    if (n1 < 0 || n2 < 0 || (version != 0 && version != 1)) return RSDET_EINVAL;
    if (n1 == 0 || n2 == 0) return RSDET_OK;
    if (!boxes1 || !boxes2 || !ious) return RSDET_EINVAL;
    if ((long long)n1 * n2 > (1ll << 40)) return RSDET_ELIMIT;
    Workspace ws(workspace, workspace_bytes);
    RBox* r1 = ws.take<RBox>(n1);
    RBox* r2 = ws.take<RBox>(n2);
    if (!ws.ok()) return RSDET_EWORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    prep_rbox_kernel<<<ceil_div(n1, 256), 256, 0, st>>>(boxes1, n1, version, zero_tiny, r1);
    prep_rbox_kernel<<<ceil_div(n2, 256), 256, 0, st>>>(boxes2, n2, version, zero_tiny, r2);
    long long tiles = (long long)ceil_div(n1, kTile) * ceil_div(n2, kTile);
    int grid = (int)(tiles < (long long)kNumSMs * 6 ? tiles : (long long)kNumSMs * 6);
    box_iou_tiles_kernel<<<grid, kIouThreads, 0, st>>>(r1, n1, r2, n2, ious);
    count_launch(3);
    return cuda_status();
}

extern "C" size_t rsdet_assign_workspace_bytes(int num_gts) {
    return ws_bytes<float>(num_gts > 0 ? num_gts : 0) + ws_bytes<int>(num_gts > 0 ? num_gts : 0);
}

extern "C" int rsdet_assign_wrt_overlaps(const float* overlaps, int num_gts, int n, float pos_iou_thr, float neg_lo,
                                            float neg_hi, float min_pos_iou, int match_low_quality, int gt_max_assign_all,
                                            const int32_t* gt_labels, int32_t labels_fill, int32_t* assigned_gt_inds,
                                            float* max_overlaps, int32_t* assigned_labels, void* workspace,
                                            size_t workspace_bytes, void* stream) {
    if (num_gts <= 0 || n <= 0) return RSDET_EINVAL;  // assigner.py:91-92,121-122 raise ValueError
    if (!overlaps || !assigned_gt_inds) return RSDET_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    float* gt_max = nullptr;
    int* gt_arg = nullptr;
    if (match_low_quality) {
        Workspace ws(workspace, workspace_bytes);
        gt_max = ws.take<float>(num_gts);
        gt_arg = ws.take<int>(num_gts);
        if (!ws.ok()) return RSDET_EWORKSPACE;
        assign_row_max_kernel<<<ceil_div(num_gts, 8), 256, 0, st>>>(overlaps, num_gts, n, gt_max, gt_arg);
        count_launch();
    }
    assign_col_kernel<<<ceil_div(n, 128), 128, 0, st>>>(overlaps, num_gts, n, pos_iou_thr, neg_lo, neg_hi, min_pos_iou,
                                                         match_low_quality, gt_max_assign_all, gt_max, gt_arg, gt_labels,
                                                         labels_fill, assigned_gt_inds, max_overlaps, assigned_labels);
    count_launch();
    return cuda_status();
}

extern "C" int rsdet_bbox_overlaps(const float* boxes1, int n1, const float* boxes2, int n2, float* ious, void* stream) {
    if (n1 < 0 || n2 < 0) return RSDET_EINVAL;
    if (n1 == 0 || n2 == 0) return RSDET_OK;
    if (!boxes1 || !boxes2 || !ious) return RSDET_EINVAL;
    if ((long long)n1 * n2 > (1ll << 40)) return RSDET_ELIMIT;
    const int row_groups = ceil_div(n1, kOvRows);
    dim3 grid(ceil_div(n2, 256), row_groups < 65535 ? row_groups : 65535);
    bbox_overlaps_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(boxes1, n1, boxes2, n2, ious);
    count_launch();
    return cuda_status();
}

static bool assign_hbb_sizes_ok(int num_gts, int n) {
    return num_gts <= RSDET_ASSIGN_HBB_MAX_GTS && n <= RSDET_ASSIGN_HBB_MAX_ANCHORS;
}

extern "C" size_t rsdet_assign_hbb_workspace_bytes(int num_gts, int n) {
    if (num_gts <= 0 || n <= 0 || !assign_hbb_sizes_ok(num_gts, n)) return 0;
    return ws_bytes<unsigned long long>(num_gts) + ws_bytes<unsigned>(1);
}

extern "C" int rsdet_assign_hbb(const float* gt_hbb, int num_gts, const float* anchors, int n, const uint8_t* valid,
                                float pos_iou_thr, float neg_lo, float neg_hi, float min_pos_iou, int match_low_quality,
                                int gt_max_assign_all, const int32_t* gt_labels, int32_t labels_fill,
                                int32_t* assigned_gt_inds, float* max_overlaps, int32_t* assigned_labels, void* workspace,
                                size_t workspace_bytes, void* stream) {
    if (num_gts <= 0 || n <= 0) return RSDET_EINVAL;  // as rsdet_assign_wrt_overlaps
    if (!gt_hbb || !anchors || !assigned_gt_inds) return RSDET_EINVAL;
    if (!assign_hbb_sizes_ok(num_gts, n)) return RSDET_ELIMIT;
    cudaStream_t st = (cudaStream_t)stream;
    unsigned long long* gt_key = nullptr;
    unsigned* first_valid = nullptr;
    if (match_low_quality) {
        Workspace ws(workspace, workspace_bytes);
        gt_key = ws.take<unsigned long long>(num_gts);
        first_valid = ws.take<unsigned>(1);
        if (!ws.ok()) return RSDET_EWORKSPACE;
        const int init_grid = ceil_div(num_gts, 256) < kNumSMs ? ceil_div(num_gts, 256) : kNumSMs;
        assign_hbb_init_kernel<<<init_grid, 256, 0, st>>>(gt_key, num_gts, first_valid);
        assign_hbb_gt_max_kernel<<<ceil_div(n, kHbbThreads), kHbbThreads, 0, st>>>(gt_hbb, num_gts, anchors, n, valid, gt_key,
                                                                                 first_valid);
        count_launch(2);
    }
    assign_hbb_col_kernel<<<ceil_div(n, kHbbThreads), kHbbThreads, 0, st>>>(
        gt_hbb, num_gts, anchors, n, valid, pos_iou_thr, neg_lo, neg_hi, min_pos_iou, match_low_quality, gt_max_assign_all,
        gt_key, first_valid, gt_labels, labels_fill, assigned_gt_inds, max_overlaps, assigned_labels);
    count_launch();
    return cuda_status();
}
