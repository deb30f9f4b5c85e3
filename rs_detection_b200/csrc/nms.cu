// nms.cu -- segmented bitmask NMS engine with four pair predicates (compile with -fmad=false).
//
// Replaces, for the whole greedy-NMS family of the reference:
//   nms_rotated_cuda_kernel + host mask scan   python/jdet/ops/nms_rotated.py:353-411, 450-493
//   nms_rotated_cpu greedy loop                python/jdet/ops/nms_rotated.py:414-449
//   ml_nms_rotated / nms_rotated glue          python/jdet/ops/nms_rotated.py:515-538
//   multiclass_nms_rotated                     python/jdet/ops/nms_rotated.py:540-596
//   poly_nms_kernel + host mask scan           python/jdet/ops/nms_poly.py:135-185, 187-232
//   py_cpu_nms_poly_fast (+ Shapely iou_poly)  python/jdet/data/devkits/result_merge.py:66-127
//   merge.py `nms`                             merge.py:14-27
//
// Design (B200-first, not a translation):
//   1. device radix sort (CUB = plumbing) by score, then stably by label -> every label group
//      ("segment": a class, or a (scene,class) pair in the merge stage) is contiguous and
//      score-descending.  Label-gated IoU (nms_rotated.py:281-286) == independent NMS per segment.
//   2. per-box preprocessing once (RBox / MBox), in sorted order.
//   3. ONE persistent kernel walks the upper-triangular 64x64 tiles of every segment (work list
//      derived on the device from a tiny segment table; no host round trip): bounding-circle / hbb
//      reject on all pairs, warp-ballot compaction of the survivors into a shared-memory queue, dense
//      evaluation of the survivors, 64-bit suppression words.  The reference launches the full n^2
//      grid (its triangular early-out is commented out, nms_rotated.py:363) over ALL labels; here the
//      mask is block-sparse per segment (sum n_s*ceil(n_s/64) words instead of n*ceil(n/64)).
//   4. on-device greedy scan, one CTA per segment: 64 rows are resolved from the diagonal word in
//      registers, then their suppression words are OR-ed into the shared-memory `remv` vector by all
//      threads.  The reference does this on the HOST after cudaDeviceSynchronize, reading the mask
//      through managed memory (nms_rotated.py:475-492).
//   5. compaction (CUB select) to the three index orders the reference's callers expect.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>
#include <thrust/iterator/counting_iterator.h>

#include <mutex>
#include <vector>

#include "common.cuh"
#include "nms_engine.cuh"
#include "poly_iou.cuh"
#include "rotated_iou.cuh"

namespace rsdet {

constexpr int kNmsThreads = 128;
constexpr int kReduceThreads = 256;
constexpr size_t kCubTempBytes = 8u << 20;
constexpr int kFastSegs = 2048;  // segment starts collected with atomics + one in-CTA bitonic sort

// ----------------------------------------------------------------------------- predicates
struct HBox { double x1, y1, x2, y2; };

template <int KIND> struct Traits;

template <> struct Traits<RSDET_NMS_ROTATED> {
    using Box = RBox; using Raw = float; using Thr = float;
    static constexpr int kRow = 5; static constexpr bool kScratch = true;
    __device__ static Box prep(const Raw* r) { return prep_rbox(r, 0); }
    // filter cascade (exact decisions, see rotated_iou.cuh): bounding circles on every pair, then -- dense, on
    // the compacted survivors -- the axis-aligned and the strip upper bounds of the IoU
    static constexpr bool kRefine = true;
    __device__ static bool cheap(const Box& a, const Box& b) { return rbox_may_overlap(a, b); }
    __device__ static bool refine1(const Box& a, const Box& b, Thr thr) { return !rbox_iou_below(a, b, thr); }
    __device__ static bool refine2(const Box& a, const Box& b, Thr thr) { return !rbox_iou_below_strips(a, b, thr); }
    __device__ static bool suppress(const Box& a, const Box& b, Thr thr, float2* q) {
        return rotated_iou_pair<kNmsThreads>(a, b, q) > thr;
    }
};
template <> struct Traits<RSDET_NMS_ROTATED_GE> : Traits<RSDET_NMS_ROTATED> {
    __device__ static bool suppress(const Box& a, const Box& b, Thr thr, float2* q) {
        return rotated_iou_pair<kNmsThreads>(a, b, q) >= thr;
    }
};
template <> struct Traits<RSDET_NMS_POLY> {
    using Box = PolyBox; using Raw = float; using Thr = float;
    static constexpr int kRow = 8; static constexpr bool kScratch = true;   // 2 x 10 polygon slots per thread
    __device__ static Box prep(const Raw* r) { return prep_polybox(r); }
    static constexpr bool kRefine = false;
    // the only pairs dropped before the exact evaluation are those whose 16 fan terms are provably all zero
    __device__ static bool cheap(const Box& a, const Box& b) { return !poly_pair_is_zero(a, b); }
    __device__ static bool refine1(const Box&, const Box&, Thr) { return true; }
    __device__ static bool refine2(const Box&, const Box&, Thr) { return true; }
    __device__ static bool suppress(const Box& a, const Box& b, Thr thr, float2* q) {
        return poly_iou_f32<kNmsThreads>(a, b, q) > thr;
    }
};
template <> struct Traits<RSDET_NMS_MERGE> {
    using Box = MBox; using Raw = double; using Thr = double;
    static constexpr int kRow = 8; static constexpr bool kScratch = false;
    __device__ static Box prep(const Raw* r) {
        Box b;
        double x1 = r[0], x2 = r[0], y1 = r[1], y2 = r[1];
        for (int i = 0; i < 4; i++) {
            b.p[2 * i] = r[2 * i]; b.p[2 * i + 1] = r[2 * i + 1];
            x1 = fmin(x1, r[2 * i]); x2 = fmax(x2, r[2 * i]);
            y1 = fmin(y1, r[2 * i + 1]); y2 = fmax(y2, r[2 * i + 1]);
        }
        b.x1 = x1; b.y1 = y1; b.x2 = x2; b.y2 = y2;
        return b;
    }
    static constexpr bool kRefine = false;
    __device__ static bool cheap(const Box& a, const Box& b) { return merge_hbb_overlap(a, b); }
    __device__ static bool refine1(const Box&, const Box&, Thr) { return true; }
    __device__ static bool refine2(const Box&, const Box&, Thr) { return true; }
    // survivors are `iou <= thr` (result_merge.py:118)
    __device__ static bool suppress(const Box& a, const Box& b, Thr thr, float2*) { return !(iou_poly_d(a, b) <= thr); }
};
template <> struct Traits<RSDET_NMS_HBB> {
    using Box = HBox; using Raw = double; using Thr = double;
    static constexpr int kRow = 4; static constexpr bool kScratch = false;
    __device__ static Box prep(const Raw* r) { Box b; b.x1 = r[0]; b.y1 = r[1]; b.x2 = r[2]; b.y2 = r[3]; return b; }
    static constexpr bool kRefine = false;
    // pairs without a proper overlap have iou = 0 / (A + B) in the reference: kept for thresh > 0 -- EXCEPT when
    // both areas are zero (0/0 = NaN, and `NaN < thresh` is false: suppressed), so those pairs pass the filter
    __device__ static bool cheap(const Box& a, const Box& b) {
        return (fmin(a.x2, b.x2) > fmax(a.x1, b.x1) && fmin(a.y2, b.y2) > fmax(a.y1, b.y1)) ||
               (a.x2 - a.x1) * (a.y2 - a.y1) + (b.x2 - b.x1) * (b.y2 - b.y1) == 0.0;
    }
    __device__ static bool refine1(const Box&, const Box&, Thr) { return true; }
    __device__ static bool refine2(const Box&, const Box&, Thr) { return true; }
    // merge.py:19-25: overlaps = prod(br - tl) * all(br > tl); survivors are `iou < thresh`
    __device__ static bool suppress(const Box& a, const Box& b, Thr thr, float2*) {
        double tlx = fmax(a.x1, b.x1), tly = fmax(a.y1, b.y1), brx = fmin(a.x2, b.x2), bry = fmin(a.y2, b.y2);
        double ov = (brx - tlx) * (bry - tly) * ((brx > tlx && bry > tly) ? 1.0 : 0.0);
        double iou = ov / ((a.x2 - a.x1) * (a.y2 - a.y1) + (b.x2 - b.x1) * (b.y2 - b.y1) - ov);
        return !(iou < thr);
    }
};

// py_cpu_nms (data/devkits/result_merge.py:143-174, used by mergebyrec): float64, "+1" widths, survivors ovr <= thresh
template <> struct Traits<RSDET_NMS_HBB_P1_F64> {
    using Box = HBox; using Raw = double; using Thr = double;
    static constexpr int kRow = 4; static constexpr bool kScratch = false;
    static constexpr bool kRefine = false;
    __device__ static Box prep(const Raw* r) { Box b; b.x1 = r[0]; b.y1 = r[1]; b.x2 = r[2]; b.y2 = r[3]; return b; }
    __device__ static bool cheap(const Box& a, const Box& b) {
        return fmin(a.x2, b.x2) - fmax(a.x1, b.x1) + 1.0 > 0.0 && fmin(a.y2, b.y2) - fmax(a.y1, b.y1) + 1.0 > 0.0;
    }
    __device__ static bool refine1(const Box&, const Box&, Thr) { return true; }
    __device__ static bool refine2(const Box&, const Box&, Thr) { return true; }
    __device__ static bool suppress(const Box& a, const Box& b, Thr thr, float2*) {
        double w = fmax(0.0, fmin(a.x2, b.x2) - fmax(a.x1, b.x1) + 1.0), h = fmax(0.0, fmin(a.y2, b.y2) - fmax(a.y1, b.y1) + 1.0);
        double inter = w * h;
        double ovr = inter / ((a.x2 - a.x1 + 1.0) * (a.y2 - a.y1 + 1.0) + (b.x2 - b.x1 + 1.0) * (b.y2 - b.y1 + 1.0) - inter);
        return !(ovr <= thr);
    }
};

// jt.nms (Jittor 1.3.4.7 misc.py `nms`, called from oriented_rpn_head.py:208): fp32 boxes, the "+1" pixel
// convention, fail condition `inter / (a_j + a_i - inter) > thr` with thr a double literal in Jittor's JIT source.
struct HBoxF { float x1, y1, x2, y2; };
template <> struct Traits<RSDET_NMS_HBB_P1> {
    using Box = HBoxF; using Raw = float; using Thr = double;
    static constexpr int kRow = 4; static constexpr bool kScratch = false;
    __device__ static Box prep(const Raw* r) { Box b; b.x1 = r[0]; b.y1 = r[1]; b.x2 = r[2]; b.y2 = r[3]; return b; }
    static constexpr bool kRefine = false;
    __device__ static bool cheap(const Box& a, const Box& b) {
        return fminf(a.x2, b.x2) - fmaxf(a.x1, b.x1) + 1.f > 0.f && fminf(a.y2, b.y2) - fmaxf(a.y1, b.y1) + 1.f > 0.f;
    }
    __device__ static bool refine1(const Box&, const Box&, Thr) { return true; }
    __device__ static bool refine2(const Box&, const Box&, Thr) { return true; }
    __device__ static bool suppress(const Box& a, const Box& b, Thr thr, float2*) {
        float iw = fmaxf(0.f, fminf(a.x2, b.x2) - fmaxf(a.x1, b.x1) + 1.f);
        float ih = fmaxf(0.f, fminf(a.y2, b.y2) - fmaxf(a.y1, b.y1) + 1.f);
        float inter = ih * iw;
        float sa = (a.x2 - a.x1 + 1.f) * (a.y2 - a.y1 + 1.f), sb = (b.x2 - b.x1 + 1.f) * (b.y2 - b.y1 + 1.f);
        return (double)(inter / (sa + sb - inter)) > thr;
    }
};

// ----------------------------------------------------------------------------- segment table
struct SegTable {
    int* hdr;              // [0]=nseg [1]=n_eff [2]=tile counter [3]=#boundaries  (+ [4..5] total tiles as long long)
    int* seg_start;        // nseg+1
    long long* tile_pref;  // nseg+1
    long long* mask_off;   // nseg+1 (in 64-bit words)
    double* seg_thr;       // nseg
};

// Ascending key = descending score.  -0.0 and +0.0 compare equal, so both get the key of +0.0: a tie, which the stable
// sorts resolve by index like every other tie (the oracle's stable sort of -scores does the same).
__device__ __forceinline__ uint32_t desc_key(float s) {
    uint32_t u = __float_as_uint(s == 0.f ? 0.f : s);
    u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
    return ~u;
}
__device__ __forceinline__ unsigned long long desc_key(double s) {
    unsigned long long u = (unsigned long long)__double_as_longlong(s == 0.0 ? 0.0 : s);
    u = (u >> 63) ? ~u : (u | 0x8000000000000000ull);
    return ~u;
}

// rows that are not live (multiclass candidates below score_thr) carry score -inf and sort last
// `reverse`: rows are handed to the (stable) radix sort in descending index order, so equal scores come out
// HIGHER index first -- the order of `scores.argsort(kind='stable')[::-1]`, the tie rule of the float64 merge
// kinds (result_merge.py:84, merge.py:16).  Text-format scores have four decimals, so ties are common there.
template <typename ScoreT, typename KeyT>
__global__ void make_keys_kernel(const ScoreT* __restrict__ scores, int n_max, KeyT* __restrict__ keys, int* __restrict__ idx,
                                 bool reverse) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_max) return;
    const int r = reverse ? n_max - 1 - i : i;
    keys[i] = (KeyT)desc_key(scores[r]);
    idx[i] = r;
}

// label_bits == 32: arbitrary int32 labels (sign-flipped key).  label_bits < 32: the caller guarantees
// 0 <= label, and every label >= 2^bits-1 (the dead-row marker) collapses onto the all-ones key, so the
// radix sort needs ceil(bits/8) passes instead of 4.
__global__ void label_keys_kernel(const int32_t* __restrict__ labels, const int* __restrict__ idx, int n_max,
                                  const int* __restrict__ n_dev, int label_bits, uint32_t* __restrict__ lkeys) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_max) return;
    int n = n_dev ? min(*n_dev, n_max) : n_max;
    uint32_t key;
    if (label_bits >= 32) key = p < n ? ((uint32_t)labels[idx[p]] ^ 0x80000000u) : 0xffffffffu;
    else {
        const uint32_t top = (1u << label_bits) - 1u;
        key = p < n ? min((uint32_t)labels[idx[p]], top) : top;
    }
    lkeys[p] = key;
}

template <int KIND>
__global__ void prep_sorted_kernel(const typename Traits<KIND>::Raw* __restrict__ dets, const int32_t* __restrict__ labels,
                                   const int* __restrict__ idx, int n_max, const int* __restrict__ n_dev,
                                   typename Traits<KIND>::Box* __restrict__ boxes, int32_t* __restrict__ label_sorted,
                                   int* __restrict__ hdr, int* __restrict__ starts_unsorted) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_max) return;
    int n = n_dev ? min(*n_dev, n_max) : n_max;
    if (p >= n) return;
    int src = idx[p];
    if (boxes) boxes[p] = Traits<KIND>::prep(dets + (size_t)src * Traits<KIND>::kRow);
    bool boundary = p == 0;
    if (labels) {
        int l = labels[src];
        label_sorted[p] = l;
        if (p > 0) boundary = labels[idx[p - 1]] != l;
    }
    if (boundary) {  // collect segment starts (unordered); segment_table_kernel sorts them
        int k = atomicAdd(&hdr[3], 1);
        if (k < kFastSegs) starts_unsorted[k] = p;
    }
}

// exclusive scan of one long long per thread across a 1024-thread CTA; returns the CTA total via *total
__device__ long long block_excl_scan(long long v, long long* s_warp, long long* total) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    long long x = v;
    for (int o = 1; o < 32; o <<= 1) {
        long long y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) s_warp[w] = x;
    __syncthreads();
    if (w == 0) {
        long long s = lane < (blockDim.x >> 5) ? s_warp[lane] : 0;
        for (int o = 1; o < 32; o <<= 1) {
            long long y = __shfl_up_sync(0xffffffffu, s, o);
            if (lane >= o) s += y;
        }
        s_warp[lane] = s;
    }
    __syncthreads();
    long long warp_off = w ? s_warp[w - 1] : 0;
    *total = s_warp[31];
    __syncthreads();
    return warp_off + x - v;
}

__global__ void __launch_bounds__(1024)
segment_table_kernel(const int32_t* __restrict__ label_sorted, int n_max, const int* __restrict__ n_dev, double thr,
                     const double* __restrict__ thr_per_label, int num_thr, SegTable tb,
                     const int* __restrict__ starts_unsorted) {
    __shared__ long long s_warp[32];
    __shared__ int s_sort[kFastSegs];
    const int tid = threadIdx.x;
    const int n = n_dev ? min(*n_dev, n_max) : n_max;
    int nseg;
    const int nb = tb.hdr[3];  // boundaries found by prep_sorted_kernel
    if (nb <= kFastSegs) {
        // few segments (the normal case: classes): sort the collected starts in shared memory
        for (int i = tid; i < kFastSegs; i += 1024) s_sort[i] = i < nb ? starts_unsorted[i] : 0x7fffffff;
        __syncthreads();
        for (int k = 2; k <= kFastSegs; k <<= 1)
            for (int j = k >> 1; j > 0; j >>= 1) {
                for (int i = tid; i < kFastSegs; i += 1024) {
                    int ixj = i ^ j;
                    if (ixj > i) {
                        int a = s_sort[i], b = s_sort[ixj];
                        bool up = (i & k) == 0;
                        if ((a > b) == up) { s_sort[i] = b; s_sort[ixj] = a; }
                    }
                }
                __syncthreads();
            }
        nseg = nb;
        for (int i = tid; i < nb; i += 1024) tb.seg_start[i] = s_sort[i];
    } else {
        // many segments: ordered compaction by a chunked scan over the sorted labels
        const int chunk = ceil_div(n > 0 ? n : 1, 1024);
        const int p0 = min(n, tid * chunk), p1 = min(n, p0 + chunk);
        int cnt = 0;
        for (int p = p0; p < p1; p++)
            cnt += (p == 0) || (label_sorted && label_sorted[p] != label_sorted[p - 1]);
        long long total;
        int off = (int)block_excl_scan(cnt, s_warp, &total);
        nseg = (int)total;
        for (int p = p0; p < p1; p++)
            if ((p == 0) || (label_sorted && label_sorted[p] != label_sorted[p - 1])) tb.seg_start[off++] = p;
    }
    if (tid == 0) tb.seg_start[nseg] = n;
    __syncthreads();
    long long carry_t = 0, carry_w = 0;
    for (int base = 0; base < nseg; base += 1024) {
        int s = base + tid;
        long long tiles = 0, words = 0;
        if (s < nseg) {
            int st = tb.seg_start[s];
            long long ns = tb.seg_start[s + 1] - st;
            long long T = (ns + 63) / 64;
            tiles = T * (T + 1) / 2;
            words = ns * T;
            double t = thr;
            if (thr_per_label && label_sorted) {
                int l = label_sorted[st];
                if (l >= 0 && l < num_thr) t = thr_per_label[l];
            }
            tb.seg_thr[s] = t;
        }
        long long tt, tw;
        long long et = block_excl_scan(tiles, s_warp, &tt);
        long long ew = block_excl_scan(words, s_warp, &tw);
        if (s < nseg) { tb.tile_pref[s] = carry_t + et; tb.mask_off[s] = carry_w + ew; }
        carry_t += tt; carry_w += tw;
    }
    if (tid == 0) {
        tb.tile_pref[nseg] = carry_t;
        tb.mask_off[nseg] = carry_w;
        tb.hdr[0] = nseg; tb.hdr[1] = n; tb.hdr[2] = 0;
        *(long long*)(tb.hdr + 4) = carry_t;
    }
}

// segment table straight from per-class live counts (multiclass path): empty classes are skipped
__global__ void __launch_bounds__(1024)
segments_from_counts_kernel(const int* __restrict__ counts, int C, double thr, SegTable tb) {
    __shared__ long long s_warp[32];
    const int tid = threadIdx.x;
    long long carry_n = 0, carry_s = 0, carry_t = 0, carry_w = 0;
    for (int base = 0; base < C; base += 1024) {
        const int c = base + tid;
        const long long ns = c < C ? counts[c] : 0;
        const long long T = (ns + 63) / 64;
        long long tn, ts, tt, tw;
        const long long en = block_excl_scan(ns, s_warp, &tn);
        const long long es = block_excl_scan(ns > 0 ? 1 : 0, s_warp, &ts);
        const long long et = block_excl_scan(T * (T + 1) / 2, s_warp, &tt);
        const long long ew = block_excl_scan(ns * T, s_warp, &tw);
        if (ns > 0) {
            const int sidx = (int)(carry_s + es);
            tb.seg_start[sidx] = (int)(carry_n + en);
            tb.tile_pref[sidx] = carry_t + et;
            tb.mask_off[sidx] = carry_w + ew;
            tb.seg_thr[sidx] = thr;
        }
        carry_n += tn; carry_s += ts; carry_t += tt; carry_w += tw;
    }
    if (tid == 0) {
        const int nseg = (int)carry_s;
        tb.seg_start[nseg] = (int)carry_n;
        tb.tile_pref[nseg] = carry_t;
        tb.mask_off[nseg] = carry_w;
        tb.hdr[0] = nseg; tb.hdr[1] = (int)carry_n; tb.hdr[2] = 0;
        *(long long*)(tb.hdr + 4) = carry_t;
    }
}

// ----------------------------------------------------------------------------- mask tiles
// Filter cascade of the mask kernels: every stage runs DENSE over the compacted survivors of the previous one
// (bounding circles on all 64 x 64 pairs -> axis-aligned bound -> strip bound -> exact clipper).  Evaluated
// inside the all-pairs loop, the bounds cost ~100 warp instructions per 32 pairs at 5 active lanes, because
// nearly every warp holds at least one pair whose circles touch (16 % of the pairs on the bench proposals).
template <typename Pred>
__device__ __forceinline__ int compact_queue(const unsigned short* __restrict__ in, int n_in, unsigned short* __restrict__ out,
                                             int* s_counter, int* s_wsum, Pred keep) {
    // n_in <= 8 * kNmsThreads (the callers' chunk size): a thread tests entries tid, tid + 128, ..., keeps its
    // verdicts in a register and the survivors are placed with ONE prefix sum (no ballot / atomic per 32 entries)
    const int tid = threadIdx.x, lane = tid & 31;
    unsigned hits = 0u;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        const int qi = tid + k * kNmsThreads;
        if (qi < n_in && keep((int)in[qi])) hits |= 1u << k;
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
    if (tid == kNmsThreads - 1) *s_counter = pos + mine;
    while (hits) {
        const int k = __ffs(hits) - 1;
        hits &= hits - 1;
        out[pos++] = in[tid + k * kNmsThreads];
    }
    __syncthreads();
    return *s_counter;
}

template <int KIND>
__global__ void __launch_bounds__(kNmsThreads)
mask_tiles_kernel(const typename Traits<KIND>::Box* __restrict__ boxes, SegTable tb, unsigned long long* __restrict__ mask,
                  const int* __restrict__ gate) {
    using Tr = Traits<KIND>;
    if (gate && *gate == 0) return;  // the sparse path (below) already produced the keep flags
    using Box = typename Tr::Box;
    __shared__ Box s_row[64];
    __shared__ Box s_col[64];
    __shared__ unsigned short s_queue[64 * 64];
    __shared__ unsigned long long s_mask[64];
    constexpr int kQ2 = Tr::kRefine ? 1024 : 1;
    __shared__ unsigned short s_queue2[kQ2];
    __shared__ unsigned short s_queue3[kQ2];
    __shared__ float2 s_pts[Tr::kScratch ? 24 * kNmsThreads : 1];
    __shared__ int s_wsum[kNmsThreads / 32];
    __shared__ int s_count;
    __shared__ int s_count2;
    __shared__ int s_count3;
    __shared__ long long s_tile;

    const int tid = threadIdx.x, lane = tid & 31;
    const int nseg = tb.hdr[0];
    const long long total = *(const long long*)(tb.hdr + 4);

    while (true) {
        __syncthreads();
        if (tid == 0) s_tile = (long long)atomicAdd((unsigned int*)&tb.hdr[2], 1u);
        __syncthreads();
        const long long t = s_tile;
        if (t >= total) break;
        // segment lookup
        int lo = 0, hi = nseg;
        while (hi - lo > 1) {
            int mid = (lo + hi) >> 1;
            if (tb.tile_pref[mid] <= t) lo = mid; else hi = mid;
        }
        const int s = lo;
        const long long u = t - tb.tile_pref[s];
        const int st = tb.seg_start[s];
        const int ns = tb.seg_start[s + 1] - st;
        const int T = (ns + 63) >> 6;
        // row-major upper triangle: row rb holds T-rb tiles, preceded by rb*T - rb*(rb-1)/2
        int rb = (int)(((2.0 * T + 1.0) - sqrt((2.0 * T + 1.0) * (2.0 * T + 1.0) - 8.0 * (double)u)) * 0.5);
        rb = max(0, min(rb, T - 1));
        while (rb > 0 && (long long)rb * T - (long long)rb * (rb - 1) / 2 > u) rb--;
        while ((long long)(rb + 1) * T - (long long)(rb + 1) * rb / 2 <= u) rb++;
        const int cb = rb + (int)(u - ((long long)rb * T - (long long)rb * (rb - 1) / 2));
        const int nr = min(64, ns - rb * 64), nc = min(64, ns - cb * 64);
        const typename Tr::Thr thr = (typename Tr::Thr)tb.seg_thr[s];

        if (tid < 64) {
            if (tid < nr) s_row[tid] = boxes[st + rb * 64 + tid];
            s_mask[tid] = 0ull;
        } else if (tid - 64 < nc) {
            s_col[tid - 64] = boxes[st + cb * 64 + tid - 64];
        }
        __syncthreads();

        // stage 1: each thread owns ONE column box (registers) and sweeps 32 rows with the cheap test; a warp
        // reads the same row box at a time (shared-memory broadcast).  Hits go to a register bit mask and are
        // compacted once per tile.
        const bool diag = rb == cb;
        {
            const int c = tid & 63, rhalf = tid >> 6;
            unsigned hits = 0u;
            if (c < nc) {
                const Box colbox = s_col[c];
#pragma unroll 4
                for (int k = 0; k < 32; k++) {
                    const int r = 2 * k + rhalf;
                    const bool cand = r < nr && (!diag || c > r) && Tr::cheap(s_row[r], colbox);
                    hits |= (cand ? 1u : 0u) << k;
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
            if (tid == kNmsThreads - 1) s_count = pos + mine;
            while (hits) {
                const int k = __ffs(hits) - 1;
                hits &= hits - 1;
                s_queue[pos++] = (unsigned short)(((2 * k + rhalf) << 6) | c);
            }
        }
        __syncthreads();
        const int cnt = s_count;
        if (Tr::kRefine) {
            for (int q0 = 0; q0 < cnt; q0 += kQ2) {
                const int n2 = compact_queue(s_queue + q0, min(kQ2, cnt - q0), s_queue2, &s_count2, s_wsum,
                                             [&](int p) { return Tr::refine1(s_row[p >> 6], s_col[p & 63], thr); });
                const int n3 = compact_queue(s_queue2, n2, s_queue3, &s_count3, s_wsum,
                                             [&](int p) { return Tr::refine2(s_row[p >> 6], s_col[p & 63], thr); });
                for (int qi = tid; qi < n3; qi += kNmsThreads) {
                    const int p = s_queue3[qi];
                    const int r = p >> 6, c = p & 63;
                    if (Tr::suppress(s_row[r], s_col[c], thr, s_pts + (Tr::kScratch ? tid : 0))) atomicOr(&s_mask[r], 1ull << c);
                }
            }
        } else {
            for (int qi = tid; qi < cnt; qi += kNmsThreads) {
                const int p = s_queue[qi];
                const int r = p >> 6, c = p & 63;
                if (Tr::suppress(s_row[r], s_col[c], thr, s_pts + (Tr::kScratch ? tid : 0))) atomicOr(&s_mask[r], 1ull << c);
            }
        }
        __syncthreads();
        if (tid < nr) mask[tb.mask_off[s] + (long long)(rb * 64 + tid) * T + cb] = s_mask[tid];
    }
}

// ----------------------------------------------------------------------------- greedy scan
// Small label groups (< kCoopMinBlocks 64-row blocks): one CTA per group walks its blocks in score
// order.  Per block: (1) thread 0 resolves the 64 rows against the accumulated `remv` word and the block's
// diagonal words (pulled into registers first, so the dependent chain is pure ALU); (2) all 256 threads
// OR the suppression words of the KEPT rows into the shared-memory `remv` vector (64 column lanes x 4
// row groups, merged with shared-memory atomics).  The next diagonal is prefetched meanwhile.
//
// Large groups (a 100k-box single-class NMS has 1563 dependent blocks and ~0.5 GB of kept-row words to
// OR): kCoopCtas co-resident CTAs share ONE group.  Column block j belongs to CTA j % kCoopCtas, which keeps
// that slice of `remv` in its shared memory.  The owner of block b resolves it and publishes the 64 keep
// bits through global memory (word + flag, release/acquire by __threadfence); every CTA ORs the kept rows
// into its own columns.  Only "publish -> next owner's one-column OR -> resolve" is on the critical path
// (~2 us per block instead of the ~25 us a single CTA needs to sweep 64 x 1563 words).
constexpr int kCoopMinBlocks = 128;
constexpr int kCoopCtas = 64;

__device__ __forceinline__ unsigned long long resolve_block(const unsigned long long* __restrict__ diag, unsigned long long r, int nr) {
    unsigned long long d[64];
#pragma unroll
    for (int i = 0; i < 64; i++) d[i] = diag[i];
    unsigned long long kb = 0ull;
    if (nr < 64) r |= ~0ull << nr;  // rows past the group end count as removed
#pragma unroll
    for (int i = 0; i < 64; i++) {
        const bool alive = ((r >> i) & 1ull) == 0ull;
        kb |= alive ? (1ull << i) : 0ull;
        r |= alive ? d[i] : 0ull;
    }
    return kb;
}

__global__ void __launch_bounds__(kReduceThreads, 1)
reduce_kernel(SegTable tb, const unsigned long long* __restrict__ mask, uint8_t* __restrict__ keep_sorted,
              unsigned long long* __restrict__ pub_keep, int* __restrict__ pub_flag, int skip_small, const int* __restrict__ gate) {
    if (gate && *gate == 0) return;
    extern __shared__ unsigned long long s_remv[];
    __shared__ unsigned long long s_diag[2][64];
    __shared__ unsigned long long s_keep;
    const int tid = threadIdx.x, lane = tid & 31;
    const int nseg = tb.hdr[0];
    // ---- phase 1: small groups, one CTA each
    int small_rank = 0;
    for (int s = 0; s < nseg; s++) {
        const int st = tb.seg_start[s];
        const int ns = tb.seg_start[s + 1] - st;
        const int T = (ns + 63) >> 6;
        if (T >= kCoopMinBlocks || skip_small) continue;  // skip_small: reduce_ov_staged_kernel<2, true> took them
        if ((small_rank++ % (int)gridDim.x) != (int)blockIdx.x) continue;
        const unsigned long long* m = mask + tb.mask_off[s];
        __syncthreads();
        for (int j = tid; j < T; j += kReduceThreads) s_remv[j] = 0ull;
        if (tid < 64) s_diag[0][tid] = tid < min(64, ns) ? m[(long long)tid * T] : 0ull;
        __syncthreads();
        for (int b = 0; b < T; b++) {
            const int nr = min(64, ns - b * 64);
            unsigned long long diag_next = 0ull;
            if (tid >= 64 && tid < 128 && b + 1 < T) {  // warps 2/3 prefetch the next diagonal
                const int i = tid - 64;
                if (i < min(64, ns - (b + 1) * 64)) diag_next = m[(long long)((b + 1) * 64 + i) * T + (b + 1)];
            }
            if (tid == 0) s_keep = resolve_block(s_diag[b & 1], s_remv[b], nr);
            __syncthreads();
            const unsigned long long kb = s_keep;
            if (tid < nr) keep_sorted[st + b * 64 + tid] = (uint8_t)((kb >> tid) & 1ull);
            if (tid >= 64 && tid < 128) s_diag[(b + 1) & 1][tid - 64] = diag_next;
            if (kb) {
                const int jj = tid & 63, rg = tid >> 6;
                const unsigned kb16 = (unsigned)((kb >> (rg * 16)) & 0xffffull);
                if (kb16) {
                    for (int j = b + 1 + jj; j < T; j += 64) {
                        unsigned long long acc = 0ull;
                        const unsigned long long* col = m + (long long)(b * 64 + rg * 16) * T + j;
#pragma unroll
                        for (int i = 0; i < 16; i++)
                            if ((kb16 >> i) & 1u) acc |= col[(long long)i * T];
                        if (acc) atomicOr(&s_remv[j], acc);
                    }
                }
            }
            __syncthreads();
        }
    }
    // ---- phase 2: large groups, kCoopCtas CTAs per group
    const int G = min(kCoopCtas, (int)gridDim.x), k = blockIdx.x;
    if (k >= G) return;
    int large_rank = 0;
    for (int s = 0; s < nseg; s++) {
        const int st = tb.seg_start[s];
        const int ns = tb.seg_start[s + 1] - st;
        const int T = (ns + 63) >> 6;
        if (T < kCoopMinBlocks) continue;
        const unsigned long long* m = mask + tb.mask_off[s];
        const int pub0 = (st >> 6) + large_rank++;  // unique publication slots for this group's blocks
        const int nloc = (T + G - 1) / G;          // my slice of remv: column j -> s_remv[j / G]
        __syncthreads();
        for (int j = tid; j < nloc; j += kReduceThreads) s_remv[j] = 0ull;
        __syncthreads();
        for (int b = 0; b < T; b++) {
            const int nr = min(64, ns - b * 64);
            const bool own = (b % G) == k, own_next = ((b + 1) % G) == k && b + 1 < T;
            // loads that do not depend on the keep bits are issued before waiting for them
            unsigned long long pre = 0ull;
            if (own && tid < 64) { if (tid < nr) pre = m[(long long)(b * 64 + tid) * T + b]; s_diag[0][tid] = pre; }
            if (own_next && tid >= 64 && tid < 128) { const int i = tid - 64; if (i < nr) pre = m[(long long)(b * 64 + i) * T + (b + 1)]; }
            __syncthreads();
            if (tid == 0) {
                unsigned long long kb;
                if (own) {
                    kb = resolve_block(s_diag[0], s_remv[b / G], nr);
                    pub_keep[pub0 + b] = kb;
                    __threadfence();
                    *(volatile int*)(pub_flag + pub0 + b) = 1;
                } else {
                    while (*(volatile int*)(pub_flag + pub0 + b) == 0) { }
                    __threadfence();
                    kb = *(volatile unsigned long long*)(pub_keep + pub0 + b);
                }
                s_keep = kb;
            }
            __syncthreads();
            const unsigned long long kb = s_keep;
            if (own && tid < nr) keep_sorted[st + b * 64 + tid] = (uint8_t)((kb >> tid) & 1ull);
            // critical path first: the next owner folds block b into column b+1 (words already in registers)
            if (own_next && tid >= 64 && tid < 128) {
                unsigned long long w = ((kb >> (tid - 64)) & 1ull) ? pre : 0ull;
                unsigned lo = __reduce_or_sync(0xffffffffu, (unsigned)w), hi = __reduce_or_sync(0xffffffffu, (unsigned)(w >> 32));
                if (lane == 0 && (lo | hi)) atomicOr(&s_remv[(b + 1) / G], ((unsigned long long)hi << 32) | lo);
            }
            // then my other columns j > b (j % G == k), 16 column lanes x 16 row groups of 4
            if (kb) {
                int j0 = b + 1 + ((k - (b + 1)) % G + G) % G;
                if (own_next) j0 += G;
                const int cl = tid & 15, rg = tid >> 4;
                const unsigned kb4 = (unsigned)((kb >> (rg * 4)) & 0xfull);
                if (kb4) {
                    for (int j = j0 + cl * G; j < T; j += 16 * G) {
                        unsigned long long acc = 0ull;
                        const unsigned long long* col = m + (long long)(b * 64 + rg * 4) * T + j;
#pragma unroll
                        for (int i = 0; i < 4; i++)
                            if ((kb4 >> i) & 1u) acc |= col[(long long)i * T];
                        if (acc) atomicOr(&s_remv[j / G], acc);
                    }
                }
            }
            __syncthreads();
        }
    }
}

// ----------------------------------------------------------------------------- shared-box mode
// multiclass_nms_rotated with class-agnostic boxes (multi_bboxes is (n,5): every class scores the SAME n
// boxes -- `reg_class_agnostic=True` in the orcnn configs, and every single-stage head).  The reference
// expands to n*C candidates and evaluates IoU per class; but IoU(a,b) does not depend on the class, so
// the pairwise decisions are computed ONCE per box pair into a directed n x n bit matrix
// (ov[a][b] = "a, as the higher-scored box, suppresses b") and each class's greedy scan reads it through
// its own score order.  C x fewer clipper calls (10x on FAIR1M, 15x on DOTA).
//
// Orientation: the reference evaluates single_box_iou_rotated(higher, lower) and its float result is not
// exactly symmetric, and which box is "higher" differs per class.  The canonical evaluation is
// (lower index, higher index); the reverse orientation is recomputed only when the IoU lies within 1e-5
// of the threshold, otherwise both directions take the same decision.
__global__ void prep_shared_kernel(const float* __restrict__ boxes, int n, RBox* __restrict__ out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = prep_rbox(boxes + (size_t)i * 5, 0);
}

template <bool GE>
__global__ void __launch_bounds__(kNmsThreads, 5)
ov_tiles_kernel(const RBox* __restrict__ boxes, int n, float thr, unsigned long long* __restrict__ ov, int pitch,
                const uint8_t* __restrict__ only_flagged, const unsigned int* __restrict__ num_flagged) {
    if (only_flagged && *num_flagged == 0u) return;  // the usual case: every tile's survivors fitted the pair queue
    __shared__ RBox s_row[64];
    __shared__ RBox s_col[64];
    __shared__ unsigned short s_queue[64 * 64];
    constexpr int kQ2 = 1024;
    __shared__ unsigned short s_queue2[kQ2];
    __shared__ unsigned short s_queue3[kQ2];
    __shared__ float2 s_pts[24 * kNmsThreads];
    __shared__ float4 s_rowc[64];
    __shared__ int s_wsum[kNmsThreads / 32];
    __shared__ int s_count;
    __shared__ int s_count2;  // one counter per stage: a stage's result is still being read when the next one resets its own
    __shared__ int s_count3;
    const int tid = threadIdx.x, lane = tid & 31;
    const int T = (n + 63) >> 6;
    const int total = T * (T + 1) / 2;
    // one tile per CTA when the grid covers them all (the usual case: the block scheduler balances the uneven
    // tiles and no CTA waits on a global counter), grid-stride otherwise
    for (int u = blockIdx.x; u < total; u += gridDim.x) {
        if (only_flagged && !only_flagged[u]) continue;  // CTA-uniform
        __syncthreads();
        int rb = (int)(((2.0 * T + 1.0) - sqrt((2.0 * T + 1.0) * (2.0 * T + 1.0) - 8.0 * (double)u)) * 0.5);
        rb = max(0, min(rb, T - 1));
        while (rb > 0 && rb * T - rb * (rb - 1) / 2 > u) rb--;
        while ((rb + 1) * T - (rb + 1) * rb / 2 <= u) rb++;
        const int cb = rb + (u - (rb * T - rb * (rb - 1) / 2));
        const int nr = min(64, n - rb * 64), nc = min(64, n - cb * 64);
        if (tid < 64) {
            float4 rc = make_float4(0.f, 0.f, -1e30f, 0.f);
            if (tid < nr) {
                const RBox bx = boxes[rb * 64 + tid];
                s_row[tid] = bx;
                rc = make_float4(bx.x, bx.y, bx.r, 0.f);
            }
            s_rowc[tid] = rc;
        } else if (tid - 64 < nc) {
            s_col[tid - 64] = boxes[cb * 64 + tid - 64];
        }
        __syncthreads();
        const bool diag = rb == cb;
        {   // stage 1: bounding circles, all pairs.  Thread = (column c, row parity): 32 rows against one column,
            // hits collected in a register bit mask and compacted ONCE per tile (a ballot + atomic per 32 pairs
            // was 65 % of the kernel's instructions: 16 % of the pairs pass, so every warp iteration paid for it)
            const int c = tid & 63, rhalf = tid >> 6;
            unsigned hits = 0u;
            if (c < nc) {
                const float cx = s_col[c].x, cy = s_col[c].y, cr = s_col[c].r;
#pragma unroll 8
                for (int k = 0; k < 32; k++) {
                    const int r = 2 * k + rhalf;
                    const float4 rc = s_rowc[r];  // x, y, radius (-1e30 past the last row): one broadcast load
                    const float rs = rc.z + cr, dx = rc.x - cx, dy = rc.y - cy;
                    const bool cand = (rs >= 0.f) && !(dx * dx + dy * dy > rs * rs) && (!diag || c > r);  // == rbox_may_overlap
                    hits |= (cand ? 1u : 0u) << k;
                }
            }
            // exclusive prefix of the per-thread hit counts over the CTA
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
            if (tid == kNmsThreads - 1) s_count = pos + mine;
            while (hits) {
                const int k = __ffs(hits) - 1;
                hits &= hits - 1;
                s_queue[pos++] = (unsigned short)(((2 * k + rhalf) << 6) | c);
            }
        }
        __syncthreads();
        const int cnt = s_count;
        for (int q0 = 0; q0 < cnt; q0 += kQ2) {
            // stage 2: axis-aligned bound; stage 3: strip bound (1.03x the truly suppressing pairs survive)
            const int n2 = compact_queue(s_queue + q0, min(kQ2, cnt - q0), s_queue2, &s_count2, s_wsum,
                                         [&](int p) { return !rbox_iou_below(s_row[p >> 6], s_col[p & 63], thr); });
            const int n3 = compact_queue(s_queue2, n2, s_queue3, &s_count3, s_wsum,
                                         [&](int p) { return !rbox_iou_below_strips(s_row[p >> 6], s_col[p & 63], thr); });
            // stage 4: exact clipper
            for (int qi = tid; qi < n3; qi += kNmsThreads) {
                const int p = s_queue3[qi];
                const int r = p >> 6, c = p & 63;
                const int a = rb * 64 + r, b = cb * 64 + c;
                const float iou_ab = rotated_iou_pair<kNmsThreads>(s_row[r], s_col[c], s_pts + tid);
                const bool d_ab = GE ? iou_ab >= thr : iou_ab > thr;
                bool d_ba = d_ab;
                if (fabsf(iou_ab - thr) <= 1e-5f) {
                    const float iou_ba = rotated_iou_pair<kNmsThreads>(s_col[c], s_row[r], s_pts + tid);
                    d_ba = GE ? iou_ba >= thr : iou_ba > thr;
                }
                if (d_ab) atomicOr(&ov[(size_t)a * pitch + (b >> 6)], 1ull << (b & 63));
                if (d_ba) atomicOr(&ov[(size_t)b * pitch + (a >> 6)], 1ull << (a & 63));
            }
        }
    }
}

template <bool GE>
__global__ void __launch_bounds__(kNmsThreads, 8)
ov_filter_kernel(const RBox* __restrict__ boxes, int n, float thr, int2* __restrict__ pairs, unsigned int cap,
                 unsigned int* __restrict__ pair_count, uint8_t* __restrict__ tile_flags) {
    __shared__ RBox s_row[64];
    __shared__ RBox s_col[64];
    __shared__ unsigned short s_queue[64 * 64];
    constexpr int kQ2 = 1024;
    __shared__ unsigned short s_queue2[kQ2];
    __shared__ unsigned short s_queue3[kQ2];
    __shared__ unsigned int s_base;
    __shared__ float4 s_rowc[64];
    __shared__ int s_wsum[kNmsThreads / 32];
    __shared__ int s_count;
    __shared__ int s_count2;  // one counter per stage: a stage's result is still being read when the next one resets its own
    __shared__ int s_count3;
    const int tid = threadIdx.x, lane = tid & 31;
    const int T = (n + 63) >> 6;
    const int total = T * (T + 1) / 2;
    // one tile per CTA when the grid covers them all (the usual case: the block scheduler balances the uneven
    // tiles and no CTA waits on a global counter), grid-stride otherwise
    for (int u = blockIdx.x; u < total; u += gridDim.x) {
        __syncthreads();
        int rb = (int)(((2.0 * T + 1.0) - sqrt((2.0 * T + 1.0) * (2.0 * T + 1.0) - 8.0 * (double)u)) * 0.5);
        rb = max(0, min(rb, T - 1));
        while (rb > 0 && rb * T - rb * (rb - 1) / 2 > u) rb--;
        while ((rb + 1) * T - (rb + 1) * rb / 2 <= u) rb++;
        const int cb = rb + (u - (rb * T - rb * (rb - 1) / 2));
        const int nr = min(64, n - rb * 64), nc = min(64, n - cb * 64);
        if (tid < 64) {
            float4 rc = make_float4(0.f, 0.f, -1e30f, 0.f);
            if (tid < nr) {
                const RBox bx = boxes[rb * 64 + tid];
                s_row[tid] = bx;
                rc = make_float4(bx.x, bx.y, bx.r, 0.f);
            }
            s_rowc[tid] = rc;
        } else if (tid - 64 < nc) {
            s_col[tid - 64] = boxes[cb * 64 + tid - 64];
        }
        __syncthreads();
        const bool diag = rb == cb;
        {   // stage 1: bounding circles, all pairs.  Thread = (column c, row parity): 32 rows against one column,
            // hits collected in a register bit mask and compacted ONCE per tile (a ballot + atomic per 32 pairs
            // was 65 % of the kernel's instructions: 16 % of the pairs pass, so every warp iteration paid for it)
            const int c = tid & 63, rhalf = tid >> 6;
            unsigned hits = 0u;
            if (c < nc) {
                const float cx = s_col[c].x, cy = s_col[c].y, cr = s_col[c].r;
#pragma unroll 8
                for (int k = 0; k < 32; k++) {
                    const int r = 2 * k + rhalf;
                    const float4 rc = s_rowc[r];  // x, y, radius (-1e30 past the last row): one broadcast load
                    const float rs = rc.z + cr, dx = rc.x - cx, dy = rc.y - cy;
                    const bool cand = (rs >= 0.f) && !(dx * dx + dy * dy > rs * rs) && (!diag || c > r);  // == rbox_may_overlap
                    hits |= (cand ? 1u : 0u) << k;
                }
            }
            // exclusive prefix of the per-thread hit counts over the CTA
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
            if (tid == kNmsThreads - 1) s_count = pos + mine;
            while (hits) {
                const int k = __ffs(hits) - 1;
                hits &= hits - 1;
                s_queue[pos++] = (unsigned short)(((2 * k + rhalf) << 6) | c);
            }
        }
        __syncthreads();
        const int cnt = s_count;
        for (int q0 = 0; q0 < cnt; q0 += kQ2) {
            // stage 2: axis-aligned bound; stage 3: strip bound (1.03x the truly suppressing pairs survive)
            const int n2 = compact_queue(s_queue + q0, min(kQ2, cnt - q0), s_queue2, &s_count2, s_wsum,
                                         [&](int p) { return !rbox_iou_below(s_row[p >> 6], s_col[p & 63], thr); });
            const int n3 = compact_queue(s_queue2, n2, s_queue3, &s_count3, s_wsum,
                                         [&](int p) { return !rbox_iou_below_strips(s_row[p >> 6], s_col[p & 63], thr); });
            // survivors go to the global pair queue (ov_clip_kernel evens them out over the whole GPU); a tile
            // that does not fit is flagged and redone by ov_tiles_kernel
            if (tid == 0) {
                const unsigned int base = n3 ? atomicAdd(pair_count, (unsigned int)n3) : 0u;
                if (n3 && base + (unsigned int)n3 > cap) { tile_flags[u] = 1; atomicAdd(pair_count + 1, 1u); }
                s_base = base;
            }
            __syncthreads();
            // a reservation that straddles the end still fills its slots below `cap` (ov_clip_kernel reads every slot
            // below min(count, cap)); the flagged tile is redone as a whole, the duplicates are idempotent ORs
            const unsigned int base = s_base;
            for (int qi = tid; qi < n3; qi += kNmsThreads) {
                if (base + (unsigned int)qi < cap) {
                    const int p = s_queue3[qi];
                    pairs[base + qi] = make_int2(rb * 64 + (p >> 6), cb * 64 + (p & 63));
                }
            }
            __syncthreads();
        }
    }
}

// exact clipper over the global pair queue: one pair per thread, grid-stride, perfectly balanced
template <bool GE>
__global__ void __launch_bounds__(kNmsThreads, 8)
ov_clip_kernel(const RBox* __restrict__ boxes, const int2* __restrict__ pairs, unsigned int cap, const unsigned int* __restrict__ pair_count,
               float thr, unsigned long long* __restrict__ ov, int pitch) {
    __shared__ float2 s_pts[24 * kNmsThreads];
    const unsigned int count = min(*pair_count, cap);
    const int tid = threadIdx.x;
    for (unsigned int i = blockIdx.x * kNmsThreads + tid; i < count; i += gridDim.x * kNmsThreads) {
        const int2 pr = pairs[i];
        const RBox A = boxes[pr.x], B = boxes[pr.y];
        const float iou_ab = rotated_iou_pair<kNmsThreads>(A, B, s_pts + tid);
        const bool d_ab = GE ? iou_ab >= thr : iou_ab > thr;
        bool d_ba = d_ab;
        if (fabsf(iou_ab - thr) <= 1e-5f) {
            const float iou_ba = rotated_iou_pair<kNmsThreads>(B, A, s_pts + tid);
            d_ba = GE ? iou_ba >= thr : iou_ba > thr;
        }
        if (d_ab) atomicOr(&ov[(size_t)pr.x * pitch + (pr.y >> 6)], 1ull << (pr.y & 63));
        if (d_ba) atomicOr(&ov[(size_t)pr.y * pitch + (pr.x >> 6)], 1ull << (pr.x & 63));
    }
}

// greedy scan of one class through the shared matrix: `remv` lives in ORIGINAL box-index space (a kept
// box ORs its whole matrix row; bits that land on already-decided boxes are harmless), the 64x64
// diagonal block of the class order is gathered bit by bit (256 threads, warp ballots).
__global__ void __launch_bounds__(kReduceThreads, 1)
reduce_ov_kernel(SegTable tb, const int* __restrict__ idx_ls, int cand_per_box, const unsigned long long* __restrict__ ov,
                 int pitch, int n_boxes, uint8_t* __restrict__ keep_sorted) {
    extern __shared__ unsigned long long s_remv[];
    __shared__ int s_box2[2][64];  // double-buffered: the OR phase of block b overlaps the loads of block b+1
    __shared__ unsigned int s_diag32[128];
    __shared__ unsigned int s_rem32[2];
    __shared__ unsigned long long s_keep;
    const int tid = threadIdx.x, lane = tid & 31;
    const int nseg = tb.hdr[0];
    const int T = (n_boxes + 63) >> 6;
    for (int s = blockIdx.x; s < nseg; s += gridDim.x) {
        const int st = tb.seg_start[s];
        const int ns = tb.seg_start[s + 1] - st;
        const int nblk = (ns + 63) >> 6;
        __syncthreads();
        for (int j = tid; j < T; j += kReduceThreads) s_remv[j] = 0ull;
        for (int b = 0; b < nblk; b++) {
            const int nr = min(64, ns - b * 64);
            int* s_box = s_box2[b & 1];
            if (tid < 64) s_box[tid] = tid < nr ? idx_ls[st + b * 64 + tid] / cand_per_box : -1;
            __syncthreads();  // also orders the previous block's OR phase before the reads below
            if (tid < 64) {
                const int a = s_box[tid];
                const bool rem = a < 0 || ((s_remv[a >> 6] >> (a & 63)) & 1ull);
                const unsigned m = __ballot_sync(0xffffffffu, rem);
                if (lane == 0) s_rem32[tid >> 5] = m;
            }
#pragma unroll 4
            for (int it = 0; it < 16; it++) {
                const int idx = it * kReduceThreads + tid;
                const int i = idx >> 6, j = idx & 63;
                bool bit = false;
                if (i < nr && j < nr && j > i) {
                    const int a = s_box[i], c = s_box[j];
                    bit = (ov[(size_t)a * pitch + (c >> 6)] >> (c & 63)) & 1ull;
                }
                const unsigned m = __ballot_sync(0xffffffffu, bit);
                if (lane == 0) s_diag32[idx >> 5] = m;
            }
            __syncthreads();
            if (tid == 0) {
                unsigned long long r = (unsigned long long)s_rem32[0] | ((unsigned long long)s_rem32[1] << 32), kb = 0ull;
#pragma unroll
                for (int i = 0; i < 64; i++) {
                    const bool alive = ((r >> i) & 1ull) == 0ull;
                    const unsigned long long d = (unsigned long long)s_diag32[2 * i] | ((unsigned long long)s_diag32[2 * i + 1] << 32);
                    kb |= alive ? (1ull << i) : 0ull;
                    r |= alive ? d : 0ull;
                }
                s_keep = kb;
            }
            __syncthreads();
            const unsigned long long kb = s_keep;
            if (tid < nr) keep_sorted[st + b * 64 + tid] = (uint8_t)((kb >> tid) & 1ull);
            if (kb && b + 1 < nblk) {
                const int jj = tid & 63, rg = tid >> 6;
                const unsigned kb16 = (unsigned)((kb >> (rg * 16)) & 0xffffull);
                if (kb16) {
                    for (int w = jj; w < T; w += 64) {
                        unsigned long long acc = 0ull;
#pragma unroll
                        for (int i = 0; i < 16; i++)
                            if ((kb16 >> i) & 1u) acc |= ov[(size_t)s_box[rg * 16 + i] * pitch + w];
                        if (acc) atomicOr(&s_remv[w], acc);
                    }
                }
            }
        }
    }
}

// Staged variant of the scan above for n_boxes <= 8192 (the per-tile case: 4000 boxes -> 63 words per row).  The
// matrix rows a class will need do not depend on its keep decisions, so block b+1's 64 rows are loaded into
// registers (16-byte loads, one warp per row; the row pitch in global memory is even) while block b is
// resolved from shared memory, and stored to the other shared buffer at the end of the block.  Per block:
//   gather  thread (j, quarter) extracts "i suppresses j" for 16 rows i -> 64 column masks   (16 independent LDS)
//   resolve one warp, fixed point over the column masks                                      (a few ballots)
//   OR      remv |= rows of the kept candidates, 4 partial ORs per word then one merge       (no atomics)
// Measured on B200 (clock64, 4000 candidates per class): 7 900 cycles per block for the L2-resident variant
// (two dependent L2 round trips in gather and OR) -> see profiles/README.md for this one.
// IDENT = true is the same scan for the generic engine's block-sparse mask: rows and bit positions are the
// group's own sorted positions (candidate p -> row p, bit p), the pitch is the group's ceil(n_s / 64), and
// groups of >= kCoopMinBlocks blocks are left to reduce_kernel's cooperative phase.
template <int NCH, bool IDENT>  // NCH 64-word chunks per row: 1 (<= 4096 columns) or 2 (<= 8192)
__global__ void __launch_bounds__(kReduceThreads, 1)
reduce_ov_staged_kernel(SegTable tb, const int* __restrict__ idx_ls, int cand_per_box, const unsigned long long* __restrict__ ov_base,
                        int pitch_arg, int n_boxes_arg, uint8_t* __restrict__ keep_sorted, const int* __restrict__ gate,
                        const int* __restrict__ seg_count = nullptr, int* __restrict__ keep_prefix = nullptr,
                        int* __restrict__ kept_count = nullptr, int* __restrict__ kept_pos = nullptr) {
    if (gate && *gate == 0) return;
    extern __shared__ unsigned long long s_dyn[];  // [remv: Ts][partials: 4 x Ts][rows: 2 x 64 x Ts][cand: n_boxes ints]
    __shared__ __align__(8) unsigned short s_col16[256];  // s_col16[4j + q]: rows i in quarter q (i < j) that suppress j
    __shared__ unsigned long long s_keep;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nseg = tb.hdr[0];
    for (int s = blockIdx.x; s < nseg; s += gridDim.x) {
        const int st = tb.seg_start[s];
        const int ns_all = seg_count ? seg_count[s] : tb.seg_start[s + 1] - st;   // seg_count: fixed-stride segments (fast multiclass path)
        const int n_boxes = IDENT ? ns_all : n_boxes_arg;
        const int ns = min(ns_all, n_boxes);            // shared matrix: one candidate per (box, class), ns <= n_boxes
        const int nblk = (ns + 63) >> 6;
        const int T = (n_boxes + 63) >> 6;
        if (IDENT && (T >= kCoopMinBlocks || T > 64 * NCH)) continue;
        const int pitch = IDENT ? T : pitch_arg;
        const unsigned long long* ov = IDENT ? ov_base + tb.mask_off[s] : ov_base;
        const int Ts = T | 1;                           // odd shared-memory pitch: lanes on different rows hit different banks
        unsigned long long* s_remv = s_dyn;
        unsigned long long* s_part = s_dyn + Ts;
        unsigned long long* s_rows = s_dyn + 5 * Ts;
        int* s_cand = reinterpret_cast<int*>(s_dyn + 5 * Ts + 2 * 64 * (size_t)Ts);
        __syncthreads();
        for (int j = tid; j < Ts; j += kReduceThreads) s_remv[j] = 0ull;
        if (!IDENT)
            for (int p = tid; p < ns; p += kReduceThreads) s_cand[p] = idx_ls[st + p] / cand_per_box;
        __syncthreads();
        auto cand = [&](int p) { return IDENT ? p : s_cand[p]; };
        // warp w holds rows w, w+8, ..., w+56 of the next block: lane l the words 2l, 2l+1 of every 64-word chunk
        ulonglong2 nxt[8][NCH];
        auto fetch = [&](int b) {
            const int nr = min(64, ns - b * 64);
#pragma unroll
            for (int k = 0; k < 8; k++) {
                const int i = warp + 8 * k;
#pragma unroll
                for (int ch = 0; ch < NCH; ch++) {
                    const int w = ch * 64 + 2 * lane;
                    nxt[k][ch] = make_ulonglong2(0ull, 0ull);
                    if (i < nr && w < pitch) {
                        const unsigned long long* src = ov + (size_t)cand(b * 64 + i) * pitch + w;
                        if (IDENT) {  // odd pitches: rows are only 8-byte aligned
                            nxt[k][ch].x = src[0];
                            if (w + 1 < pitch) nxt[k][ch].y = src[1];
                        } else {
                            nxt[k][ch] = *reinterpret_cast<const ulonglong2*>(src);
                        }
                    }
                }
            }
        };
        auto stash = [&](int b) {
            unsigned long long* dst = s_rows + (size_t)(b & 1) * 64 * Ts;
#pragma unroll
            for (int k = 0; k < 8; k++) {
                const int i = warp + 8 * k;
#pragma unroll
                for (int ch = 0; ch < NCH; ch++) {
                    const int w = ch * 64 + 2 * lane;
                    if (w < Ts) dst[i * Ts + w] = nxt[k][ch].x;
                    if (w + 1 < Ts) dst[i * Ts + w + 1] = nxt[k][ch].y;
                }
            }
        };
        if (nblk > 0) { fetch(0); stash(0); }
        __syncthreads();
        int kept_run = 0;   // kept candidates of the blocks before b (fast multiclass path: exclusive prefix for the output ranks)
        for (int b = 0; b < nblk; b++) {
            const int nr = min(64, ns - b * 64);
            const unsigned long long* R = s_rows + (size_t)(b & 1) * 64 * Ts;
            if (b + 1 < nblk) fetch(b + 1);  // in flight while this block is resolved
            {
                const int j = tid & 63, q = tid >> 6;
                unsigned bits = 0u;
                if (j < nr) {
                    const int c = cand(b * 64 + j);
                    const unsigned long long* col = R + (c >> 6);
                    const int sh = c & 63;
#pragma unroll
                    for (int ii = 0; ii < 16; ii++) {
                        const int i = q * 16 + ii;
                        bits |= (unsigned)((col[i * Ts] >> sh) & 1ull) << ii;
                    }
                    // rows i >= j (and rows past the block) do not count
                    const int lim = j - q * 16;
                    bits &= lim >= 16 ? 0xffffu : (lim <= 0 ? 0u : ((1u << lim) - 1u));
                }
                s_col16[4 * j + q] = (unsigned short)bits;
            }
            __syncthreads();
            if (warp == 0) {
                // greedy resolve as a fixed point: a candidate dies once a KEPT lower candidate suppresses it and
                // is kept once every lower candidate that suppresses it is dead; the lowest undecided candidate
                // is always decidable, so the loop ends after at most 64 rounds (a handful in practice).
                unsigned long long col[2];
                bool und[2];
                unsigned long long dead = 0ull, kept = 0ull;
#pragma unroll
                for (int h = 0; h < 2; h++) {
                    const int j = lane + 32 * h;
                    col[h] = *reinterpret_cast<const unsigned long long*>(&s_col16[4 * j]);
                    const int a = j < nr ? cand(b * 64 + j) : -1;
                    const bool rem = a < 0 || ((s_remv[a >> 6] >> (a & 63)) & 1ull);
                    dead |= (unsigned long long)__ballot_sync(0xffffffffu, rem) << (32 * h);
                    und[h] = !rem;
                }
                while (true) {
                    bool nd[2], nk[2];
#pragma unroll
                    for (int h = 0; h < 2; h++) {
                        nd[h] = und[h] && (col[h] & kept) != 0ull;
                        nk[h] = und[h] && !nd[h] && (col[h] & ~dead) == 0ull;
                        und[h] = und[h] && !nd[h] && !nk[h];
                    }
                    const unsigned long long d2 = (unsigned long long)__ballot_sync(0xffffffffu, nd[0]) |
                                                  ((unsigned long long)__ballot_sync(0xffffffffu, nd[1]) << 32);
                    const unsigned long long k2 = (unsigned long long)__ballot_sync(0xffffffffu, nk[0]) |
                                                  ((unsigned long long)__ballot_sync(0xffffffffu, nk[1]) << 32);
                    if ((d2 | k2) == 0ull) break;
                    dead |= d2;
                    kept |= k2;
                }
                if (lane == 0) s_keep = kept;
            }
            __syncthreads();
            const unsigned long long kb = s_keep;
            if (tid < nr) {
                keep_sorted[st + b * 64 + tid] = (uint8_t)((kb >> tid) & 1ull);
                if (keep_prefix) {   // fast multiclass path: exclusive prefix of the keep flags and the compacted kept list
                    const int pre = kept_run + __popcll(kb & ((1ull << tid) - 1ull));
                    keep_prefix[st + b * 64 + tid] = pre;
                    if ((kb >> tid) & 1ull) kept_pos[st + pre] = b * 64 + tid;
                }
            }
            kept_run += __popcll(kb);
            {
                // partial ORs: row group rg = tid / 64 covers 16 rows, lane column w (+64 for the second chunk)
                const int jj = tid & 63, rg = tid >> 6;
                const unsigned kb16 = (unsigned)((kb >> (rg * 16)) & 0xffffull);
#pragma unroll
                for (int ch = 0; ch < NCH; ch++) {
                    const int w = ch * 64 + jj;
                    if (w < Ts) {
                        unsigned long long acc = 0ull;
#pragma unroll
                        for (int i = 0; i < 16; i++) acc |= ((kb16 >> i) & 1u) ? R[(rg * 16 + i) * Ts + w] : 0ull;
                        s_part[rg * Ts + w] = acc;
                    }
                }
            }
            if (b + 1 < nblk) stash(b + 1);
            __syncthreads();
            for (int w = tid; w < Ts; w += kReduceThreads)
                s_remv[w] |= s_part[w] | s_part[Ts + w] | s_part[2 * Ts + w] | s_part[3 * Ts + w];
            __syncthreads();  // next block's rows and this block's ORs are in place
        }
        if (kept_count && tid == 0) kept_count[s] = kept_run;
    }
}

// Software-pipelined form of the staged scan for the shared decision matrix (IDENT = false): the column masks of block
// b+1 do not depend on the running suppression mask, so warps 1-7 extract them (from rows staged one block earlier)
// WHILE warp 0 resolves block b.  A column mask is read with lanes = rows (odd row pitch: conflict-free, the staged
// kernel's lanes = candidates read arbitrary columns of one row: 4-5 way bank conflicts) and assembled by two ballots;
// the kept rows are ORed into the mask with native 32-bit shared-memory atomics, which removes the partial-OR merge
// pass.  Three row buffers (block b for the OR, b+1 for the extraction, b+2 arriving), two
// column mask buffers, two block barriers per block instead of four.  Same decisions and outputs as reduce_ov_staged_kernel.
// column masks of the candidates first, first + STRIDE, ... (< 64) of a block, by one warp: lanes = rows.  All loads of
// the warp's candidates are issued before the first ballot (two warps per scheduler: latency is hidden by ILP only).
template <int STRIDE>
__device__ __forceinline__ void colmask_warp(const unsigned long long* __restrict__ R, int Ts, const int* __restrict__ cand, int nr,
                                             int first, int lane, unsigned long long* __restrict__ out) {
    constexpr int MAXJ = (64 + STRIDE - 1) / STRIDE;
    int c[MAXJ];
    unsigned long long v0[MAXJ], v1[MAXJ];
#pragma unroll
    for (int u = 0; u < MAXJ; u++) {
        const int j = first + u * STRIDE;
        c[u] = j < nr ? cand[j] : -1;
    }
#pragma unroll
    for (int u = 0; u < MAXJ; u++) {
        const int w = c[u] >= 0 ? c[u] >> 6 : 0;
        v0[u] = R[lane * Ts + w];
        v1[u] = R[(lane + 32) * Ts + w];
    }
#pragma unroll
    for (int u = 0; u < MAXJ; u++) {
        const int j = first + u * STRIDE;
        if (j < 64) {                                        // warp-uniform
            const int sh = c[u] & 63;
            const unsigned lo = __ballot_sync(0xffffffffu, (v0[u] >> sh) & 1ull);
            const unsigned hi = __ballot_sync(0xffffffffu, (v1[u] >> sh) & 1ull);
            unsigned long long m = ((unsigned long long)hi << 32) | lo;
            m = c[u] >= 0 ? m & ((1ull << j) - 1ull) : 0ull;   // rows i >= j do not count (rows past the block are zero)
            if (lane == 0) out[j] = m;
        }
    }
}

template <int NCH, int THREADS>   // THREADS: 256 or 512 (more warps = more latency hiding for a kernel of dependent shared-memory steps)
__global__ void __launch_bounds__(THREADS, 1)
reduce_ov_pipe_kernel(SegTable tb, const int* __restrict__ idx_ls, int cand_per_box, const unsigned long long* __restrict__ ov,
                      int pitch, int n_boxes, uint8_t* __restrict__ keep_sorted, const int* __restrict__ seg_count,
                      int* __restrict__ keep_prefix, int* __restrict__ kept_count, int* __restrict__ kept_pos) {
    extern __shared__ unsigned long long s_dyn[];  // [remv: Ts][rows: 3 x 64 x Ts][cand: n_boxes ints]
    __shared__ unsigned long long s_colmask[2][64];          // [buffer][j]: rows i < j of the block that suppress candidate j
    __shared__ unsigned long long s_keep;
    constexpr int NW = THREADS / 32, RPW = 64 / NW;     // warps; rows of a block per warp
    constexpr int NG = THREADS / 64, RPG = 64 / NG;     // row groups of the OR phase; rows per group
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nseg = tb.hdr[0];
    const int T = (n_boxes + 63) >> 6, Ts = T | 1;
    unsigned long long* s_remv = s_dyn;
    unsigned long long* s_rows = s_dyn + Ts;
    int* s_cand = reinterpret_cast<int*>(s_dyn + Ts + 3 * 64 * (size_t)Ts);
    for (int s = blockIdx.x; s < nseg; s += gridDim.x) {
        const int st = tb.seg_start[s];
        const int ns = min(seg_count ? seg_count[s] : tb.seg_start[s + 1] - st, n_boxes);
        const int nblk = (ns + 63) >> 6;
        __syncthreads();
        for (int j = tid; j < Ts; j += THREADS) s_remv[j] = 0ull;
        for (int p = tid; p < ns; p += THREADS) s_cand[p] = idx_ls[st + p] / cand_per_box;
        __syncthreads();
        ulonglong2 nxt[RPW][NCH];   // warp w: rows w, w+NW, ... of a block; lane l: words 2l, 2l+1 of every 64-word chunk
        auto fetch = [&](int b) {
            const int nr = min(64, ns - b * 64);
#pragma unroll
            for (int k = 0; k < RPW; k++) {
                const int i = warp + NW * k;
#pragma unroll
                for (int ch = 0; ch < NCH; ch++) {
                    const int w = ch * 64 + 2 * lane;
                    nxt[k][ch] = make_ulonglong2(0ull, 0ull);
                    if (i < nr && w < pitch)
                        nxt[k][ch] = *reinterpret_cast<const ulonglong2*>(ov + (size_t)s_cand[b * 64 + i] * pitch + w);
                }
            }
        };
        auto stash = [&](int b) {
            unsigned long long* dst = s_rows + (size_t)(b % 3) * 64 * Ts;
#pragma unroll
            for (int k = 0; k < RPW; k++) {
                const int i = warp + NW * k;
#pragma unroll
                for (int ch = 0; ch < NCH; ch++) {
                    const int w = ch * 64 + 2 * lane;
                    if (w < Ts) dst[i * Ts + w] = nxt[k][ch].x;
                    if (w + 1 < Ts) dst[i * Ts + w + 1] = nxt[k][ch].y;
                }
            }
        };
        if (nblk > 0) { fetch(0); stash(0); }
        if (nblk > 1) { fetch(1); stash(1); }
        __syncthreads();
        if (nblk > 0) colmask_warp<NW>(s_rows, Ts, s_cand, min(64, ns), warp, lane, s_colmask[0]);
        if (nblk > 2) fetch(2);                     // in flight during iteration 0
        __syncthreads();
        int kept_run = 0;
        for (int b = 0; b < nblk; b++) {
            const int nr = min(64, ns - b * 64);
            if (warp == 0) {
                // greedy resolve as a fixed point (see reduce_ov_staged_kernel)
                unsigned long long col[2];
                bool und[2];
                unsigned long long dead = 0ull, kept = 0ull;
#pragma unroll
                for (int h = 0; h < 2; h++) {
                    const int j = lane + 32 * h;
                    col[h] = s_colmask[b & 1][j];
                    const int a = j < nr ? s_cand[b * 64 + j] : -1;
                    const bool rem = a < 0 || ((s_remv[a >> 6] >> (a & 63)) & 1ull);
                    dead |= (unsigned long long)__ballot_sync(0xffffffffu, rem) << (32 * h);
                    und[h] = !rem;
                }
                while (true) {
                    bool nd[2], nk[2];
#pragma unroll
                    for (int h = 0; h < 2; h++) {
                        nd[h] = und[h] && (col[h] & kept) != 0ull;
                        nk[h] = und[h] && !nd[h] && (col[h] & ~dead) == 0ull;
                        und[h] = und[h] && !nd[h] && !nk[h];
                    }
                    const unsigned long long d2 = (unsigned long long)__ballot_sync(0xffffffffu, nd[0]) |
                                                  ((unsigned long long)__ballot_sync(0xffffffffu, nd[1]) << 32);
                    const unsigned long long k2 = (unsigned long long)__ballot_sync(0xffffffffu, nk[0]) |
                                                  ((unsigned long long)__ballot_sync(0xffffffffu, nk[1]) << 32);
                    if ((d2 | k2) == 0ull) break;
                    dead |= d2;
                    kept |= k2;
                }
                if (lane == 0) s_keep = kept;
            } else if (b + 1 < nblk) {
                colmask_warp<NW - 1>(s_rows + (size_t)((b + 1) % 3) * 64 * Ts, Ts, s_cand + (b + 1) * 64,
                                                      min(64, ns - (b + 1) * 64), warp - 1, lane, s_colmask[(b + 1) & 1]);
            }
            __syncthreads();
            const unsigned long long kb = s_keep;
            if (tid < nr) {
                keep_sorted[st + b * 64 + tid] = (uint8_t)((kb >> tid) & 1ull);
                if (keep_prefix) {
                    const int pre = kept_run + __popcll(kb & ((1ull << tid) - 1ull));
                    keep_prefix[st + b * 64 + tid] = pre;
                    if ((kb >> tid) & 1ull) kept_pos[st + pre] = b * 64 + tid;
                }
            }
            kept_run += __popcll(kb);
            {
                // OR of the kept rows into the running mask: row group rg = tid / 64 covers RPG rows, lane column w (+64 for
                // the second chunk); the four groups meet in native 32-bit shared-memory atomics (a 64-bit OR is a CAS loop)
                const unsigned long long* R = s_rows + (size_t)(b % 3) * 64 * Ts;
                const int jj = tid & 63, rg = tid >> 6;
                const unsigned kbg = (unsigned)((kb >> (rg * RPG)) & ((1ull << RPG) - 1ull));
                if (kbg) {
#pragma unroll
                    for (int ch = 0; ch < NCH; ch++) {
                        const int w = ch * 64 + jj;
                        if (w < Ts) {
                            unsigned long long acc = 0ull;
#pragma unroll
                            for (int i = 0; i < RPG; i++) acc |= ((kbg >> i) & 1u) ? R[(rg * RPG + i) * Ts + w] : 0ull;
                            unsigned* dst = reinterpret_cast<unsigned*>(&s_remv[w]);
                            if ((unsigned)acc) atomicOr(dst, (unsigned)acc);
                            if ((unsigned)(acc >> 32)) atomicOr(dst + 1, (unsigned)(acc >> 32));
                        }
                    }
                }
            }
            if (b + 2 < nblk) stash(b + 2);
            if (b + 3 < nblk) fetch(b + 3);
            __syncthreads();
        }
        if (kept_count && tid == 0) kept_count[s] = kept_run;
    }
}

// ----------------------------------------------------------------------------- outputs
__global__ void scatter_keep_kernel(const uint8_t* __restrict__ keep_sorted, const int* __restrict__ idx, int n_max,
                                    const int* __restrict__ n_dev, uint8_t* __restrict__ keep_mask) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_max) return;
    int n = n_dev ? min(*n_dev, n_max) : n_max;
    keep_mask[idx[p]] = p < n ? keep_sorted[p] : (uint8_t)0;
}

__global__ void score_order_flags_kernel(const uint8_t* __restrict__ keep_mask, const int* __restrict__ idx_score, int n_max,
                                         uint8_t* __restrict__ flags, int64_t* __restrict__ vals) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_max) return;
    int i = idx_score[p];
    flags[p] = keep_mask[i];
    vals[p] = (int64_t)i;
}

// ----------------------------------------------------------------------------- engine

// ----------------------------------------------------------------------------- sparse greedy NMS (merge stage)
// A 10k x 10k scene holds ~10^5 small detections: the dense engine tests n_s^2 / 2 hbb pairs per (scene, class)
// group and scans n_s / 64 dependent blocks (7.3 ms for 90k detections, 90 % in those two kernels).  The overlap
// graph is sparse (~10 neighbours per detection), so for large MERGE calls:
//   1. sweep and prune: detections sorted by (group, x1); each looks ahead while the next x1 is left of its x2
//      and keeps the pairs whose hbbs overlap (the reference's prefilter, result_merge.py:97-100) -- counted, prefix
//      summed and written without atomics;
//   2. the polygon IoU of every candidate pair, one per thread; "p suppresses q" (p the higher-scored one) becomes an
//      in-edge of q in a CSR graph (degree count -> prefix sum -> fill);
//   3. greedy NMS as a FIXED POINT over that graph, the same rule as the staged scan's warp resolve: a detection
//      dies once a KEPT in-neighbour exists, is kept once all its in-neighbours are dead.  The highest-scored
//      undecided detection is always decidable, so this is exactly the sequential greedy result; the number of
//      rounds is the longest kept/dead dependency chain (a handful).  One persistent kernel with a grid barrier.
// Anything that does not fit the workspace carved from the (unused) dense mask falls back to the dense kernels,
// which are always enqueued and exit on a device flag.
constexpr int kSparseMinBoxes = 8192;
constexpr int kSparseCtas = kNumSMs;
constexpr int kSparseThreads = 512;

struct SparseWs {
    unsigned long long *keyA, *keyB;   // (group << 32 | ordered float x1), double buffer
    int *valA, *valB;                  // sorted position of the detection
    int* seg_of;                       // group index of a sorted position
    int* cnt;                          // n+1: candidates found by each x-sorted detection -> exclusive prefix
    int* indeg;                        // n+1: in-degree -> row pointers
    int* cursor;                       // n: fill cursors
    unsigned char* state;              // n: 0 undecided, 1 kept, 2 dead
    unsigned long long* cand;          // capC: (dst << 32 | src)
    unsigned char* flag;               // capC: candidate suppresses
    int* adj;                          // capE: in-neighbours (sources)
    int* ctl;                          // [0] gate (1 = run the dense path) [1] barrier count [2] barrier generation [3..4] changed
    long long capC, capE;
};

__device__ __forceinline__ unsigned int ord_f32(float f) {
    unsigned int u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord_f32_inv(unsigned int u) {
    return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

// What the sparse path needs to know about a box type: an axis-aligned extent (sweep order / bands), the candidate
// test of the sweep (cheap, exact: it may only drop pairs that cannot suppress) and the suppression predicate.
template <int KIND> struct SpAdapt;
template <> struct SpAdapt<RSDET_NMS_MERGE> {
    using Box = MBox;
    static constexpr int kScratchSlots = 0;
    __device__ static double x1(const Box& b) { return b.x1; }
    __device__ static double x2(const Box& b) { return b.x2; }
    __device__ static double y1(const Box& b) { return b.y1; }
    __device__ static double y2(const Box& b) { return b.y2; }
    __device__ static bool cand(const Box& a, const Box& b, double) { return merge_hbb_overlap(a, b); }
    // survivors are `iou <= thr` (result_merge.py:118)
    __device__ static bool sup(const Box& a, const Box& b, double thr, float2*) { return !(iou_poly_d(a, b) <= thr); }
};
// rotated boxes (dense single-stage candidates, BASELINE config 4): extent = the square around the bounding circle;
// candidates = circles overlap and the axis-aligned upper bound of the IoU does not already rule the pair out;
// predicate = strip bound, then the exact clipper (the same cascade as mask_tiles_kernel, so decisions are identical)
template <bool GE> struct SpAdaptRot {
    using Box = RBox;
    static constexpr int kScratchSlots = 24;
    __device__ static double x1(const Box& b) { return (double)b.x - (double)fmaxf(b.r, 0.f); }
    __device__ static double x2(const Box& b) { return (double)b.x + (double)fmaxf(b.r, 0.f); }
    __device__ static double y1(const Box& b) { return (double)b.y - (double)fmaxf(b.r, 0.f); }
    __device__ static double y2(const Box& b) { return (double)b.y + (double)fmaxf(b.r, 0.f); }
    __device__ static bool cand(const Box& a, const Box& b, double thr) {
        return rbox_may_overlap(a, b) && !rbox_iou_below(a, b, (float)thr);
    }
    __device__ static bool sup(const Box& a, const Box& b, double thr, float2* q) {
        if (rbox_iou_below_strips(a, b, (float)thr)) return false;
        const float iou = rotated_iou_pair<kNmsThreads>(a, b, q);
        return GE ? iou >= (float)thr : iou > (float)thr;
    }
};
template <> struct SpAdapt<RSDET_NMS_ROTATED> : SpAdaptRot<false> {};
template <> struct SpAdapt<RSDET_NMS_ROTATED_GE> : SpAdaptRot<true> {};

// ctl[5], ctl[6]: float bits of the largest extent height / width (positive floats order like ints)
template <int KIND>
__global__ void sp_extent_kernel(const typename SpAdapt<KIND>::Box* __restrict__ boxes, SegTable tb, int n_max, SparseWs w) {
    using A = SpAdapt<KIND>;
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    const int n_eff = min(tb.hdr[1], n_max);
    float h = 0.f, wd = 0.f;
    if (p < n_eff) {
        h = __double2float_ru(A::y2(boxes[p]) - A::y1(boxes[p]));
        wd = __double2float_ru(A::x2(boxes[p]) - A::x1(boxes[p]));
    }
    for (int o = 16; o; o >>= 1) {
        h = fmaxf(h, __shfl_xor_sync(0xffffffffu, h, o));
        wd = fmaxf(wd, __shfl_xor_sync(0xffffffffu, wd, o));
    }
    if ((threadIdx.x & 31) == 0) {
        if (h > 0.f) atomicMax(w.ctl + 5, __float_as_int(h));
        if (wd > 0.f) atomicMax(w.ctl + 6, __float_as_int(wd));
    }
}

// y band of a coordinate: bands are as high as the tallest hbb of the call, so a box touches its own band and at most
// the next one.  Out-of-range bands are clamped (that only merges bands, i.e. adds candidates).
constexpr int kBandBits = 14;
__device__ __forceinline__ unsigned int sp_band(double y, double band_h) {
    const double b = floor(y / band_h) + (double)(1 << (kBandBits - 1));
    return (unsigned int)fmin(fmax(b, 0.0), (double)((1 << kBandBits) - 1));
}
__device__ __forceinline__ double sp_band_h(const SparseWs& w) { return fmax((double)__int_as_float(w.ctl[5]) * 1.000001, 1e-6); }

template <int KIND>
__global__ void sp_keys_kernel(const typename SpAdapt<KIND>::Box* __restrict__ boxes, SegTable tb, int n_max, SparseWs w) {
    using A = SpAdapt<KIND>;
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p > n_max) return;
    if (p == n_max) { w.cnt[p] = 0; w.indeg[p] = 0; return; }
    w.cnt[p] = 0; w.indeg[p] = 0; w.cursor[p] = 0; w.state[p] = 0;
    const int n_eff = min(tb.hdr[1], n_max), nseg = tb.hdr[0];
    w.valA[p] = p;
    if (p >= n_eff) { w.keyA[p] = ~0ull; w.seg_of[p] = -1; return; }
    int lo = 0, hi = nseg;  // largest s with seg_start[s] <= p
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (tb.seg_start[mid] <= p) lo = mid; else hi = mid;
    }
    w.seg_of[p] = lo;
    // (group | y band | x1 rounded DOWN: never right of the true x1)
    w.keyA[p] = ((unsigned long long)lo << (32 + kBandBits)) | ((unsigned long long)sp_band(A::y1(boxes[p]), sp_band_h(w)) << 32) |
                ord_f32(__double2float_rd(A::x1(boxes[p])));
}

// How many neighbours the sweep below would VISIT in total (two binary searches per detection instead of the walk):
// the sparse path pays off when the overlap graph is sparse -- a 10k x 10k scene, dense single-stage candidates on a
// large canvas -- and loses against the dense tiles in a crowd where every box's x extent covers thousands of
// others (100k boxes on a 1024^2 canvas: 2600 visits per box).  ctl[7] accumulates visits / 64 per warp; the sweep
// hands the call to the dense kernels (gate ctl[0]) when the mean exceeds kSparseMaxVisits per box.
constexpr int kSparseMaxVisits = 640;
template <int KIND>
__global__ void sp_estimate_kernel(const typename SpAdapt<KIND>::Box* __restrict__ boxes, SegTable tb, int n_max,
                                   const unsigned long long* __restrict__ key, const int* __restrict__ val, SparseWs w) {
    using A = SpAdapt<KIND>;
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    const int n_eff = min(tb.hdr[1], n_max);
    unsigned visits = 0;
    if (q < n_eff) {
        const unsigned long long kq = key[q];
        const unsigned int run = (unsigned int)(kq >> 32);
        const auto bi = boxes[val[q]];
        const unsigned int x2k = ord_f32(__double2float_ru(A::x2(bi)));
        auto first_at_or_after = [&](unsigned long long k, int lo) {      // first r >= lo with key[r] >= k
            int hi = n_eff;
            while (lo < hi) { const int mid = (lo + hi) >> 1; if (key[mid] < k) lo = mid + 1; else hi = mid; }
            return lo;
        };
        visits = (unsigned)(first_at_or_after(((unsigned long long)run << 32) | x2k, q + 1) - (q + 1));
        const double band_h = sp_band_h(w);
        const unsigned int band = run & ((1u << kBandBits) - 1u);
        if (band + 1 < (1u << kBandBits) && sp_band(A::y2(bi), band_h) > band) {
            const float maxw = __int_as_float(w.ctl[6]);
            const unsigned long long lo = ((unsigned long long)(run + 1) << 32) | ord_f32(__double2float_rd(A::x1(bi) - (double)maxw * 1.000001));
            const int a = first_at_or_after(lo, q + 1);
            visits += (unsigned)(first_at_or_after(((unsigned long long)(run + 1) << 32) | x2k, a) - a);
        }
    }
    for (int o = 16; o; o >>= 1) visits += __shfl_xor_sync(0xffffffffu, visits, o);
    if ((threadIdx.x & 31) == 0 && visits) atomicAdd((unsigned int*)w.ctl + 7, (visits + 63) >> 6);
}

// FILL = false: count the candidate pairs of each sorted detection; FILL = true: write them at the prefix offsets.
// Candidates of detection i: later members of its own (group, band) run whose x1 is left of x2_i, and -- when i
// reaches into the next band -- the members of that run whose x1 lies in (x1_i - widest hbb, x2_i).
template <int KIND, bool FILL>
__global__ void sp_sweep_kernel(const typename SpAdapt<KIND>::Box* __restrict__ boxes, SegTable tb, int n_max,
                                const unsigned long long* __restrict__ key, const int* __restrict__ val, SparseWs w) {
    using A = SpAdapt<KIND>;
    using Box = typename A::Box;
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    const int n_eff = min(tb.hdr[1], n_max);
    if (q >= n_eff) return;
    if ((unsigned long long)(unsigned int)w.ctl[7] * 64ull > (unsigned long long)kSparseMaxVisits * (unsigned long long)n_eff + 4096ull) {
        if (q == 0) w.ctl[0] = 1;   // a crowd: the dense kernels take the call
        return;
    }
    if (FILL && (long long)w.cnt[n_max] > w.capC) { if (q == 0) w.ctl[0] = 1; return; }
    const unsigned long long kq = key[q];
    const unsigned int run = (unsigned int)(kq >> 32);
    const int i = val[q];
    const Box bi = boxes[i];
    const double bx1 = A::x1(bi), bx2 = A::x2(bi), by2 = A::y2(bi);
    const double thr = tb.seg_thr[w.seg_of[i]];
    int found = 0;
    long long out = FILL ? (long long)w.cnt[q] : 0;
    auto visit = [&](int r0, unsigned int want_run) {
        for (int r = r0; r < n_eff; r++) {
            const unsigned long long kr = key[r];
            if ((unsigned int)(kr >> 32) != want_run) break;
            if (!((double)ord_f32_inv((unsigned int)kr) < bx2)) break;  // every later x1 is at or right of my x2
            const int j = val[r];
            if (A::cand(bi, boxes[j], thr)) {
                if (FILL) {
                    const int src = min(i, j), dst = max(i, j);  // lower sorted position = higher score
                    w.cand[out++] = ((unsigned long long)dst << 32) | (unsigned int)src;
                }
                found++;
            }
        }
    };
    visit(q + 1, run);
    const double band_h = sp_band_h(w);
    const unsigned int band = run & ((1u << kBandBits) - 1u);
    if (band + 1 < (1u << kBandBits) && sp_band(by2, band_h) > band) {
        const unsigned int next_run = run + 1;
        const float maxw = __int_as_float(w.ctl[6]);
        const unsigned long long lokey = ((unsigned long long)next_run << 32) | ord_f32(__double2float_rd(bx1 - (double)maxw * 1.000001));
        int lo = q + 1, hi = n_eff;  // first r with key[r] >= lokey (the next band sorts after mine)
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (key[mid] < lokey) lo = mid + 1; else hi = mid;
        }
        visit(lo, next_run);
    }
    if (!FILL) w.cnt[q] = found;
}

template <int KIND>
__global__ void __launch_bounds__(kNmsThreads) sp_iou_kernel(const typename SpAdapt<KIND>::Box* __restrict__ boxes, SegTable tb,
                                                             int n_max, SparseWs w) {
    using A = SpAdapt<KIND>;
    __shared__ float2 s_pts[A::kScratchSlots ? A::kScratchSlots * kNmsThreads : 1];
    const long long total = w.cnt[n_max];
    if (total > w.capC || w.ctl[0]) return;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const unsigned long long c = w.cand[e];
        const int src = (int)(unsigned int)c, dst = (int)(c >> 32);
        const double thr = tb.seg_thr[w.seg_of[src]];
        const bool sup = A::sup(boxes[src], boxes[dst], thr, s_pts + (A::kScratchSlots ? threadIdx.x : 0));
        w.flag[e] = sup ? 1 : 0;
        if (sup) atomicAdd(&w.indeg[dst], 1);
    }
}

__global__ void sp_fill_kernel(int n_max, SparseWs w) {
    const long long total = w.cnt[n_max];
    if (total > w.capC || w.ctl[0]) return;
    if ((long long)w.indeg[n_max] > w.capE) { if (blockIdx.x == 0 && threadIdx.x == 0) w.ctl[0] = 1; return; }
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        if (!w.flag[e]) continue;
        const unsigned long long c = w.cand[e];
        const int dst = (int)(c >> 32);
        w.adj[w.indeg[dst] + atomicAdd(&w.cursor[dst], 1)] = (int)(unsigned int)c;
    }
}

__device__ __forceinline__ void sp_grid_barrier(int* ctl, int nblocks) {
    __syncthreads();
    if (threadIdx.x == 0) {
        volatile int* gen = ctl + 2;
        const int g = *gen;
        __threadfence();
        if (atomicAdd(ctl + 1, 1) == nblocks - 1) {
            ctl[1] = 0;
            __threadfence();
            atomicAdd(ctl + 2, 1);
        } else {
            while (*gen == g) { }
        }
        __threadfence();
    }
    __syncthreads();
}

// persistent: kSparseCtas co-resident CTAs, one fixed-point round per grid barrier
__global__ void __launch_bounds__(kSparseThreads, 1)
sp_resolve_kernel(SegTable tb, int n_max, SparseWs w, uint8_t* __restrict__ keep_sorted) {
    if (w.ctl[0] || (long long)w.cnt[n_max] > w.capC || (long long)w.indeg[n_max] > w.capE) {
        if (blockIdx.x == 0 && threadIdx.x == 0) w.ctl[0] = 1;
        return;  // uniform over the grid: every CTA reads the same three words
    }
    const int n_eff = min(tb.hdr[1], n_max);
    const int tid = blockIdx.x * blockDim.x + threadIdx.x, stride = gridDim.x * blockDim.x;
    volatile unsigned char* state = w.state;
    for (int round = 0;; round++) {
        int* changed = w.ctl + 3 + (round & 1);
        bool any = false;
        for (int p = tid; p < n_eff; p += stride) {
            if (state[p]) continue;
            const int lo = w.indeg[p], hi = w.indeg[p + 1];
            bool dead = false, all_dead = true;
            for (int e = lo; e < hi; e++) {
                const unsigned char sv = state[w.adj[e]];
                dead |= sv == 1;
                all_dead &= sv == 2;
            }
            if (dead) { state[p] = 2; any = true; }
            else if (all_dead) { state[p] = 1; any = true; }
        }
        if (any) *changed = 1;
        // states written in this round may or may not be seen by the other threads of the same round: either way a
        // value that is read is final, so the rule stays sound; the barrier publishes them for the next round
        sp_grid_barrier(w.ctl, gridDim.x);
        const int c = *(volatile int*)changed;
        sp_grid_barrier(w.ctl, gridDim.x);   // everybody has read `changed` before it is cleared for round + 2
        if (tid == 0) *changed = 0;
        if (!c) break;
    }
    for (int p = tid; p < n_max; p += stride) keep_sorted[p] = (p < n_eff && state[p] == 1) ? 1 : 0;
}

static size_t box_bytes(int kind) {
    switch (kind) {
        case RSDET_NMS_ROTATED: case RSDET_NMS_ROTATED_GE: return sizeof(RBox);
        case RSDET_NMS_POLY: return sizeof(PolyBox);
        case RSDET_NMS_MERGE: return sizeof(MBox);
        case RSDET_NMS_HBB_P1: return sizeof(HBoxF);
        default: return sizeof(HBox);
    }
}

constexpr int kMaxNmsBoxes = 1 << 18;  // dense n x n/64 mask: 8.6 GB at the limit; the remv vector fits shared memory

// mask_words = 0: worst case (every box in one label group)
size_t nms_ws_bytes(int kind, int n, size_t mask_words) {
    size_t N = (size_t)(n > 0 ? n : 1);
    size_t b = 0;
    b += 2 * ws_bytes<unsigned long long>(N);  // score keys (double buffer)
    b += 4 * ws_bytes<int>(N);                 // idx (pass 1, pass 2 double buffers)
    b += 2 * ws_bytes<uint32_t>(N);            // label keys
    b += align256(box_bytes(kind) * N);
    b += ws_bytes<int32_t>(N);                                         // label_sorted
    b += ws_bytes<int>(64) + ws_bytes<int>(N + 2) + 2 * ws_bytes<long long>(N + 2) + ws_bytes<double>(N + 1);
    b += ws_bytes<unsigned long long>(mask_words ? mask_words : N * ((N + 63) / 64));  // mask (worst case: one group)
    b += 3 * ws_bytes<uint8_t>(N);                                     // keep_sorted, keep_mask tmp, flags
    b += 2 * ws_bytes<int64_t>(N);                                     // vals, scratch index output
    b += ws_bytes<int>(64) + ws_bytes<int>(kFastSegs);                 // scratch count, unordered segment starts
    b += ws_bytes<unsigned long long>(2 * N / 64 + 8) + ws_bytes<int>(2 * N / 64 + 8);  // published keep words + flags
    b += align256(kCubTempBytes + 16 * N);
    return b;
}

template <int KIND>
static void launch_kind(const NmsArgs& a, const int* idx, void* boxes, int32_t* label_sorted, SegTable tb,
                        unsigned long long* mask, cudaStream_t st, bool mask_phase, int* starts_unsorted, const int* gate = nullptr) {
    using Tr = Traits<KIND>;
    if (!mask_phase) {
        prep_sorted_kernel<KIND><<<ceil_div(a.n_max, 256), 256, 0, st>>>((const typename Tr::Raw*)a.dets, a.labels, idx, a.n_max,
                                                                        a.n_dev, (typename Tr::Box*)boxes, label_sorted,
                                                                        tb.hdr, starts_unsorted);
    } else {
        long long T = (a.n_max + 63) / 64;
        long long tiles = T * (T + 1) / 2;
        int grid = (int)(tiles < (long long)kNumSMs * 5 ? tiles : (long long)kNumSMs * 5);  // 5 CTAs/SM fit (39 KB smem, 91 regs)
        mask_tiles_kernel<KIND><<<grid, kNmsThreads, 0, st>>>((const typename Tr::Box*)boxes, tb, mask, gate);
    }
    count_launch();
}

static void dispatch_kind(const NmsArgs& a, const int* idx, void* boxes, int32_t* label_sorted, SegTable tb,
                          unsigned long long* mask, cudaStream_t st, bool mask_phase, int* starts_unsorted, const int* gate = nullptr) {
    switch (a.kind) {
        case RSDET_NMS_ROTATED: launch_kind<RSDET_NMS_ROTATED>(a, idx, boxes, label_sorted, tb, mask, st, mask_phase, starts_unsorted, gate); break;
        case RSDET_NMS_ROTATED_GE: launch_kind<RSDET_NMS_ROTATED_GE>(a, idx, boxes, label_sorted, tb, mask, st, mask_phase, starts_unsorted, gate); break;
        case RSDET_NMS_POLY: launch_kind<RSDET_NMS_POLY>(a, idx, boxes, label_sorted, tb, mask, st, mask_phase, starts_unsorted, gate); break;
        case RSDET_NMS_MERGE: launch_kind<RSDET_NMS_MERGE>(a, idx, boxes, label_sorted, tb, mask, st, mask_phase, starts_unsorted, gate); break;
        case RSDET_NMS_HBB_P1: launch_kind<RSDET_NMS_HBB_P1>(a, idx, boxes, label_sorted, tb, mask, st, mask_phase, starts_unsorted, gate); break;
        case RSDET_NMS_HBB_P1_F64: launch_kind<RSDET_NMS_HBB_P1_F64>(a, idx, boxes, label_sorted, tb, mask, st, mask_phase, starts_unsorted, gate); break;
        default: launch_kind<RSDET_NMS_HBB>(a, idx, boxes, label_sorted, tb, mask, st, mask_phase, starts_unsorted, gate); break;
    }
}

constexpr int kSparseMinRotated = 32768;  // below this the dense tiles + staged scan are faster (tools/sweep.py)

template <int KIND>
static void sp_launch_kind(int step, const void* boxes, SegTable tb, int n, const unsigned long long* key, const int* val,
                           const SparseWs& w, cudaStream_t st) {
    using Box = typename SpAdapt<KIND>::Box;
    const Box* b = (const Box*)boxes;
    switch (step) {
        case 0: sp_extent_kernel<KIND><<<ceil_div(n, 256), 256, 0, st>>>(b, tb, n, w); break;
        case 1: sp_keys_kernel<KIND><<<ceil_div(n + 1, 256), 256, 0, st>>>(b, tb, n, w); break;
        case 5: sp_estimate_kernel<KIND><<<ceil_div(n, 128), 128, 0, st>>>(b, tb, n, key, val, w); break;
        case 2: sp_sweep_kernel<KIND, false><<<ceil_div(n, 128), 128, 0, st>>>(b, tb, n, key, val, w); break;
        case 3: sp_sweep_kernel<KIND, true><<<ceil_div(n, 128), 128, 0, st>>>(b, tb, n, key, val, w); break;
        default: sp_iou_kernel<KIND><<<kNumSMs * 8, kNmsThreads, 0, st>>>(b, tb, n, w); break;
    }
}
static void sp_launch(int kind, int step, const void* boxes, SegTable tb, int n, const unsigned long long* key, const int* val,
                      const SparseWs& w, cudaStream_t st) {
    if (kind == RSDET_NMS_MERGE) sp_launch_kind<RSDET_NMS_MERGE>(step, boxes, tb, n, key, val, w, st);
    else if (kind == RSDET_NMS_ROTATED_GE) sp_launch_kind<RSDET_NMS_ROTATED_GE>(step, boxes, tb, n, key, val, w, st);
    else sp_launch_kind<RSDET_NMS_ROTATED>(step, boxes, tb, n, key, val, w, st);
}

// One directed n x n decision matrix "a suppresses b" for class-agnostic boxes (shared by every class): RBox prep, filter
// cascade into a global pair queue, exact clipper over the queue, flagged-tile fallback.  mask: nb x pitch words followed
// by the tile flags and the pair queue (mask_cap words in total); cnt_scratch[32..33]: queue counters.
static void launch_ov_matrix(const float* shared_boxes, int nb, float thr, bool ge, RBox* sb, unsigned long long* mask, size_t mask_cap,
                             int* cnt_scratch, cudaStream_t st) {
        const int Tov = (nb + 63) / 64;
        const int pitch = (Tov + 1) & ~1;
        prep_shared_kernel<<<ceil_div(nb, 256), 256, 0, st>>>(shared_boxes, nb, sb);
        cudaMemsetAsync(mask, 0, sizeof(unsigned long long) * (size_t)nb * pitch, st);
        long long tiles = (long long)Tov * (Tov + 1) / 2;
        int grid = (int)(tiles < (1ll << 22) ? tiles : (1ll << 22));
        // the part of the mask buffer the n x pitch matrix does not use holds the tile flags and the pair queue
        const size_t used = (size_t)nb * pitch, flag_words = ((size_t)tiles + 7) / 8 + 1;
        const bool split = grid == tiles && mask_cap > used + flag_words + 4096;
        if (split) {
            uint8_t* tile_flags = (uint8_t*)(mask + used);
            int2* pairs = (int2*)(mask + used + flag_words);
            const size_t capz = mask_cap - used - flag_words;
            const unsigned int cap = (unsigned int)(capz < 0x7fffffffull ? capz : 0x7fffffffull);
            unsigned int* pair_count = (unsigned int*)(cnt_scratch + 32);
            cudaMemsetAsync(tile_flags, 0, flag_words * 8, st);
            cudaMemsetAsync(pair_count, 0, 2 * sizeof(int), st);
            // one pair per thread when the survivors fit (CTAs past the count exit at once); fallback: few CTAs scan the flags
            const int cgrid = (int)(tiles < (long long)kNumSMs * 8 ? (long long)kNumSMs * 8 : (tiles < (long long)kNumSMs * 64 ? tiles : (long long)kNumSMs * 64));
            const int fgrid = (int)(tiles < (long long)kNumSMs * 2 ? tiles : (long long)kNumSMs * 2);
            if (ge) {
                ov_filter_kernel<true><<<grid, kNmsThreads, 0, st>>>(sb, nb, thr, pairs, cap, pair_count, tile_flags);
                ov_clip_kernel<true><<<cgrid, kNmsThreads, 0, st>>>(sb, pairs, cap, pair_count, thr, mask, pitch);
                ov_tiles_kernel<true><<<fgrid, kNmsThreads, 0, st>>>(sb, nb, thr, mask, pitch, tile_flags, pair_count + 1);
            } else {
                ov_filter_kernel<false><<<grid, kNmsThreads, 0, st>>>(sb, nb, thr, pairs, cap, pair_count, tile_flags);
                ov_clip_kernel<false><<<cgrid, kNmsThreads, 0, st>>>(sb, pairs, cap, pair_count, thr, mask, pitch);
                ov_tiles_kernel<false><<<fgrid, kNmsThreads, 0, st>>>(sb, nb, thr, mask, pitch, tile_flags, pair_count + 1);
            }
            count_launch(2);
        } else if (ge) {
            ov_tiles_kernel<true><<<grid, kNmsThreads, 0, st>>>(sb, nb, thr, mask, pitch, nullptr, nullptr);
        } else {
            ov_tiles_kernel<false><<<grid, kNmsThreads, 0, st>>>(sb, nb, thr, mask, pitch, nullptr, nullptr);
        }
}

// cudaFuncSetAttribute is per device and the library may drive several GPUs from several host threads: set the
// attribute on every call (it is a cheap driver call) instead of caching it in a process-wide flag
static inline void allow_dyn_smem(const void* func, size_t bytes) {
    cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

int nms_run(const NmsArgs& a, void* workspace, size_t workspace_bytes, cudaStream_t st) {
    const int n = a.n_max;
    if (n < 0 || a.kind < 0 || a.kind > RSDET_NMS_HBB_P1_F64) return RSDET_EINVAL;
    if (n == 0) {
        if (a.num_keep) cudaMemsetAsync(a.num_keep, 0, sizeof(int32_t), st);
        return cuda_status();
    }
    if (!a.dets || !a.scores) return RSDET_EINVAL;
    if (n > (a.mask_words ? (1 << 20) : kMaxNmsBoxes)) return RSDET_ELIMIT;
    if (workspace_bytes < nms_ws_bytes(a.kind, n, a.mask_words)) return RSDET_EWORKSPACE;
    const bool f64 = a.kind == RSDET_NMS_MERGE || a.kind == RSDET_NMS_HBB || a.kind == RSDET_NMS_HBB_P1_F64;
    const size_t N = (size_t)n;

    Workspace ws(workspace, workspace_bytes);
    unsigned long long* keyA = ws.take<unsigned long long>(N);
    unsigned long long* keyB = ws.take<unsigned long long>(N);
    int* idxA = ws.take<int>(N);
    int* idxB = ws.take<int>(N);
    int* idxC = ws.take<int>(N);
    int* idxD = ws.take<int>(N);
    uint32_t* lkA = ws.take<uint32_t>(N);
    uint32_t* lkB = ws.take<uint32_t>(N);
    void* boxes = ws.take<char>(box_bytes(a.kind) * N);
    int32_t* label_sorted = ws.take<int32_t>(N);
    SegTable tb;
    tb.hdr = ws.take<int>(64);
    tb.seg_start = ws.take<int>(N + 2);
    tb.tile_pref = ws.take<long long>(N + 2);
    tb.mask_off = ws.take<long long>(N + 2);
    tb.seg_thr = ws.take<double>(N + 1);
    unsigned long long* mask = ws.take<unsigned long long>(a.mask_words ? a.mask_words : N * ((N + 63) / 64));
    uint8_t* keep_sorted = ws.take<uint8_t>(N);
    uint8_t* keep_tmp = ws.take<uint8_t>(N);
    uint8_t* flags = ws.take<uint8_t>(N);
    int64_t* vals = ws.take<int64_t>(N);
    int64_t* idx_scratch = ws.take<int64_t>(N);
    int* cnt_scratch = ws.take<int>(64);
    int* starts_unsorted = ws.take<int>(kFastSegs);
    unsigned long long* pub_keep = ws.take<unsigned long long>(2 * N / 64 + 8);
    int* pub_flag = ws.take<int>(2 * N / 64 + 8);
    size_t cub_bytes = kCubTempBytes + 16 * N;
    void* cub_tmp = ws.take<char>(cub_bytes);
    if (!ws.ok()) return RSDET_EWORKSPACE;

    // 1. sort by score (descending, stable: lower index first on ties for the fp32 kinds -- Jittor's argsort --,
    //    higher index first for the float64 merge kinds, see make_keys_kernel)
    const int* idx_score;
    if (f64) {
        make_keys_kernel<double, unsigned long long><<<ceil_div(n, 256), 256, 0, st>>>((const double*)a.scores, n, keyA, idxA, true);
        cub::DoubleBuffer<unsigned long long> dk(keyA, keyB);
        cub::DoubleBuffer<int> dv(idxA, idxB);
        size_t need = 0;
        cub::DeviceRadixSort::SortPairs(nullptr, need, dk, dv, n, 0, 64, st);
        if (need > cub_bytes) return RSDET_EWORKSPACE;
        cub::DeviceRadixSort::SortPairs(cub_tmp, need, dk, dv, n, 0, 64, st);
        idx_score = dv.Current();
    } else {
        uint32_t* kA = (uint32_t*)keyA;
        uint32_t* kB = (uint32_t*)keyB;
        make_keys_kernel<float, uint32_t><<<ceil_div(n, 256), 256, 0, st>>>((const float*)a.scores, n, kA, idxA, false);
        cub::DoubleBuffer<uint32_t> dk(kA, kB);
        cub::DoubleBuffer<int> dv(idxA, idxB);
        size_t need = 0;
        cub::DeviceRadixSort::SortPairs(nullptr, need, dk, dv, n, 0, 32, st);
        if (need > cub_bytes) return RSDET_EWORKSPACE;
        cub::DeviceRadixSort::SortPairs(cub_tmp, need, dk, dv, n, 0, 32, st);
        idx_score = dv.Current();
    }
    count_launch(4);
    // 2. stable sort by label -> segments
    const int* idx_ls = idx_score;
    if (a.labels) {
        const int lbits = a.label_bits >= 1 && a.label_bits < 32 ? a.label_bits : 32;
        label_keys_kernel<<<ceil_div(n, 256), 256, 0, st>>>(a.labels, idx_score, n, a.n_dev, lbits, lkA);
        cudaMemcpyAsync(idxC, idx_score, sizeof(int) * N, cudaMemcpyDeviceToDevice, st);
        cub::DoubleBuffer<uint32_t> dk(lkA, lkB);
        cub::DoubleBuffer<int> dv(idxC, idxD);
        size_t need = 0;
        cub::DeviceRadixSort::SortPairs(nullptr, need, dk, dv, n, 0, lbits, st);
        if (need > cub_bytes) return RSDET_EWORKSPACE;
        cub::DeviceRadixSort::SortPairs(cub_tmp, need, dk, dv, n, 0, lbits, st);
        idx_ls = dv.Current();
        count_launch(5);
    }
    // 3. per-box preprocessing in sorted order, segment table
    const bool shared = a.shared_boxes != nullptr;
    if (shared && (a.kind > RSDET_NMS_ROTATED_GE || a.n_shared <= 0 || a.n_shared > n)) return RSDET_EINVAL;
    if (a.class_counts && shared) {
        segments_from_counts_kernel<<<1, 1024, 0, st>>>(a.class_counts, a.num_classes, a.thr, tb);
    } else {
        cudaMemsetAsync(tb.hdr, 0, 64 * sizeof(int), st);
        dispatch_kind(a, idx_ls, shared ? nullptr : boxes, label_sorted, tb, mask, st, false, starts_unsorted);
        segment_table_kernel<<<1, 1024, 0, st>>>(a.labels ? label_sorted : nullptr, n, a.n_dev, a.thr, a.thr_per_label, a.num_thr,
                                                 tb, starts_unsorted);
    }
    count_launch();
    if (shared) {
        // 4'. one directed decision matrix for all classes, 5'. per-class scans through it
        const int nb = a.n_shared, Tov = (nb + 63) / 64;
        const int pitch = (Tov + 1) & ~1;  // even row pitch: 16-byte aligned rows for the staged scan's vector loads
        RBox* sb = (RBox*)boxes;
        const size_t mask_cap = a.mask_words ? a.mask_words : N * ((N + 63) / 64);
        launch_ov_matrix(a.shared_boxes, nb, (float)a.thr, a.kind == RSDET_NMS_ROTATED_GE, sb, mask, mask_cap, cnt_scratch, st);
        allow_dyn_smem((const void*)reduce_ov_kernel, 200 * 1024);
        allow_dyn_smem((const void*)reduce_ov_staged_kernel<1, false>, 200 * 1024);
        allow_dyn_smem((const void*)reduce_ov_staged_kernel<2, false>, 200 * 1024);
        const size_t Ts = (size_t)(Tov | 1);
        const size_t staged = sizeof(unsigned long long) * (5 * Ts + 2 * 64 * Ts) + sizeof(int) * (size_t)nb;
        if (Tov <= 64 && staged <= 200 * 1024)
            reduce_ov_staged_kernel<1, false><<<kNumSMs, kReduceThreads, staged, st>>>(tb, idx_ls, a.cand_per_box, mask, pitch, nb, keep_sorted, nullptr);
        else if (Tov <= 128 && staged <= 200 * 1024)
            reduce_ov_staged_kernel<2, false><<<kNumSMs, kReduceThreads, staged, st>>>(tb, idx_ls, a.cand_per_box, mask, pitch, nb, keep_sorted, nullptr);
        else
            reduce_ov_kernel<<<kNumSMs, kReduceThreads, sizeof(unsigned long long) * (size_t)Tov, st>>>(tb, idx_ls, a.cand_per_box, mask, pitch,
                                                                                                      nb, keep_sorted);
        count_launch(5);
    } else {
    // 4'. large merge calls: sparse path first; the dense kernels below then run only if it raised the gate
    const int* gate = nullptr;
    const size_t mask_cap = a.mask_words ? a.mask_words : N * ((N + 63) / 64);
    const bool sparse_kind = a.kind == RSDET_NMS_MERGE || ((a.kind == RSDET_NMS_ROTATED || a.kind == RSDET_NMS_ROTATED_GE) && !a.labels);
    if (sparse_kind && n >= (a.kind == RSDET_NMS_MERGE ? kSparseMinBoxes : kSparseMinRotated)) {
        Workspace mw(mask, mask_cap * sizeof(unsigned long long));
        SparseWs w;
        w.keyA = mw.take<unsigned long long>(N);
        w.keyB = mw.take<unsigned long long>(N);
        w.valA = mw.take<int>(N);
        w.valB = mw.take<int>(N);
        w.seg_of = mw.take<int>(N);
        w.cnt = mw.take<int>(N + 1);
        w.indeg = mw.take<int>(N + 1);
        w.cursor = mw.take<int>(N);
        w.state = mw.take<unsigned char>(N);
        w.ctl = cnt_scratch + 40;
        const size_t left = mw.used < mw.size ? mw.size - mw.used : 0;
        long long cap = (long long)(left / 14);              // 8 (cand) + 1 (flag) + 4 (adj) bytes per entry, + alignment slack
        if (cap > 128ll * n) cap = 128ll * n;
        if (cap > 0x3fffffffll) cap = 0x3fffffffll;
        if (cap >= 8ll * n) {
            w.capC = cap;
            w.capE = cap;
            w.cand = mw.take<unsigned long long>((size_t)cap);
            w.flag = mw.take<unsigned char>((size_t)cap);
            w.adj = mw.take<int>((size_t)cap);
        }
        if (cap >= 8ll * n && mw.ok()) {
            int nbits = 1;
            while ((1ll << nbits) < (long long)n + 1) nbits++;
            cudaMemsetAsync(w.ctl, 0, 8 * sizeof(int), st);
            sp_launch(a.kind, 0, boxes, tb, n, nullptr, nullptr, w, st);   // extents
            sp_launch(a.kind, 1, boxes, tb, n, nullptr, nullptr, w, st);   // keys
            cub::DoubleBuffer<unsigned long long> dk(w.keyA, w.keyB);
            cub::DoubleBuffer<int> dv(w.valA, w.valB);
            size_t need = 0;
            const int kbits = 32 + kBandBits + nbits < 64 ? 32 + kBandBits + nbits : 64;
            cub::DeviceRadixSort::SortPairs(nullptr, need, dk, dv, n, 0, kbits, st);
            if (need > cub_bytes) return RSDET_EWORKSPACE;
            cub::DeviceRadixSort::SortPairs(cub_tmp, need, dk, dv, n, 0, kbits, st);
            const unsigned long long* key = dk.Current();
            const int* val = dv.Current();
            sp_launch(a.kind, 5, boxes, tb, n, key, val, w, st);           // sparse enough?
            sp_launch(a.kind, 2, boxes, tb, n, key, val, w, st);           // sweep: count
            need = 0;
            cub::DeviceScan::ExclusiveSum(nullptr, need, w.cnt, w.cnt, n + 1, st);
            if (need > cub_bytes) return RSDET_EWORKSPACE;
            cub::DeviceScan::ExclusiveSum(cub_tmp, need, w.cnt, w.cnt, n + 1, st);
            sp_launch(a.kind, 3, boxes, tb, n, key, val, w, st);           // sweep: fill
            sp_launch(a.kind, 4, boxes, tb, n, key, val, w, st);           // predicate on the candidates
            cub::DeviceScan::ExclusiveSum(cub_tmp, need, w.indeg, w.indeg, n + 1, st);
            sp_fill_kernel<<<kNumSMs * 8, 256, 0, st>>>(n, w);
            {   // grid barrier inside: cooperative launch = the driver guarantees the 148 CTAs are co-resident even when
                // several such kernels are in flight on different streams
                int n_arg = n;
                void* args[] = {(void*)&tb, (void*)&n_arg, (void*)&w, (void*)&keep_sorted};
                cudaError_t ce = cudaLaunchCooperativeKernel((const void*)sp_resolve_kernel, dim3(kSparseCtas), dim3(kSparseThreads), args, 0, st);
                if (ce != cudaSuccess) return (int)ce;
            }
            count_launch(16);
            gate = w.ctl;
        }
    }
    // 4. suppression mask over the upper-triangular tiles of every segment
    dispatch_kind(a, idx_ls, boxes, label_sorted, tb, mask, st, true, starts_unsorted, gate);
    // 5. greedy scan
    {
        size_t smem = sizeof(unsigned long long) * ((N + 63) / 64);
        allow_dyn_smem((const void*)reduce_kernel, 200 * 1024);
        allow_dyn_smem((const void*)reduce_ov_staged_kernel<2, true>, 200 * 1024);
        // groups of < kCoopMinBlocks blocks: staged scan (rows through shared memory); larger ones: cooperative phase
        const size_t Tmax = (size_t)(kCoopMinBlocks - 1) | 1;
        reduce_ov_staged_kernel<2, true><<<kNumSMs, kReduceThreads, sizeof(unsigned long long) * (5 * Tmax + 2 * 64 * Tmax), st>>>(
            tb, nullptr, 1, mask, 0, 0, keep_sorted, gate);
        count_launch();
        if ((N + 63) / 64 >= (size_t)kCoopMinBlocks) {
            cudaMemsetAsync(pub_flag, 0, sizeof(int) * (2 * N / 64 + 8), st);
            {   // CTAs of one group wait for each other's published keep words: cooperative launch (co-residency)
                int skip_small = 1;
                const unsigned long long* mask_c = mask;
                void* args[] = {(void*)&tb, (void*)&mask_c, (void*)&keep_sorted, (void*)&pub_keep, (void*)&pub_flag, (void*)&skip_small,
                                (void*)&gate};
                cudaError_t ce = cudaLaunchCooperativeKernel((const void*)reduce_kernel, dim3(kNumSMs), dim3(kReduceThreads), args, smem, st);
                if (ce != cudaSuccess) return (int)ce;
            }
            count_launch();
        }
    }
    }
    // 6. outputs
    uint8_t* km = a.keep_mask ? a.keep_mask : keep_tmp;
    scatter_keep_kernel<<<ceil_div(n, 256), 256, 0, st>>>(keep_sorted, idx_ls, n, a.n_dev, km);
    count_launch();
    bool counted = false;
    if (a.keep_sorted_idx || (a.num_keep && !a.keep_score_idx)) {
        int64_t* out = a.keep_sorted_idx ? a.keep_sorted_idx : idx_scratch;
        int* cnt = a.num_keep ? a.num_keep : cnt_scratch;
        thrust::counting_iterator<int64_t> it(0);
        size_t need = 0;
        cub::DeviceSelect::Flagged(nullptr, need, it, km, out, cnt, n, st);
        if (need > cub_bytes) return RSDET_EWORKSPACE;
        cub::DeviceSelect::Flagged(cub_tmp, need, it, km, out, cnt, n, st);
        counted = true;
        count_launch(2);
    }
    if (a.keep_score_idx) {
        score_order_flags_kernel<<<ceil_div(n, 256), 256, 0, st>>>(km, idx_score, n, flags, vals);
        int* cnt = (a.num_keep && !counted) ? a.num_keep : cnt_scratch;
        size_t need = 0;
        cub::DeviceSelect::Flagged(nullptr, need, vals, flags, a.keep_score_idx, cnt, n, st);
        if (need > cub_bytes) return RSDET_EWORKSPACE;
        cub::DeviceSelect::Flagged(cub_tmp, need, vals, flags, a.keep_score_idx, cnt, n, st);
        count_launch(3);
    }
    return cuda_status();
}

// ----------------------------------------------------------------------------- multiclass_nms_rotated
// nms_rotated.py:562-575: expand (n, C) candidates in row-major order; invalid ones get score -inf and
// label INT_MAX so that both sorts push them behind the *n_valid live rows.
constexpr int kMcHist = 1024;  // classes counted through a shared-memory histogram

__global__ void mc_expand_kernel(const float* __restrict__ bboxes, int bbox_dim, const float* __restrict__ scores, int n, int C,
                                 float score_thr, const float* __restrict__ factors, float* __restrict__ cbox,
                                 float* __restrict__ cscore, int32_t* __restrict__ clabel, int* __restrict__ n_valid,
                                 int* __restrict__ class_counts) {
    __shared__ int s_hist[kMcHist];
    const bool hist = class_counts != nullptr && C <= kMcHist;
    if (hist) {
        for (int i = threadIdx.x; i < C; i += blockDim.x) s_hist[i] = 0;
        __syncthreads();
    }
    int e = blockIdx.x * blockDim.x + threadIdx.x;
    bool in = e < n * C;
    int i = in ? e / C : 0, c = in ? e % C : 0;
    float s = in ? scores[(size_t)i * (C + 1) + c + 1] : 0.f;
    bool valid = in && s > score_thr;
    if (in) {
        const float* b = bbox_dim > 5 ? bboxes + (size_t)i * bbox_dim + (c + 1) * 5 : bboxes + (size_t)i * 5;
#pragma unroll
        for (int k = 0; k < 5; k++) cbox[(size_t)e * 5 + k] = b[k];
        if (factors) s = s * factors[i];
        cscore[e] = valid ? s : -INFINITY;
        clabel[e] = valid ? c : 0x7fffffff;
    }
    unsigned m = __ballot_sync(0xffffffffu, valid);
    if ((threadIdx.x & 31) == 0 && m) atomicAdd(n_valid, __popc(m));
    if (hist) {
        if (valid) atomicAdd(&s_hist[c], 1);
        __syncthreads();
        for (int i = threadIdx.x; i < C; i += blockDim.x)
            if (s_hist[i]) atomicAdd(&class_counts[i], s_hist[i]);
    }
}

// nms_rotated.py:577-596: kept candidates arrive in descending-score order; apply the max_num slice.
__global__ void mc_output_kernel(const int64_t* __restrict__ keep_score_idx, const int32_t* __restrict__ num_keep, int max_num,
                                 const float* __restrict__ cbox, const float* __restrict__ cscore,
                                 const int32_t* __restrict__ clabel, float* __restrict__ out_dets,
                                 int32_t* __restrict__ out_labels, int32_t* __restrict__ out_count, int cap) {
    int nk = *num_keep;
    int cnt = nk;
    if (nk > max_num) cnt = max_num >= 0 ? max_num : max(nk + max_num, 0);  // python inds[:max_num]
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r == 0) *out_count = cnt;
    if (r >= cnt || r >= cap) return;
    int e = (int)keep_score_idx[r];
#pragma unroll
    for (int k = 0; k < 5; k++) out_dets[(size_t)r * 6 + k] = cbox[(size_t)e * 5 + k];
    out_dets[(size_t)r * 6 + 5] = cscore[e];
    out_labels[r] = clabel[e];
}

// iou_poly (nms_poly.py:247-252) for n aligned pairs of float64 quads
__global__ void iou_poly_pairs_kernel(const double* __restrict__ a, const double* __restrict__ b, int n, double* __restrict__ out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    MBox A = Traits<RSDET_NMS_MERGE>::prep(a + (size_t)i * 8);
    MBox B = Traits<RSDET_NMS_MERGE>::prep(b + (size_t)i * 8);
    out[i] = iou_poly_d(A, B);
}

// ----------------------------------------------------------------------------- SURVEY 8(f) rank 3: voc_eval matching
// voc_eval_dota (python/jdet/data/devkits/voc_eval.py:236-318): for every detection (already in descending
// confidence order) the best-overlapping ground truth of ITS image: hbb prefilter with the reference's `+1`
// convention (:262-285), then iou_poly (Shapely in the reference) on the survivors, np.argmax = first maximum.
// One warp per detection, lanes over the image's ground truths.
__global__ void voc_best_gt_kernel(const double* __restrict__ det, const int32_t* __restrict__ det_img, int nd,
                                   const double* __restrict__ gt, const int32_t* __restrict__ gt_start, int num_imgs,
                                   double* __restrict__ ovmax, int32_t* __restrict__ jmax) {
    const int d = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (d >= nd) return;
    const int img = det_img[d];
    double best = -INFINITY;
    int bj = 0x7fffffff;
    if (img >= 0 && img < num_imgs) {
        const MBox D = Traits<RSDET_NMS_MERGE>::prep(det + (size_t)d * 8);
        for (int j = gt_start[img] + lane; j < gt_start[img + 1]; j += 32) {
            const MBox G = Traits<RSDET_NMS_MERGE>::prep(gt + (size_t)j * 8);
            const double iw = fmax(fmin(G.x2, D.x2) - fmax(G.x1, D.x1) + 1., 0.);
            const double ih = fmax(fmin(G.y2, D.y2) - fmax(G.y1, D.y1) + 1., 0.);
            const double inters = iw * ih;
            const double uni = (D.x2 - D.x1 + 1.) * (D.y2 - D.y1 + 1.) + (G.x2 - G.x1 + 1.) * (G.y2 - G.y1 + 1.) - inters;
            if (inters / uni > 0) {
                const double ov = iou_poly_d(G, D);  // iou_func(BBGT_keep[index], bb)
                if (ov > best) { best = ov; bj = j; }
            }
        }
    }
    for (int o = 16; o; o >>= 1) {
        const double ob = __shfl_xor_sync(0xffffffffu, best, o);
        const int oj = __shfl_xor_sync(0xffffffffu, bj, o);
        if (ob > best || (ob == best && oj < bj)) { best = ob; bj = oj; }
    }
    if (lane == 0) { ovmax[d] = best; jmax[d] = bj == 0x7fffffff ? -1 : bj; }
}

// the sequential TP/FP marking (:303-311) without the sequence: a ground truth is claimed by the FIRST
// (highest-confidence) detection that matches it
__global__ void voc_claim_kernel(const double* __restrict__ ovmax, const int32_t* __restrict__ jmax, const uint8_t* __restrict__ difficult,
                                 int nd, double thr, int32_t* __restrict__ claim) {
    const int d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= nd) return;
    const int j = jmax[d];
    if (j >= 0 && ovmax[d] > thr && !difficult[j]) atomicMin(&claim[j], d);
}

__global__ void voc_mark_kernel(const double* __restrict__ ovmax, const int32_t* __restrict__ jmax, const uint8_t* __restrict__ difficult,
                                int nd, double thr, const int32_t* __restrict__ claim, uint8_t* __restrict__ tp, uint8_t* __restrict__ fp) {
    const int d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= nd) return;
    const int j = jmax[d];
    uint8_t t = 0, f = 0;
    if (j >= 0 && ovmax[d] > thr) {
        if (!difficult[j]) { if (claim[j] == d) t = 1; else f = 1; }
    } else f = 1;
    tp[d] = t;
    fp[d] = f;
}

__global__ void fill_i32_kernel(int32_t* p, int n, int32_t v) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

}  // namespace rsdet

using namespace rsdet;

extern "C" int rsdet_iou_poly_pairs(const double* polys1, const double* polys2, int n, double* ious, void* stream) {
    if (n < 0) return RSDET_EINVAL;
    if (n == 0) return RSDET_OK;
    if (!polys1 || !polys2 || !ious) return RSDET_EINVAL;
    iou_poly_pairs_kernel<<<ceil_div(n, 128), 128, 0, (cudaStream_t)stream>>>(polys1, polys2, n, ious);
    count_launch();
    return cuda_status();
}

extern "C" int rsdet_voc_match(const double* det_polys, const int32_t* det_img, int nd, const double* gt_polys,
                               const int32_t* gt_start, const uint8_t* gt_difficult, int num_imgs, int num_gts, double ovthresh,
                               double* ovmax, int32_t* jmax, int32_t* claim, uint8_t* tp, uint8_t* fp, void* stream) {
    if (nd < 0 || num_imgs < 0 || num_gts < 0) return RSDET_EINVAL;
    if (nd == 0) return RSDET_OK;
    if (!det_polys || !det_img || !gt_start || !ovmax || !jmax || !claim || !tp || !fp) return RSDET_EINVAL;
    if (num_gts > 0 && (!gt_polys || !gt_difficult)) return RSDET_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    voc_best_gt_kernel<<<ceil_div(nd, 8), 256, 0, st>>>(det_polys, det_img, nd, gt_polys, gt_start, num_imgs, ovmax, jmax);
    if (num_gts > 0) fill_i32_kernel<<<ceil_div(num_gts, 256), 256, 0, st>>>(claim, num_gts, 0x7fffffff);
    voc_claim_kernel<<<ceil_div(nd, 256), 256, 0, st>>>(ovmax, jmax, gt_difficult, nd, ovthresh, claim);
    voc_mark_kernel<<<ceil_div(nd, 256), 256, 0, st>>>(ovmax, jmax, gt_difficult, nd, ovthresh, claim, tp, fp);
    count_launch(4);
    return cuda_status();
}

extern "C" size_t rsdet_nms_workspace_bytes(int kind, int n) { return n > kMaxNmsBoxes ? 0 : nms_ws_bytes(kind, n); }

extern "C" int rsdet_nms(int kind, const void* dets, const void* scores, const int32_t* labels, int n, double thr,
                         const double* thr_per_label, int num_thr, uint8_t* keep_mask, int64_t* keep_sorted_idx,
                         int64_t* keep_score_idx, int32_t* num_keep, void* workspace, size_t workspace_bytes, void* stream) {
    NmsArgs a{kind, dets, scores, labels, n, nullptr, thr, thr_per_label, num_thr, keep_mask, keep_sorted_idx, keep_score_idx, num_keep};
    return nms_run(a, workspace, workspace_bytes, (cudaStream_t)stream);
}

// every class holds at most n candidates -> the block-sparse mask needs at most C * n * ceil(n/64) words
// ----------------------------------------------------------------------------- multiclass_nms_rotated, fast path
// Class-agnostic boxes, n <= 8192 (every Oriented R-CNN test config): the generic engine's front end -- expand to n x C
// candidates, two device-wide radix sorts (score, then label) over all of them, a segment table -- and its back end --
// scatter to a keep mask, two stream compactions, the output gather -- were 20 launches of mostly latency (78 us of
// library sort / select kernels per tile in the round-1 launch list).  Here:
//   mc_class_sort_kernel   one CTA per class: the class's valid candidates as 64-bit keys (descending score, then
//                          candidate index) sorted in shared memory (bitonic, <= 8192 keys), written as a fixed-stride
//                          segment (class c at c*n) -> no expand, no device-wide sort, no segment kernel;
//   launch_ov_matrix       the shared decision matrix (unchanged);
//   reduce_ov_staged_kernel  the per-class scan (unchanged) also emits the exclusive prefix of its keep flags;
//   mc_fast_output_kernel  rank of a kept candidate in the global score order = sum over classes of the kept candidates
//                          with a smaller key (one binary search per class, lanes = classes) -> written straight to its
//                          output row; no keep mask, no compaction.
// Same keys, same tie rule (lower candidate index first), same decisions: results are identical to the generic engine's.
constexpr int kMcFastMaxBoxes = 8192;
constexpr int kPipeThreads = 512;   // measured: 256 -> 0.181, 512 -> 0.169, 1024 -> 0.175 ms per 4000x10 call
constexpr int kMcFastMaxClasses = 4096;

__global__ void __launch_bounds__(1024)
mc_class_sort_kernel(const float* __restrict__ scores, const float* __restrict__ factors, int n, int C, float score_thr,
                     unsigned long long* __restrict__ skey, int* __restrict__ idx_ls, int* __restrict__ seg_count, SegTable tb) {
    // keys (descending-score bits) and box indices live in two shared arrays (6 bytes per candidate instead of one 64-bit
    // word: the bitonic network is bound by shared-memory bandwidth); n <= 8192 -> 32 KB + 16 KB
    extern __shared__ unsigned int s_k32[];          // [Pmax] keys, then [Pmax] unsigned short box indices
    __shared__ int s_warp_cnt[32], s_base;
    const int c = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int Pmax = 64;
    while (Pmax < n) Pmax <<= 1;
    unsigned short* s_i16 = reinterpret_cast<unsigned short*>(s_k32 + Pmax);
    if (tid == 0) s_base = 0;
    __syncthreads();
    // valid candidates of this class, compacted in index order (ballot ranks; rounds of 1024 boxes)
    for (int i0 = 0; i0 < n; i0 += 1024) {
        const int i = i0 + tid;
        bool valid = false;
        float sc = 0.f;
        if (i < n) {
            sc = scores[(size_t)i * (C + 1) + c + 1];
            valid = sc > score_thr;                  // nms_rotated.py:562-570: the threshold sees the raw score
            if (valid && factors) sc = sc * factors[i];
        }
        const unsigned m = __ballot_sync(0xffffffffu, valid);
        if (lane == 0) s_warp_cnt[warp] = __popc(m);
        __syncthreads();
        int before = s_base;                         // candidates of earlier rounds
        for (int w = 0; w < warp; w++) before += s_warp_cnt[w];
        if (valid) {
            const int pos = before + __popc(m & ((1u << lane) - 1u));
            s_k32[pos] = desc_key(sc);
            s_i16[pos] = (unsigned short)i;
        }
        __syncthreads();
        if (tid == 0) {
            int t = 0;
            for (int w = 0; w < 32; w++) t += s_warp_cnt[w];
            s_base += t;
        }
        __syncthreads();
    }
    const int cnt = s_base;
    int P = 2;
    while (P < cnt) P <<= 1;                         // the network covers the valid candidates only
    for (int q = cnt + tid; q < P; q += 1024) { s_k32[q] = 0xffffffffu; s_i16[q] = 0xffffu; }   // padding sorts last
    __syncthreads();
    // bitonic network.  A warp owns a chunk of P/32 (>= 64) consecutive elements: steps whose partner distance j stays
    // inside the chunk need only a warp barrier (58 of the 78 steps of a 4096-key sort); steps that cross chunks are
    // framed by block barriers.
    const int chunk = P >= 2048 ? P >> 5 : 64, pairs = chunk >> 1, active_warps = P >= 64 ? P / chunk : 1;
    auto exchange = [&](int t, int j, int k) {
        const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1)), l = i | j;
        const unsigned int ka = s_k32[i], kb = s_k32[l];
        const unsigned short ia = s_i16[i], ib = s_i16[l];
        const bool gt = ka > kb || (ka == kb && ia > ib);   // equal scores: lower box index first
        if (gt == ((i & k) == 0)) { s_k32[i] = kb; s_k32[l] = ka; s_i16[i] = ib; s_i16[l] = ia; }
    };
    for (int k = 2; k <= P; k <<= 1) {
        int j = k >> 1;
        if (j >= chunk) {
            __syncthreads();                                 // the previous phase ended with warp-local steps
            for (; j >= chunk; j >>= 1) {
                for (int t = tid; t < (P >> 1); t += 1024) exchange(t, j, k);
                __syncthreads();
            }
        }
        if (warp < active_warps)
            for (; j > 0; j >>= 1) {
                for (int u = lane; u < pairs && warp * pairs + u < (P >> 1); u += 32) exchange(warp * pairs + u, j, k);
                __syncwarp();
            }
    }
    __syncthreads();
    for (int q = tid; q < cnt; q += 1024) {
        const unsigned e = (unsigned)s_i16[q] * (unsigned)C + (unsigned)c;       // candidate index in the n x C expansion
        skey[(size_t)c * n + q] = ((unsigned long long)s_k32[q] << 32) | e;
        idx_ls[(size_t)c * n + q] = (int)e;
    }
    if (tid == 0) {
        seg_count[c] = cnt;
        tb.seg_start[c] = c * n;
        if (c == 0) tb.hdr[0] = C;
        if (c == C - 1) tb.seg_start[C] = C * n;
    }
}

// one warp per kept candidate (class cs, r-th kept): lanes = classes, each does one binary search
__global__ void __launch_bounds__(256)
mc_fast_output_kernel(const float* __restrict__ bboxes, const float* __restrict__ scores, const float* __restrict__ factors, int n, int C,
                      const unsigned long long* __restrict__ skey, const int* __restrict__ seg_count, const int* __restrict__ kept_pos,
                      const int* __restrict__ keep_prefix, const int* __restrict__ kept_count, int max_num,
                      float* __restrict__ out_dets, int32_t* __restrict__ out_labels, int32_t* __restrict__ out_count) {
    const int lane = threadIdx.x & 31;
    const int cs = blockIdx.y, r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (r >= kept_count[cs] && !(r == 0 && cs == 0)) return;
    int nk = 0;
    for (int c2 = lane; c2 < C; c2 += 32) nk += kept_count[c2];
    for (int o = 16; o > 0; o >>= 1) nk += __shfl_xor_sync(0xffffffffu, nk, o);
    int cnt = nk;
    if (nk > max_num) cnt = max_num >= 0 ? max_num : max(nk + max_num, 0);   // python inds[:max_num]
    if (r == 0 && cs == 0 && lane == 0) *out_count = cnt;
    if (r >= kept_count[cs]) return;
    const int qs = kept_pos[(size_t)cs * n + r];
    const unsigned long long key = skey[(size_t)cs * n + qs];
    int rank = 0;
    for (int c2 = lane; c2 < C; c2 += 32) {
        if (c2 == cs) { rank += r; continue; }
        const unsigned long long* kk = skey + (size_t)c2 * n;
        const int len = seg_count[c2];
        int lo = 0, hi = len;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (kk[mid] < key) lo = mid + 1; else hi = mid;
        }
        rank += lo < len ? keep_prefix[(size_t)c2 * n + lo] : kept_count[c2];
    }
    for (int o = 16; o > 0; o >>= 1) rank += __shfl_xor_sync(0xffffffffu, rank, o);
    if (rank < cnt && lane < 7) {
        const int e = (int)(unsigned)(key & 0xffffffffull), i = e / C;
        if (lane < 5) out_dets[(size_t)rank * 6 + lane] = bboxes[(size_t)i * 5 + lane];
        else if (lane == 5) {
            float sc = scores[(size_t)i * (C + 1) + cs + 1];
            if (factors) sc = sc * factors[i];
            out_dets[(size_t)rank * 6 + 5] = sc;
        } else out_labels[rank] = cs;
    }
}

// The class sort (C CTAs) and the decision matrix (thousands of CTAs) are independent until the scan: the sort runs on a
// side stream forked from the caller's stream and joined before the scan (events only -- also valid while the caller's
// stream is being captured into a CUDA graph: the side stream joins the capture at the fork and leaves it at the join).
// One lane per (device, caller stream); calls on one stream are issued by one host thread at a time, lanes are created
// under a mutex.
struct SideLane { cudaStream_t side; cudaEvent_t fork, join; };
static SideLane* side_lane(cudaStream_t user) {
    struct Key { int dev; cudaStream_t st; SideLane lane; };
    static std::vector<Key>* lanes = new std::vector<Key>();
    static std::mutex mu;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
    std::lock_guard<std::mutex> lk(mu);
    for (auto& k : *lanes)
        if (k.dev == dev && k.st == user) return &k.lane;
    if (lanes->size() >= 256) return nullptr;            // callers that churn through streams fall back to one stream
    if (lanes->capacity() < 256) lanes->reserve(256);   // pointers into the vector stay valid
    Key k;
    k.dev = dev; k.st = user;
    if (cudaStreamCreateWithFlags(&k.lane.side, cudaStreamNonBlocking) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    if (cudaEventCreateWithFlags(&k.lane.fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&k.lane.join, cudaEventDisableTiming) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    lanes->push_back(k);
    return &lanes->back().lane;
}

static bool mc_fast_ok(int bbox_dim, int n, int C) {
    return bbox_dim == 5 && n >= 1 && n <= kMcFastMaxBoxes && C <= kMcFastMaxClasses;
}
static size_t mc_mask_words(int n, int num_classes);

static int mc_fast_run(const float* bboxes, const float* scores, int n, int C, float score_thr, float iou_thr, int max_num,
                       const float* factors, float* out_dets, int32_t* out_labels, int32_t* out_count, void* workspace,
                       size_t workspace_bytes, cudaStream_t st) {
    const size_t cap = (size_t)n * C;
    Workspace ws(workspace, workspace_bytes);
    unsigned long long* skey = ws.take<unsigned long long>(cap);
    int* idx_ls = ws.take<int>(cap);
    uint8_t* keep_sorted = ws.take<uint8_t>(cap);
    int* keep_prefix = ws.take<int>(cap);
    int* kept_pos = ws.take<int>(cap);
    int* seg_count = ws.take<int>(C);
    int* kept_count = ws.take<int>(C);
    int* cnt_scratch = ws.take<int>(64);
    SegTable tb;
    tb.hdr = ws.take<int>(64);
    tb.seg_start = ws.take<int>((size_t)C + 2);
    tb.tile_pref = nullptr; tb.mask_off = nullptr; tb.seg_thr = nullptr;
    RBox* sb = ws.take<RBox>(n);
    const size_t mask_cap = mc_mask_words(n, C);
    unsigned long long* mask = ws.take<unsigned long long>(mask_cap);
    if (!ws.ok()) return RSDET_EWORKSPACE;
    int P = 64;
    while (P < n) P <<= 1;
    const size_t sort_smem = (sizeof(unsigned int) + sizeof(unsigned short)) * (size_t)P;
    allow_dyn_smem((const void*)mc_class_sort_kernel, sort_smem);
    SideLane* sl = side_lane(st);
    if (sl && cudaEventRecord(sl->fork, st) == cudaSuccess && cudaStreamWaitEvent(sl->side, sl->fork, 0) == cudaSuccess) {
        mc_class_sort_kernel<<<C, 1024, sort_smem, sl->side>>>(scores, factors, n, C, score_thr, skey, idx_ls, seg_count, tb);
        cudaEventRecord(sl->join, sl->side);
    } else {
        cudaGetLastError();
        sl = nullptr;
        mc_class_sort_kernel<<<C, 1024, sort_smem, st>>>(scores, factors, n, C, score_thr, skey, idx_ls, seg_count, tb);
    }
    const int Tov = (n + 63) / 64, pitch = (Tov + 1) & ~1;
    launch_ov_matrix(bboxes, n, iou_thr, false, sb, mask, mask_cap, cnt_scratch, st);
    if (sl) cudaStreamWaitEvent(st, sl->join, 0);
    const size_t Ts = (size_t)(Tov | 1);
    const size_t piped = sizeof(unsigned long long) * (Ts + 3 * 64 * Ts) + sizeof(int) * (size_t)n;       // three row buffers
    const size_t staged = sizeof(unsigned long long) * (5 * Ts + 2 * 64 * Ts) + sizeof(int) * (size_t)n;  // two (n close to 8192)
    const int grid = C < kNumSMs ? C : kNumSMs;
    if (piped + 2048 <= 227 * 1024) {
        if (Tov <= 64) {
            allow_dyn_smem((const void*)reduce_ov_pipe_kernel<1, kPipeThreads>, piped);
            reduce_ov_pipe_kernel<1, kPipeThreads><<<grid, kPipeThreads, piped, st>>>(tb, idx_ls, C, mask, pitch, n, keep_sorted, seg_count, keep_prefix,
                                                                         kept_count, kept_pos);
        } else {
            allow_dyn_smem((const void*)reduce_ov_pipe_kernel<2, kPipeThreads>, piped);
            reduce_ov_pipe_kernel<2, kPipeThreads><<<grid, kPipeThreads, piped, st>>>(tb, idx_ls, C, mask, pitch, n, keep_sorted, seg_count, keep_prefix,
                                                                         kept_count, kept_pos);
        }
    } else {
        allow_dyn_smem((const void*)reduce_ov_staged_kernel<2, false>, 200 * 1024);
        reduce_ov_staged_kernel<2, false><<<grid, kReduceThreads, staged, st>>>(tb, idx_ls, C, mask, pitch, n, keep_sorted, nullptr, seg_count,
                                                                              keep_prefix, kept_count, kept_pos);
    }
    mc_fast_output_kernel<<<dim3((unsigned)((n + 7) / 8), (unsigned)C), 256, 0, st>>>(bboxes, scores, factors, n, C, skey, seg_count, kept_pos,
                                                                                     keep_prefix, kept_count, max_num, out_dets, out_labels,
                                                                                     out_count);
    count_launch(8);
    return cuda_status();
}

static size_t mc_mask_words(int n, int num_classes) {
    size_t N = (size_t)(n > 0 ? n : 1);
    return (size_t)(num_classes > 0 ? num_classes : 1) * N * ((N + 63) / 64 + 1);  // + 1: the shared matrix uses an even row pitch
}

extern "C" size_t rsdet_multiclass_nms_rotated_workspace_bytes(int n, int num_classes) {
    size_t cap = (size_t)(n > 0 ? n : 1) * (size_t)(num_classes > 0 ? num_classes : 1);
    if (cap > (1u << 20) || n > kMaxNmsBoxes) return 0;  // the call itself answers RSDET_ELIMIT
    return ws_bytes<float>(cap * 5) + ws_bytes<float>(cap) + ws_bytes<int32_t>(cap) + ws_bytes<int>(64) +
           ws_bytes<int64_t>(cap) + ws_bytes<int32_t>(64) + ws_bytes<int>(kMcHist) +
           nms_ws_bytes(RSDET_NMS_ROTATED, (int)cap, mc_mask_words(n, num_classes));
}

extern "C" int rsdet_multiclass_nms_rotated(const float* multi_bboxes, int bbox_dim, const float* multi_scores, int n,
                                            int num_classes, float score_thr, float iou_thr, int max_num,
                                            const float* score_factors, float* out_dets, int32_t* out_labels,
                                            int32_t* out_count, void* workspace, size_t workspace_bytes, void* stream) {
    if (n < 0 || num_classes <= 0 || !out_count) return RSDET_EINVAL;
    if (bbox_dim != 5 && bbox_dim != 5 * (num_classes + 1)) return RSDET_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    if (n == 0) {
        cudaMemsetAsync(out_count, 0, sizeof(int32_t), st);
        return cuda_status();
    }
    if (!multi_bboxes || !multi_scores || !out_dets || !out_labels) return RSDET_EINVAL;
    long long capll = (long long)n * num_classes;
    if (capll > (1 << 20) || n > kMaxNmsBoxes) return RSDET_ELIMIT;
    int cap = (int)capll;
    if (workspace_bytes < rsdet_multiclass_nms_rotated_workspace_bytes(n, num_classes)) return RSDET_EWORKSPACE;
    if (mc_fast_ok(bbox_dim, n, num_classes))
        return mc_fast_run(multi_bboxes, multi_scores, n, num_classes, score_thr, iou_thr, max_num, score_factors, out_dets, out_labels,
                           out_count, workspace, workspace_bytes, st);
    Workspace ws(workspace, workspace_bytes);
    float* cbox = ws.take<float>((size_t)cap * 5);
    float* cscore = ws.take<float>(cap);
    int32_t* clabel = ws.take<int32_t>(cap);
    int* n_valid = ws.take<int>(64);
    int64_t* kidx = ws.take<int64_t>(cap);
    int32_t* nkeep = ws.take<int32_t>(64);
    int* class_counts = ws.take<int>(kMcHist);
    void* sub = ws.base + ws.used;
    size_t sub_bytes = workspace_bytes - ws.used;
    const bool use_counts = bbox_dim == 5 && num_classes <= kMcHist;
    cudaMemsetAsync(n_valid, 0, sizeof(int), st);
    if (use_counts) cudaMemsetAsync(class_counts, 0, sizeof(int) * num_classes, st);
    mc_expand_kernel<<<ceil_div(cap, 256), 256, 0, st>>>(multi_bboxes, bbox_dim, multi_scores, n, num_classes, score_thr,
                                                        score_factors, cbox, cscore, clabel, n_valid,
                                                        use_counts ? class_counts : nullptr);
    count_launch();
    NmsArgs a{RSDET_NMS_ROTATED, cbox, cscore, clabel, cap, n_valid, (double)iou_thr, nullptr, 0, nullptr, nullptr, kidx, nkeep};
    a.mask_words = mc_mask_words(n, num_classes);
    a.label_bits = 1;
    while ((1 << a.label_bits) - 1 < num_classes) a.label_bits++;  // classes 0..C-1, dead rows -> all ones
    if (bbox_dim == 5) {  // class-agnostic boxes: pairwise decisions are shared by all classes
        a.shared_boxes = multi_bboxes;
        a.n_shared = n;
        a.cand_per_box = num_classes;
        if (use_counts) { a.class_counts = class_counts; a.num_classes = num_classes; }
    }
    int rc = nms_run(a, sub, sub_bytes, st);
    if (rc != RSDET_OK) return rc;
    mc_output_kernel<<<ceil_div(cap, 256), 256, 0, st>>>(kidx, nkeep, max_num, cbox, cscore, clabel, out_dets, out_labels,
                                                        out_count, cap);
    count_launch();
    return cuda_status();
}
