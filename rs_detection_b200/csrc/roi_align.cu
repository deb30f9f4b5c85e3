// roi_align.cu -- multi-level RoIAlignRotated forward / backward for sm_100a.
//
// Replaces ROIAlignRotatedForward / ROIAlignBackward (python/jdet/ops/roi_align_rotated_v1.py:71-147,
// 193-298; v0: roi_align_rotated.py:60-126, 164-254) AND the Python level loop around them
// (python/jdet/models/roi_extractors/oriented_single_level.py:91-114): RoI extension, level mapping,
// four per-level launches, boolean gathers and masked scatter-adds become ONE launch.
//
// The op is a gather (fwd) / scatter (bwd): ~0.6 FLOP per byte, HBM/L2 bound.  Plan:
//   * features are read channels-last (NHWC): one bilinear tap = one contiguous C*4-byte row, read as
//     coalesced 16-byte vectors (a warp covers 512 contiguous bytes).  NCHW inputs (Jittor's layout)
//     are transposed once per call by a tiled transpose into the workspace; callers that keep a
//     channels-last pyramid skip it (RSDET_ROI_NHWC_MAPS in cfg.channels_last).
//   * one CTA per RoI.  Phase A: the RoI's sampling grid (pooled_h*pooled_w*grid^2 samples -> 4 tap
//     offsets + 4 weights each) is computed ONCE by the first threads and staged in shared memory; the
//     reference recomputes it, sin/cos included, in every one of its K*C*49 threads.
//   * Phase B: thread = (channel quad, bin group); 16 independent 16-byte loads in flight per bin.
//   * the (C,7,7) output block of a RoI is contiguous in the reference layout; results are staged in
//     shared memory in a [k][bin][quad+1] layout (conflict-free both ways) and written with streaming
//     16-byte stores, so the 50 KB block leaves the SM fully coalesced and does not evict features
//     from L2.
//   * backward: same tap table; gradients are accumulated channels-last with 16-byte vector
//     reductions (red.global.add.v4.f32: one L2 atomic op per 4 channels instead of the reference's 4
//     scalar atomicAdd), then transposed back to NCHW, which also produces the dense zero-filled
//     output the reference gets from cudaMemsetAsync.
//
// Sample coordinates are computed with explicitly un-contracted IEEE operations in the reference's
// order: the validity test `y < -1 || y > H` is discontinuous, so coordinates must not drift.
//
// Element types (include/rsdet.h): feature maps, grad_out and gradient maps may be fp16 or bf16 as well as fp32.  Every
// kernel below is templated on them; a half value is converted exactly to fp32 where it is read, the arithmetic is the
// fp32 arithmetic unchanged, and a half result is rounded once, to nearest-even, where it is stored.  Four consecutive
// channels are the unit of every vector access: a float4 (16 bytes) or four 2-byte values (8 bytes).
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <mutex>
#include <type_traits>

#include "common.cuh"

namespace rsdet {

constexpr int kRoiThreads = 256;
constexpr int kMaxSamples = 1024;  // fast path: pooled_h*pooled_w*grid_h*grid_w

// ---------------------------------------------------------------------------------- element types
template <typename T> struct Quad { using V = float4; };            // four channels as one vector
template <> struct Quad<__half> { using V = uint2; };
template <> struct Quad<__nv_bfloat16> { using V = uint2; };
template <typename T> constexpr bool kIsF32 = std::is_same<T, float>::value;

__device__ __forceinline__ float to_f32(float v) { return v; }
__device__ __forceinline__ float to_f32(__half v) { return __half2float(v); }
__device__ __forceinline__ float to_f32(__nv_bfloat16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T from_f32(float v) {
    if constexpr (std::is_same<T, __half>::value) return __float2half_rn(v);
    else if constexpr (std::is_same<T, __nv_bfloat16>::value) return __float2bfloat16_rn(v);
    else return v;
}
template <typename T> __device__ __forceinline__ float4 unpack4(uint2 u) {   // four 2-byte values -> fp32, exact
    if constexpr (std::is_same<T, __half>::value) {
        const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&u.x));
        const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
        return make_float4(a.x, a.y, b.x, b.y);
    } else {
        return make_float4(__uint_as_float(u.x << 16), __uint_as_float(u.x & 0xffff0000u),
                           __uint_as_float(u.y << 16), __uint_as_float(u.y & 0xffff0000u));
    }
}
template <typename T> __device__ __forceinline__ uint2 pack4(float4 v) {     // fp32 -> four 2-byte values, nearest-even
    uint2 u;
    if constexpr (std::is_same<T, __half>::value) {
        const __half2 a = __floats2half2_rn(v.x, v.y), b = __floats2half2_rn(v.z, v.w);
        u.x = *reinterpret_cast<const unsigned*>(&a); u.y = *reinterpret_cast<const unsigned*>(&b);
    } else {
        const __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
        u.x = *reinterpret_cast<const unsigned*>(&a); u.y = *reinterpret_cast<const unsigned*>(&b);
    }
    return u;
}
// read-only 4-channel load / 4-channel store (p aligned to 4 * sizeof(T))
template <typename T> __device__ __forceinline__ float4 ldg4_ro(const T* p) {
    if constexpr (kIsF32<T>) return __ldg(reinterpret_cast<const float4*>(p));
    else return unpack4<T>(__ldg(reinterpret_cast<const uint2*>(p)));
}
template <typename T> __device__ __forceinline__ void st4(T* p, float4 v) {
    if constexpr (kIsF32<T>) *reinterpret_cast<float4*>(p) = v;
    else *reinterpret_cast<uint2*>(p) = pack4<T>(v);
}

struct LevelSet {
    const float* feat[RSDET_MAX_LEVELS];  // channels-last maps; their element type is the kernel's T (feat_base)
    float* grad[RSDET_MAX_LEVELS];
    int H[RSDET_MAX_LEVELS], W[RSDET_MAX_LEVELS];
    float scale[RSDET_MAX_LEVELS];
    int num_levels, batch, C;
    int PH, PW, sampling_ratio, version;
    float extend_w, extend_h, finest_scale;
};
template <typename T> __device__ __forceinline__ const T* feat_base(const LevelSet& L, int level) {
    return reinterpret_cast<const T*>(L.feat[level]);
}

// ---------------------------------------------------------------------------------- transposes
// (N, C, HW) <-> (N, HW, C), 64x64 tiles through padded shared memory; source elements S, destination elements D
// (fp32 tile: a half source converts exactly, a half destination rounds to nearest-even).
struct TransposeJob {
    const void* src[RSDET_MAX_LEVELS];
    void* dst[RSDET_MAX_LEVELS];
    int HW[RSDET_MAX_LEVELS];
    int tile_begin[RSDET_MAX_LEVELS + 1];  // prefix of tiles over levels
    int num_levels, N, C;
};

// 64(channels) x 64(pixels) tiles, 4-channel vector accesses on both sides (16 bytes for fp32, 8 for half): a thread
// reads four elements along the source's contiguous dimension, scatters them into a padded shared tile, and writes four
// along the destination's contiguous dimension.  Falls back to scalar accesses at ragged edges / unaligned bases.
template <typename S, typename D, bool TO_NHWC>
__device__ __forceinline__ void transpose_tile(const TransposeJob& job, int t, float (*tile)[65]) {
    int l = 0;
    while (l + 1 < job.num_levels && t >= job.tile_begin[l + 1]) l++;
    t -= job.tile_begin[l];
    const int HW = job.HW[l], C = job.C;
    const int tiles_hw = ceil_div(HW, 64), tiles_c = ceil_div(C, 64);
    const int n = t / (tiles_hw * tiles_c);
    const int r = t % (tiles_hw * tiles_c);
    const int hw0 = (r % tiles_hw) * 64, c0 = (r / tiles_hw) * 64;
    const S* src = static_cast<const S*>(job.src[l]) + (size_t)n * C * HW;
    D* dst = static_cast<D*>(job.dst[l]) + (size_t)n * C * HW;
    const int tid = threadIdx.x;
    // source: rows of `SR` index, contiguous along `SC`; destination the other way round
    const int srcRows = TO_NHWC ? C : HW, srcCols = TO_NHWC ? HW : C;      // src[row * srcCols + col]
    const int r0 = TO_NHWC ? c0 : hw0, q0 = TO_NHWC ? hw0 : c0;            // tile origin (row, col) in the source
    const bool vec_in = (srcCols & 3) == 0 && ((size_t)src & (4 * sizeof(S) - 1)) == 0;
    const bool vec_out = (srcRows & 3) == 0 && ((size_t)dst & (4 * sizeof(D) - 1)) == 0;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int idx = tid + 256 * k;            // 1024 4-element slots: 64 rows x 16 slots
        const int rr = idx >> 4, cc = (idx & 15) * 4;
        const int gr = r0 + rr, gc = q0 + cc;
        if (gr < srcRows) {
            if (vec_in && gc + 3 < srcCols) {
                const float4 v = ldg4_ro(src + (size_t)gr * srcCols + gc);
                tile[rr][cc] = v.x; tile[rr][cc + 1] = v.y; tile[rr][cc + 2] = v.z; tile[rr][cc + 3] = v.w;
            } else {
                for (int e = 0; e < 4; e++)
                    if (gc + e < srcCols) tile[rr][cc + e] = to_f32(__ldg(src + (size_t)gr * srcCols + gc + e));
            }
        }
    }
    __syncthreads();
    // destination: dst[col * srcRows + row]; a float4 covers 4 consecutive source rows of one source column
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int idx = tid + 256 * k;
        const int cc = idx >> 4, rr = (idx & 15) * 4;  // cc = source column (dest row), rr = first of 4 source rows
        const int gc = q0 + cc, gr = r0 + rr;
        if (gc < srcCols) {
            if (vec_out && gr + 3 < srcRows) {
                const float4 v = make_float4(tile[rr][cc], tile[rr + 1][cc], tile[rr + 2][cc], tile[rr + 3][cc]);
                st4(dst + (size_t)gc * srcRows + gr, v);
            } else {
                for (int e = 0; e < 4; e++)
                    if (gr + e < srcRows) dst[(size_t)gc * srcRows + gr + e] = from_f32<D>(tile[rr + e][cc]);
            }
        }
    }
}

template <typename S, typename D, bool TO_NHWC>
__global__ void __launch_bounds__(256) transpose_kernel(TransposeJob job) {
    __shared__ float tile[64][65];
    transpose_tile<S, D, TO_NHWC>(job, blockIdx.x, tile);
}

// fp32 accumulators -> a caller's half gradient maps in the same layout, rounded to nearest-even (blockIdx.y = level).
// Four elements per step: a 16-byte load (the accumulators are workspace slices, 256-byte aligned) and an 8-byte store
// when the destination allows it, scalar stores otherwise.
struct ConvertJob {
    const float* src[RSDET_MAX_LEVELS];
    void* dst[RSDET_MAX_LEVELS];
    size_t n[RSDET_MAX_LEVELS];
};
template <typename D>
__global__ void __launch_bounds__(256) convert_maps_kernel(ConvertJob job) {
    const float* __restrict__ src = job.src[blockIdx.y];
    D* __restrict__ dst = static_cast<D*>(job.dst[blockIdx.y]);
    const size_t n = job.n[blockIdx.y];
    const bool vec = ((size_t)dst & (4 * sizeof(D) - 1)) == 0;
    for (size_t i = 4 * ((size_t)blockIdx.x * blockDim.x + threadIdx.x); i < n; i += 4 * (size_t)gridDim.x * blockDim.x) {
        if (i + 3 < n) {
            const float4 v = __ldcs(reinterpret_cast<const float4*>(src + i));
            if (vec) st4(dst + i, v);
            else { dst[i] = from_f32<D>(v.x); dst[i + 1] = from_f32<D>(v.y); dst[i + 2] = from_f32<D>(v.z); dst[i + 3] = from_f32<D>(v.w); }
        } else {
            for (size_t e = i; e < n; e++) dst[e] = from_f32<D>(src[e]);
        }
    }
}

struct LevelSet;
struct RoiGeom;
struct PrepArgs {                 // order block and geometry blocks riding along with the NCHW->NHWC transpose
    const LevelSet* L;
    const float* rois;
    int K;
    int* order;
    RoiGeom* geoms;
    int32_t* levels_out;
    unsigned* counter;
};
template <typename S, typename D>
static int launch_transpose(bool to_nhwc, const S* const* src, D* const* dst, const int* H, const int* W, int L, int N,
                            int C, cudaStream_t st, const PrepArgs* prep = nullptr);

// ---------------------------------------------------------------------------------- geometry
struct alignas(16) RoiGeom {   // 48 bytes = three 16-byte words (copied as such by the order kernels)
    int batch, level, gh, gw;
    float cw, ch, bin_h, bin_w, start_h, start_w, cosv, sinv;
};

// oriented_single_level.py:73-89 (roi_rescale), :53-71 (map_roi_levels); roi_align_rotated_v1.py:85-120
__device__ __forceinline__ int roi_level(float w, float h, const LevelSet& L) {   // w, h: extended sizes
    if (L.num_levels <= 1) return 0;
    float s = sqrtf(__fmul_rn(w, h));
    float t = floorf(log2f(__fadd_rn(__fdiv_rn(s, L.finest_scale), 1e-6f)));
    t = fminf(fmaxf(t, 0.f), (float)(L.num_levels - 1));
    return (int)t;
}
__device__ __forceinline__ int roi_level(const float* __restrict__ r, const LevelSet& L) {
    return roi_level(__fmul_rn(L.extend_w, r[3]), __fmul_rn(L.extend_h, r[4]), L);
}
__device__ __forceinline__ RoiGeom roi_geometry(const float* __restrict__ r, const LevelSet& L) {
    RoiGeom g;
    g.batch = (int)r[0];
    float w = __fmul_rn(L.extend_w, r[3]);
    float h = __fmul_rn(L.extend_h, r[4]);
    const int lvl = roi_level(w, h, L);
    g.level = lvl;
    const float sc = L.scale[lvl];
    if (L.version == 1) {
        g.cw = __fsub_rn(__fmul_rn(r[1], sc), 0.5f);
        g.ch = __fsub_rn(__fmul_rn(r[2], sc), 0.5f);
    } else {
        g.cw = __fmul_rn(r[1], sc);
        g.ch = __fmul_rn(r[2], sc);
    }
    float rw = fmaxf(__fmul_rn(w, sc), 1.f);
    float rh = fmaxf(__fmul_rn(h, sc), 1.f);
    g.bin_h = __fdiv_rn(rh, (float)L.PH);
    g.bin_w = __fdiv_rn(rw, (float)L.PW);
    g.gh = L.sampling_ratio > 0 ? L.sampling_ratio : (int)ceilf(__fdiv_rn(rh, (float)L.PH));
    g.gw = L.sampling_ratio > 0 ? L.sampling_ratio : (int)ceilf(__fdiv_rn(rw, (float)L.PW));
    g.start_h = -rh * 0.5f;
    g.start_w = -rw * 0.5f;
    g.cosv = cosf(r[5]);
    g.sinv = sinf(r[5]);
    return g;
}

__device__ __forceinline__ void sample_xy(const RoiGeom& g, int version, int ph, int pw, int iy, int ix, float& x, float& y) {
    float yy = __fadd_rn(__fadd_rn(g.start_h, __fmul_rn((float)ph, g.bin_h)),
                         __fdiv_rn(__fmul_rn((float)iy + .5f, g.bin_h), (float)g.gh));
    float xx = __fadd_rn(__fadd_rn(g.start_w, __fmul_rn((float)pw, g.bin_w)),
                         __fdiv_rn(__fmul_rn((float)ix + .5f, g.bin_w), (float)g.gw));
    if (version == 1) {  // clockwise-positive, roi_align_rotated_v1.py:133-134
        x = __fadd_rn(__fadd_rn(__fmul_rn(xx, g.cosv), __fmul_rn(yy, g.sinv)), g.cw);
        y = __fadd_rn(__fsub_rn(__fmul_rn(yy, g.cosv), __fmul_rn(xx, g.sinv)), g.ch);
    } else {  // roi_align_rotated.py:116-117
        x = __fadd_rn(__fsub_rn(__fmul_rn(xx, g.cosv), __fmul_rn(yy, g.sinv)), g.cw);
        y = __fadd_rn(__fadd_rn(__fmul_rn(xx, g.sinv), __fmul_rn(yy, g.cosv)), g.ch);
    }
}

struct Taps {
    int o[4];    // pixel offsets (y*W+x) of lt, rt, lb, rb; all 0 when the sample is out of range
    float w[4];  // bilinear weights; all 0 when out of range
};

// bilinear_interpolate(_gradient): roi_align_rotated_v1.py:23-68, 149-190
__device__ __forceinline__ Taps make_taps(int H, int W, float y, float x) {
    Taps t;
    if (y < -1.0f || y > (float)H || x < -1.0f || x > (float)W) {
        t.o[0] = t.o[1] = t.o[2] = t.o[3] = 0;
        t.w[0] = t.w[1] = t.w[2] = t.w[3] = 0.f;
        return t;
    }
    if (y < 0) y = 0;
    if (x < 0) x = 0;
    int y_low = (int)y, x_low = (int)x, y_high, x_high;
    if (y_low >= H - 1) { y_high = y_low = H - 1; y = (float)y_low; } else y_high = y_low + 1;
    if (x_low >= W - 1) { x_high = x_low = W - 1; x = (float)x_low; } else x_high = x_low + 1;
    float ly = __fsub_rn(y, (float)y_low), lx = __fsub_rn(x, (float)x_low);
    float hy = __fsub_rn(1.f, ly), hx = __fsub_rn(1.f, lx);
    t.o[0] = y_low * W + x_low;  t.o[1] = y_low * W + x_high;
    t.o[2] = y_high * W + x_low; t.o[3] = y_high * W + x_high;
    t.w[0] = __fmul_rn(hy, hx); t.w[1] = __fmul_rn(hy, lx); t.w[2] = __fmul_rn(ly, hx); t.w[3] = __fmul_rn(ly, lx);
    return t;
}

// base + off*16 as ONE mad.wide.u32 (the compiler otherwise builds the 64-bit address in 4 instructions)
__device__ __forceinline__ const float* tap_ptr(const float4* base, unsigned off16) {
    unsigned long long a;
    asm("mad.wide.u32 %0, %1, 16, %2;" : "=l"(a) : "r"(off16), "l"((unsigned long long)base));
    return reinterpret_cast<const float*>(a);
}
// base + off * sizeof(Quad<T>::V) as ONE mad.wide.u32: tap offsets count 4-channel units of a channels-last map
template <typename T>
__device__ __forceinline__ const T* quad_ptr(const typename Quad<T>::V* base, unsigned off) {
    unsigned long long a;
    asm("mad.wide.u32 %0, %1, %2, %3;" : "=l"(a) : "r"(off), "n"((int)sizeof(typename Quad<T>::V)), "l"((unsigned long long)base));
    return reinterpret_cast<const T*>(a);
}
// four channels at p through the non-coherent path as the raw vector: one 16-byte load (fp32) or one 8-byte load
template <typename T>
__device__ __forceinline__ typename Quad<T>::V ldg4_raw(const T* p) {
    if constexpr (kIsF32<T>) {
        float4 r;
        asm volatile("ld.global.nc.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
        return r;
    } else {
        uint2 u;
        asm volatile("ld.global.nc.v2.b32 {%0,%1}, [%2];" : "=r"(u.x), "=r"(u.y) : "l"(p));
        return u;
    }
}
// the conversion of a raw vector to fp32: a loop that keeps 2-byte values in flight converts right before their FMAs
template <typename T> __device__ __forceinline__ decltype(auto) quad_f32(const typename Quad<T>::V& v) {
    if constexpr (kIsF32<T>) return (v);    // a reference: the fp32 kernels compile exactly as without this step
    else return unpack4<T>(v);
}
// the same load as fp32
template <typename T> __device__ __forceinline__ float4 ldg4(const T* p) { return quad_f32<T>(ldg4_raw(p)); }

__device__ __forceinline__ float4 ldg_cs_v4(const float* p) {
    float4 r;
    asm volatile("ld.global.cs.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
}
template <typename T>
__device__ __forceinline__ float4 ldcs4(const T* p) {     // streaming 4-channel load
    if constexpr (kIsF32<T>) {
        return ldg_cs_v4(p);
    } else {
        uint2 u;
        asm volatile("ld.global.cs.v2.b32 {%0,%1}, [%2];" : "=r"(u.x), "=r"(u.y) : "l"(p));
        return unpack4<T>(u);
    }
}
template <typename T>
__device__ __forceinline__ void stcs1(T* p, T v) {           // streaming scalar store
    if constexpr (kIsF32<T>) __stcs(p, v);
    else asm volatile("st.global.cs.b16 [%0], %1;" ::"l"(p), "h"(*reinterpret_cast<const unsigned short*>(&v)) : "memory");
}
// streaming 4-channel store of an fp32 quad: one 16-byte store (fp32) or one 8-byte store of values rounded to
// nearest-even (p aligned to 4 * sizeof(T)); stcs4_scalar: the same values with four scalar stores
template <typename T>
__device__ __forceinline__ void stcs4(T* p, float4 v) {
    if constexpr (kIsF32<T>) __stcs(reinterpret_cast<float4*>(p), v);
    else { const uint2 u = pack4<T>(v); asm volatile("st.global.cs.v2.b32 [%0], {%1,%2};" ::"l"(p), "r"(u.x), "r"(u.y) : "memory"); }
}
template <typename T>
__device__ __forceinline__ void stcs4_scalar(T* p, float4 v) {
    stcs1(p, from_f32<T>(v.x)); stcs1(p + 1, from_f32<T>(v.y)); stcs1(p + 2, from_f32<T>(v.z)); stcs1(p + 3, from_f32<T>(v.w));
}
// 4-channel store with an L2 cache policy (createpolicy): 16 bytes (fp32) or 8 bytes of values rounded to nearest-even
template <typename T>
__device__ __forceinline__ void st4_policy(T* p, float4 v, unsigned long long pol) {
    if constexpr (kIsF32<T>) {
        asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1,%2,%3,%4}, %5;" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w),
                     "l"(pol) : "memory");
    } else {
        const uint2 u = pack4<T>(v);
        asm volatile("st.global.L2::cache_hint.v2.b32 [%0], {%1,%2}, %3;" ::"l"(p), "r"(u.x), "r"(u.y), "l"(pol) : "memory");
    }
}
// shared -> global bulk copy (cp.async.bulk, SASS UBLKCP) with an evict-first L2 policy: the output stream must
// not push the feature pyramid out of L2.  Returns once the source has been read (shared memory may be reused
// or the CTA may exit); global visibility follows at kernel end.
__device__ __forceinline__ void bulk_store_evict_first(void* dst, const void* src_smem, unsigned bytes) {
    unsigned long long pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;"
                 ::"l"(dst), "r"((unsigned)__cvta_generic_to_shared(src_smem)), "r"(bytes), "l"(pol) : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
__device__ __forceinline__ void red_add_v4(float* p, float4 v) {
    asm volatile("red.global.add.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// shared-memory layout of the fast path
//   taps   : nsamp * Taps (32 B each)
//   stage  : [4][nbins][Q+1] floats   (k = channel within quad, Q = quads per CTA chunk)
// merged tap lists: bin pitch cap + 1 entries of 8 bytes, region rounded to 16 bytes (float4 staging follows)
__host__ __device__ inline size_t list_bytes(size_t nbins, size_t cap) { return (8 * nbins * (cap + 1) + 15) & ~(size_t)15; }
__host__ __device__ inline int quads_per_chunk(int C) { return (C / 4) < 64 ? (C / 4) : 64; }

// ---------------------------------------------------------------------------------- processing order
// RoIs are independent, so the ORDER in which CTAs take them is free.  A one-CTA counting sort buckets
// them by (level, 128-pixel image cell): CTAs that run at the same time then read the same few MB of
// one feature level, which keeps the gather inside L2 (the 200 MB output stream would otherwise push
// the 89 MB pyramid out between re-reads).  Output positions are untouched (roi index = output row).
constexpr int kCellShift = 7;   // 128-pixel cells in image coordinates
constexpr int kCellsPerAxis = 16;
constexpr int kBuckets = RSDET_MAX_LEVELS * kCellsPerAxis * kCellsPerAxis;

// bucket of a RoI in the locality order.  One image: (level, 128-px cell, boustrophedon rows).  A batch of images: the image
// is the major key -- CTAs that run at the same time then read ONE image's maps (8 images x 89 MB do not fit L2 together) --
// with 256-px cells so that (image slot, level, cell) still fits kBuckets.
__device__ __forceinline__ int roi_bucket(const float* __restrict__ r, int lvl, const LevelSet& L) {
    if (L.batch > 1 && L.num_levels * 64 <= kBuckets) {
        const int slots = kBuckets / (L.num_levels * 64);
        int cx = min(max((int)r[1] >> (kCellShift + 1), 0), 7);
        const int cy = min(max((int)r[2] >> (kCellShift + 1), 0), 7);
        if (cy & 1) cx = 7 - cx;
        const int b = min(max((int)r[0], 0), L.batch - 1) % slots;
        return ((b * L.num_levels + lvl) * 8 + cy) * 8 + cx;
    }
    int cx = min(max((int)r[1] >> kCellShift, 0), kCellsPerAxis - 1);
    const int cy = min(max((int)r[2] >> kCellShift, 0), kCellsPerAxis - 1);
    if (cy & 1) cx = kCellsPerAxis - 1 - cx;                      // boustrophedon rows: neighbouring buckets = neighbouring cells
    return (lvl * kCellsPerAxis + cy) * kCellsPerAxis + cx;
}

constexpr int kPrepMaxRois = 16384;
// The locality order of a call as ONE block of any size: block 0 of roi_prep_kernel, or for NCHW callers an extra block
// of the NCHW->NHWC transpose, whose other SMs are busy for 30 us on a 1024^2 pyramid anyway (the order is a 7.8 us
// single-CTA latency chain).  Doing the geometry in the same block as well was measured and dropped: sin/cos/log2 of 4000
// RoIs on one SM take longer than the launch they replace.  s_hist: kBuckets ints, s_warp: 32 ints.
static_assert(kBuckets <= 65536, "bucket ids are cached as unsigned short");
template <int THREADS>
__device__ __forceinline__ void roi_order_block(const LevelSet& L, const float* __restrict__ rois, int K,
                                                int* __restrict__ order, int* s_hist, int* s_warp, unsigned short* s_bkt, int bkt_cap) {
    const int tid = threadIdx.x;
    for (int i = tid; i < kBuckets; i += THREADS) s_hist[i] = 0;
    __syncthreads();
    auto bucket_of = [&](const float* r, int lvl) { return roi_bucket(r, lvl, L); };
    for (int i = tid; i < K; i += THREADS) {   // s_bkt: the buckets of the first bkt_cap RoIs are kept for the scatter pass
        const float* r = rois + (size_t)i * 6;
        const int bkt = bucket_of(r, roi_level(r, L));
        if (i < bkt_cap) s_bkt[i] = (unsigned short)bkt;
        atomicAdd(&s_hist[bkt], 1);
    }
    __syncthreads();
    // exclusive scan of kBuckets counters, kBuckets / THREADS consecutive ones per thread
    constexpr int PER = kBuckets / THREADS;
    int a[PER], sum = 0;
#pragma unroll
    for (int k = 0; k < PER; k++) { a[k] = s_hist[PER * tid + k]; sum += a[k]; }
    int x = sum;
    const int lane = tid & 31, w = tid >> 5;
    for (int o = 1; o < 32; o <<= 1) { int y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
    if (lane == 31) s_warp[w] = x;
    __syncthreads();
    if (w == 0) {
        int v = lane < THREADS / 32 ? s_warp[lane] : 0;
        for (int o = 1; o < 32; o <<= 1) { int y = __shfl_up_sync(0xffffffffu, v, o); if (lane >= o) v += y; }
        s_warp[lane] = v;
    }
    __syncthreads();
    int excl = (w ? s_warp[w - 1] : 0) + x - sum;
#pragma unroll
    for (int k = 0; k < PER; k++) { s_hist[PER * tid + k] = excl; excl += a[k]; }
    __syncthreads();
    for (int i = tid; i < K; i += THREADS) {
        const float* r = rois + (size_t)i * 6;
        const int bkt = i < bkt_cap ? (int)s_bkt[i] : bucket_of(r, roi_level(r, L));
        order[atomicAdd(&s_hist[bkt], 1)] = i;
    }
}

// The prologue of a fast call, ONE launch: block 0 = the locality order (when there is one), the other blocks = the
// per-RoI geometry records BY ROI INDEX + the reset of the persistent forward kernel's work counter (when there is one:
// the backward has none).  The gather kernels look a record up through order[] (the persistent one while it gathers the
// previous item), so nothing has to be written in processing order and order and geometry do not depend on each other.
// sin/cos/log2/sqrt and six divisions per RoI are done by K parallel threads here instead of by thread 0 of every RoI's
// CTA (a ~1.5 us serial chain in front of each CTA's barrier).
constexpr int kPrepBucketCache = 16384;   // buckets cached by the order block: 32 KB + the 8 KB histogram of static smem
__device__ __forceinline__ void roi_geometry_by_index(const LevelSet& L, const float* __restrict__ rois, int K, int i,
                                                      RoiGeom* __restrict__ geoms, int32_t* __restrict__ levels_out) {
    if (i >= K) return;
    const RoiGeom g = roi_geometry(rois + (size_t)i * 6, L);
    geoms[i] = g;
    if (levels_out) levels_out[i] = g.level;
}
__global__ void __launch_bounds__(1024) roi_prep_kernel(LevelSet L, const float* __restrict__ rois, int K, int* __restrict__ order,
                                                        RoiGeom* __restrict__ geoms, int32_t* __restrict__ levels_out,
                                                        unsigned* __restrict__ counter) {
    int gb = blockIdx.x;
    if (order) {
        if (gb == 0) {
            __shared__ int s_hist[kBuckets + 32];
            __shared__ unsigned short s_bkt[kPrepBucketCache];
            roi_order_block<1024>(L, rois, K, order, s_hist, s_hist + kBuckets, s_bkt, kPrepBucketCache);
            return;
        }
        gb--;
    }
    if (gb == 0 && threadIdx.x == 0 && counter) *counter = 0u;
    roi_geometry_by_index(L, rois, K, gb * 1024 + threadIdx.x, geoms, levels_out);
}

// NCHW callers: the pyramid transpose with the order block riding along as block 0 and the geometry blocks after it
template <typename T>
__global__ void __launch_bounds__(256) transpose_prep_kernel(TransposeJob job, LevelSet L, const float* __restrict__ rois, int K,
                                                             int* __restrict__ order, RoiGeom* __restrict__ geoms,
                                                             int32_t* __restrict__ levels_out, unsigned* __restrict__ counter,
                                                             int geom_blocks) {
    __shared__ float tile[64][65];
    static_assert(sizeof(float) * 64 * 65 >= sizeof(int) * (kBuckets + 32), "the prep block borrows the transpose tile");
    if (blockIdx.x == 0) {
        int* s_hist = reinterpret_cast<int*>(&tile[0][0]);
        unsigned short* s_bkt = reinterpret_cast<unsigned short*>(s_hist + kBuckets + 32);
        const int bkt_cap = (int)((sizeof(float) * 64 * 65 - sizeof(int) * (kBuckets + 32)) / sizeof(unsigned short));
        roi_order_block<256>(L, rois, K, order, s_hist, s_hist + kBuckets, s_bkt, bkt_cap);
        return;
    }
    if ((int)blockIdx.x <= geom_blocks) {      // geometry records by RoI index, 256 per block
        if (blockIdx.x == 1 && threadIdx.x == 0) *counter = 0u;
        roi_geometry_by_index(L, rois, K, ((int)blockIdx.x - 1) * 256 + threadIdx.x, geoms, levels_out);
        return;
    }
    transpose_tile<T, T, true>(job, blockIdx.x - 1 - geom_blocks, tile);
}

// S == D: either direction (NCHW -> NHWC may carry the prep blocks); S != D: NHWC fp32 accumulators -> NCHW half maps
template <typename S, typename D>
static int launch_transpose(bool to_nhwc, const S* const* src, D* const* dst, const int* H, const int* W, int L, int N,
                            int C, cudaStream_t st, const PrepArgs* prep) {
    TransposeJob job;
    job.num_levels = L; job.N = N; job.C = C;
    int total = 0;
    for (int l = 0; l < L; l++) {
        job.src[l] = src[l]; job.dst[l] = dst[l]; job.HW[l] = H[l] * W[l];
        job.tile_begin[l] = total;
        total += N * ceil_div(job.HW[l], 64) * ceil_div(C, 64);
    }
    job.tile_begin[L] = total;
    if constexpr (std::is_same<S, D>::value) {
        if (prep && to_nhwc) {
            const int geom_blocks = ceil_div(prep->K, 256);
            transpose_prep_kernel<S><<<total + 1 + geom_blocks, 256, 0, st>>>(job, *prep->L, prep->rois, prep->K, prep->order,
                                                                               prep->geoms, prep->levels_out, prep->counter,
                                                                               geom_blocks);
            count_launch();
            return cuda_status();
        }
        if (total == 0) return RSDET_OK;
        if (to_nhwc) transpose_kernel<S, D, true><<<total, 256, 0, st>>>(job);
        else transpose_kernel<S, D, false><<<total, 256, 0, st>>>(job);
    } else {
        if (to_nhwc || total == 0) return to_nhwc ? RSDET_EINVAL : RSDET_OK;
        transpose_kernel<S, D, false><<<total, 256, 0, st>>>(job);
    }
    count_launch();
    return cuda_status();
}

// ---------------------------------------------------------------------------------- tap lists
// Shared by forward and backward.  Measured on B200 (profiles/README.md): the gather is bound by L2
// round trips and L1 load wavefronts -- every bilinear tap is a 512-byte warp load and a RoI issues 784
// of them per 128 channels, ~9x its own output -- not by HBM.  So the sampling grid is computed once per
// RoI (A1) AND merged per bin (A2): taps of the bin's samples that land on the same pixel are summed
// into one (offset, weight) entry and zero-weight taps are dropped; on the benchmark proposals 16 taps
// collapse to ~9.  Offsets are in 16-byte units of the channels-last map (one mad.wide per address).
//   s_list [nbins*(cap+1)] int2 {offset, weight bits} (bin pitch cap + 1: conflict-free per-bin lanes),
//   s_cnt [nbins], tmp: 3*nbins*(cap+1) words of scratch.
//   unit: stored offset = pixel * unit (C/4: 4-channel units)
// Called by all kRoiThreads threads of the CTA.
__device__ __forceinline__ void build_tap_lists(const RoiGeom& g, const LevelSet& L, int H, int W, int2* s_list, int* s_cnt,
                                                float* tmp, int unit) {
    const int tid = threadIdx.x;
    const int PW_ = L.PW;
    const int nbins = L.PH * L.PW;
    const int spb = L.sampling_ratio * L.sampling_ratio;
    const int nsamp = nbins * spb, cap = 4 * spb, ntaps = nbins * cap;
    const int C4 = unit;
    int* s_off = reinterpret_cast<int*>(tmp);
    float* s_w = tmp + ntaps + nbins;      // room for the cap + 1 pitch
    float* s_wsum = tmp + 2 * (ntaps + nbins);
    // A1: one thread per sample.  Scratch pitch per bin = cap + 1 words when the per-bin merge below reads it
    // with one lane per bin (lane stride 17 words: conflict-free; 16 would be a 16-way bank conflict).
    const int tp = cap == 16 ? 17 : cap;
    for (int s = tid; s < nsamp; s += kRoiThreads) {
        int b = s / spb, q = s % spb;
        int ph = b / PW_, pw = b % PW_, iy = q / g.gw, ix = q % g.gw;
        float x, y;
        sample_xy(g, L.version, ph, pw, iy, ix, x, y);
        const Taps t = make_taps(H, W, y, x);
#pragma unroll
        for (int k = 0; k < 4; k++) {
            s_off[b * tp + q * 4 + k] = t.o[k] * C4;
            s_w[b * tp + q * 4 + k] = t.w[k];
        }
    }
    __syncthreads();
    if (cap == 16) {
        // A2 (2x2 sampling grid, the Oriented R-CNN setting): ONE LANE PER BIN, everything in registers.  The
        // warp-cooperative variant it replaces (below, still used for cap == 4) spent 32 shuffles per 16 taps:
        // 4.1 M SHFL per 4000 RoIs = 6.9 M of the kernel's 29.8 M L1 wavefronts (shuffles share the data pipe
        // of the gather loads, profiles/README.md).  Same arithmetic: a tap is a LEADER if its weight is
        // non-zero and no earlier live tap of the bin hits the same pixel; a leader adds the weights of its
        // later duplicates in tap order; leaders are compacted in tap order.
        for (int b = tid; b < nbins; b += kRoiThreads) {
            int o[16];
            float w[16];
#pragma unroll
            for (int j = 0; j < 16; j++) { o[j] = s_off[b * 17 + j]; w[j] = s_w[b * 17 + j]; }
            int pos = 0;
#pragma unroll
            for (int j = 0; j < 16; j++) {
                float acc = w[j];
#pragma unroll
                for (int i = 0; i < 16; i++) {
                    if (i <= j) continue;                            // constant trip count: stays in registers
                    const bool same = o[i] == o[j] && w[j] != 0.f;   // w[j] == 0: dead or already absorbed
                    acc += same ? w[i] : 0.f;
                    w[i] = same ? 0.f : w[i];
                }
                if (w[j] != 0.f) s_list[b * 17 + pos++] = make_int2(o[j], __float_as_int(acc));
            }
            s_cnt[b] = pos;
        }
        __syncthreads();
        return;
    }
    if (cap == 4) {
        // A2 (fast): cap lanes per bin, everything in registers.  Each lane walks the cap lanes of its bin with
        // warp shuffles (uniform trip count): it is a LEADER if no earlier live lane hits the same pixel, and it
        // sums the weights of all live lanes on its pixel in lane order; a ballot of the leaders gives each
        // one its slot in the bin's compacted list.
        const int lane = tid & 31;
        const int rounds = (ntaps + kRoiThreads - 1) / kRoiThreads;
        for (int rd = 0; rd < rounds; rd++) {
            const int t = rd * kRoiThreads + tid;
            const bool in = t < ntaps;
            const int b = in ? t / cap : 0, j = in ? t - b * cap : 0;
            const int o = in ? s_off[t] : -1;
            const float w = in ? s_w[t] : 0.f;
            const bool live = in && w != 0.f;
            const int seg = lane & ~(cap - 1);                        // first lane of my bin inside the warp
            bool leader = live;
            float wsum = 0.f;
            for (int i = 0; i < cap; i++) {                           // same trip count on every lane
                const int oi = __shfl_sync(0xffffffffu, o, seg + i);
                const float wi = __shfl_sync(0xffffffffu, w, seg + i);
                const bool same = live && wi != 0.f && oi == o;
                if (same && i < (lane - seg)) leader = false;
                if (same) wsum += wi;
            }
            const unsigned leaders = __ballot_sync(0xffffffffu, leader);
            const unsigned segmask = ((1u << cap) - 1u) << seg;       // cap is 4 or 16 here
            if (leader) s_list[b * (cap + 1) + __popc(leaders & segmask & ((1u << lane) - 1u))] = make_int2(o, __float_as_int(wsum));
            if (in && j == 0) s_cnt[b] = __popc(leaders & segmask);
        }
        __syncthreads();
        return;
    }
    // A2a: one thread per tap: a tap is a LEADER if its weight is non-zero and no earlier tap of the bin
    // hits the same pixel; a leader collects the weights of its later duplicates (fixed order).
    for (int t = tid; t < ntaps; t += kRoiThreads) {
        const int b = t / cap, j = t - b * cap;
        const int* ob = s_off + b * cap;
        const float* wb = s_w + b * cap;
        const int o = ob[j];
        float w = wb[j];
        bool leader = w != 0.f;
        for (int i = 0; i < j && leader; i++) leader = !(ob[i] == o && wb[i] != 0.f);
        if (leader)
            for (int i = j + 1; i < cap; i++)
                if (ob[i] == o) w += wb[i];
        s_wsum[t] = leader ? w : 0.f;
    }
    __syncthreads();
    // A2b: compaction (position = number of leaders before me in my bin)
    for (int t = tid; t < ntaps; t += kRoiThreads) {
        const int b = t / cap, j = t - b * cap;
        const float* ws = s_wsum + b * cap;
        const float w = ws[j];
        int pos = 0;
        for (int i = 0; i < j; i++) pos += ws[i] != 0.f;
        if (w != 0.f) s_list[b * (cap + 1) + pos] = make_int2(s_off[t], __float_as_int(w));
        if (j == cap - 1) s_cnt[b] = pos + (w != 0.f);
    }
    __syncthreads();
}

// Conflict-free access to the [c][bin] staging block.  A warp touches channels 4*lane + i of one bin at a
// time; with all lanes on the same component i the 32 addresses fall on 8 banks (4-way conflict: 7.2 M of the
// forward kernel's 34 M L1 wavefronts in profiles/r1_d).  Lane octet o = lane/8 therefore handles component
// (i + o) & 3 at step i: for an odd bin count the four octets land on the four residues mod 4 and the 32
// banks are distinct.  rot4 rotates a quad left by o so that step i finds its value in slot i.
__device__ __forceinline__ float4 rot4(float4 v, int o) {
    if (o & 1) v = make_float4(v.y, v.z, v.w, v.x);
    if (o & 2) v = make_float4(v.z, v.w, v.x, v.y);
    return v;
}
__device__ __forceinline__ float4 unrot4(float4 v, int o) { return rot4(v, (4 - o) & 3); }

// ---------------------------------------------------------------------------------- forward (fast)
// One CTA per (RoI, chunk of up to 64 channel quads), thread = (channel quad(s), bin group).  QPT = 2:
// the second channel quad is an immediate +512 B off the same address.  Launch bounds for THREE CTAs per SM: the driver then
// picks the 196 KB carve-out (60 KB of L1 instead of 28) -- 143.2 -> 131.9 us per bench tile (profiles/README.md, third pass).
// NHWC_OUT: out is (K, PH, PW, C) -- a thread stores its channel quads of a bin straight to global memory, with vector stores
// when out's base is aligned to four elements (scalar stores otherwise), and the staging block is only phase-A scratch.
template <int QPT, typename T = float, typename O = float, bool NHWC_OUT = false>   // T: feature elements, O: output elements
__global__ void __launch_bounds__(kRoiThreads, 3)
roi_align_fwd_kernel(LevelSet L, const int* __restrict__ order, const RoiGeom* __restrict__ geoms, int K, O* __restrict__ out) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int roi = order ? order[blockIdx.x] : blockIdx.x;
    const int tid = threadIdx.x;
    const int nbins = L.PH * L.PW;
    const int spb = L.sampling_ratio * L.sampling_ratio;  // samples per bin (fast path: fixed grid)
    const int cap = 4 * spb;                               // taps per bin before merging
    const int C = L.C;
    const int Q = quads_per_chunk(C);
    const int chunk0 = blockIdx.y * Q * 4;                 // first channel of this chunk
    const int Qc = min(Q, (C - chunk0) / 4);               // quads in this chunk
    // smem: [merged lists: nbins*cap int2][counts: nbins int, padded][staging [c][bin] | phase-A scratch]
    int2* s_list = reinterpret_cast<int2*>(smem_raw);
    int* s_cnt = reinterpret_cast<int*>(smem_raw + list_bytes(nbins, cap));
    O* s_stage = reinterpret_cast<O*>(smem_raw + list_bytes(nbins, cap) + ((nbins * 4 + 15) & ~15));

    const RoiGeom g = geoms[roi];
    const int H = L.H[g.level], W = L.W[g.level];
    build_tap_lists(g, L, H, W, s_list, s_cnt, reinterpret_cast<float*>(s_stage), C >> 2);   // the scratch is dead after its final barrier

    const int lanes = QPT == 2 ? 32 : Qc;                  // threads per bin group
    const int groups = kRoiThreads / lanes;
    const int cq = tid % lanes, grp = tid / lanes;
    const int oct = (cq >> 3) & 3;
    const typename Quad<T>::V* __restrict__ feat =
        reinterpret_cast<const typename Quad<T>::V*>(feat_base<T>(L, g.level) + (size_t)g.batch * H * W * C + chunk0) + cq;
    const bool pow2 = (spb & (spb - 1)) == 0;
    const float count = (float)max(spb, 1), inv_count = 1.f / count;
    [[maybe_unused]] const bool out_vec = (((size_t)out) & (4 * sizeof(O) - 1)) == 0;
    if (grp < groups) {
        for (int b = grp; b < nbins; b += groups) {
            float4 acc[QPT];
#pragma unroll
            for (int u = 0; u < QPT; u++) acc[u] = make_float4(0.f, 0.f, 0.f, 0.f);
            const int2* lp = s_list + b * (cap + 1);
            const int cnt = s_cnt[b];
            for (int e = 0; e < cnt; e += 4) {
                int2 en[4];
#pragma unroll
                for (int k = 0; k < 4; k++) en[k] = lp[min(e + k, cnt - 1)];  // warp-uniform broadcast reads
                float4 v[QPT][4];
#pragma unroll
                for (int k = 0; k < 4; k++)
                    if (e + k < cnt) {
#pragma unroll
                        for (int u = 0; u < QPT; u++) v[u][k] = ldg4(quad_ptr<T>(feat, (unsigned)en[k].x) + u * 128);
                    }
#pragma unroll
                for (int k = 0; k < 4; k++)
                    if (e + k < cnt) {
                        const float wt = __int_as_float(en[k].y);
#pragma unroll
                        for (int u = 0; u < QPT; u++) {
                            acc[u].x = fmaf(wt, v[u][k].x, acc[u].x);
                            acc[u].y = fmaf(wt, v[u][k].y, acc[u].y);
                            acc[u].z = fmaf(wt, v[u][k].z, acc[u].z);
                            acc[u].w = fmaf(wt, v[u][k].w, acc[u].w);
                        }
                    }
            }
#pragma unroll
            for (int u = 0; u < QPT; u++) {
                // output_val /= count (:143); a power-of-two count makes the reciprocal multiply exact
                if (pow2) { acc[u].x *= inv_count; acc[u].y *= inv_count; acc[u].z *= inv_count; acc[u].w *= inv_count; }
                else { acc[u].x /= count; acc[u].y /= count; acc[u].z /= count; acc[u].w /= count; }
                const int c0 = (cq + u * 32) * 4;
                if constexpr (NHWC_OUT) {
                    O* const p = out + ((size_t)roi * nbins + b) * C + chunk0 + c0;
                    if (out_vec) stcs4(p, acc[u]);
                    else stcs4_scalar(p, acc[u]);
                    continue;
                }
                const float4 r = rot4(acc[u], oct);
                s_stage[(c0 + ((0 + oct) & 3)) * nbins + b] = from_f32<O>(r.x);
                s_stage[(c0 + ((1 + oct) & 3)) * nbins + b] = from_f32<O>(r.y);
                s_stage[(c0 + ((2 + oct) & 3)) * nbins + b] = from_f32<O>(r.z);
                s_stage[(c0 + ((3 + oct) & 3)) * nbins + b] = from_f32<O>(r.w);
            }
        }
    }
    if constexpr (NHWC_OUT) return;
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    // the staged block IS the output block of this (roi, chunk): one bulk copy shared -> global (TMA) when it is
    // 16-byte aligned, else a coalesced copy with streaming stores
    O* __restrict__ dst = out + ((size_t)roi * C + chunk0) * nbins;
    const int total = Qc * 4 * nbins;
    constexpr int kVec = 16 / sizeof(O);                   // elements per 16 bytes
    if ((((size_t)roi * C + chunk0) * nbins % kVec) == 0 && (total % kVec) == 0 && (((size_t)out) & 15) == 0) {
        if (tid == 0) bulk_store_evict_first(dst, s_stage, (unsigned)(total * sizeof(O)));
    } else {
        for (int e = tid; e < total; e += kRoiThreads) stcs1(dst + e, s_stage[e]);
    }
}

// ---------------------------------------------------------------------------------- forward (7x7, persistent) -- the default
// The Oriented R-CNN geometry (7x7 bins, 2x2 samples, 256-channel chunks) with everything roi_align_fwd_kernel reads at
// run time fixed at compile time, and the gather loop restructured around what the per-instruction stall samples of
// that kernel showed (profiles/README.md "round 2, second pass"): of its 18 000 warp instructions per RoI only 3 800 were
// FFMA and 940 LDG -- the rest were index clamps, 64-bit address pairs, run-time pitches and the rotate/stage arithmetic
// -- and a third of the gather's stall samples sat on the LEA that waits for the tap-list LDS, i.e. every batch paid TWO
// dependent L1 round trips (list entries, then pixels) behind the other CTAs' queued loads.  Here
//   * the list entries of the NEXT batch (or of the warp's next bin) are read while the current batch's pixel loads are
//     in flight, so a batch is one round trip;
//   * a warp walks its bins as one flat sequence of batches; the [c][bin] staging stores of a finished bin are issued
//     after the first loads of the next bin, not before them;
//   * the CTA is PERSISTENT, three per SM (profiles/README.md "third pass"): 148 x 3 CTAs of 8 warps take (RoI,
//     256-channel chunk) items from a counter in the workspace (dynamic: RoIs differ in tap count); the counter is zeroed
//     by the prologue (roi_prep_kernel or transpose_prep_kernel), which always runs in front of this kernel on the same
//     stream, so concurrent calls on different streams and CUDA-graph replays need nothing else;
//   * three CTAs instead of four leave the compiler 78 registers (no spill at 8 warps) and -- what the experiments that
//     forced the CTA count by padding shared memory could not show -- let the driver pick the 196 KB carve-out: L1 grows
//     from 28 to 60 KB, its hit rate from 14 % to 27 %, the bytes pulled through the SM's L2 port fall by 16 %;
//   * the merged lists are built IN PLACE (A1 writes the sixteen raw taps of a bin into the bin's own list slots, A2
//     reads them into registers and writes the merged entries back), so the list build does not borrow the staging
//     block and runs while the previous item's bulk store is still reading it; the next item's geometry record is
//     fetched with cp.async during the gather.
// Lists have a pitch of 18 entries (16-byte aligned: a batch's four entries are two LDS.128; the count sits in entry 16).
// Arithmetic and tap order are those of roi_align_fwd_kernel<2>: bit-identical results.  The measured variants (warps,
// CTAs per SM, taps per batch, load flavours, one CTA per RoI) are in profiles/README.md.
constexpr int kFwd77pWarps = 8, kFwd77pCtasPerSm = 3;
constexpr int kFwd77pTaps = 4;   // list entries per batch: 8 vector loads in flight per thread
constexpr size_t kStage77pOffset = (8 * 49 * 18 + 16 + 48 + 127) & ~(size_t)127;   // lists | next item | next record | staging
// T: feature elements (a half map halves the bytes of every tap load: two 8-byte loads per lane and tap); O: output
// elements (a half output halves the staging block and its bulk store).  NHWC_OUT: out is (K, 7, 7, C); a lane's two
// channel quads of a bin are contiguous 16-byte (8-byte when half) pieces of it, stored straight from registers with the
// same evict-first L2 policy -- no staging block, no bulk copy, and only the lists and the record in shared memory.
template <typename T, typename O, bool NHWC_OUT = false>
__global__ void __launch_bounds__(32 * kFwd77pWarps, kFwd77pCtasPerSm)
roi_align_fwd77p_kernel(LevelSet L, const int* __restrict__ order, const RoiGeom* __restrict__ geoms, int K, int chunks,
                        O* __restrict__ out, unsigned* __restrict__ counter) {
    constexpr int NB = 49, PITCH = 18, WARPS = kFwd77pWarps, TAPS = kFwd77pTaps, THREADS = 32 * WARPS;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int2* s_list = reinterpret_cast<int2*>(smem_raw);
    volatile int* s_next = reinterpret_cast<volatile int*>(smem_raw + 8 * NB * PITCH);
    volatile int* s_roi = reinterpret_cast<volatile int*>(smem_raw + 8 * NB * PITCH + 4);      // RoI index of the record in s_geom
    const RoiGeom* s_geom = reinterpret_cast<const RoiGeom*>(smem_raw + 8 * NB * PITCH + 16);
    O* s_stage = reinterpret_cast<O*>(smem_raw + kStage77pOffset);
    const int C = L.C, items = K * chunks;
    const int oct = (lane >> 3) & 3;
    O* const sbase = s_stage + lane * 4 * NB;
    [[maybe_unused]] unsigned long long pol = 0;   // NHWC_OUT: the output stores' L2 policy
    if constexpr (NHWC_OUT) asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    int idx = blockIdx.x;
    if (tid < 3 && idx < items) {
        const int r = order ? order[idx / chunks] : idx / chunks;      // position in processing order -> RoI
        reinterpret_cast<float4*>(smem_raw + 8 * NB * PITCH + 16)[tid] = reinterpret_cast<const float4*>(geoms + r)[tid];
        if (tid == 0) *s_roi = r;
    }
    __syncthreads();
#pragma unroll 1
    while (idx < items) {
        RoiGeom g = *s_geom;                   // this item's record (prefetched during the previous gather)
        const int roi = *s_roi;
        g.gh = 2; g.gw = 2;
        const int chunk0 = (idx % chunks) * 256;
        const int H = L.H[g.level], W = L.W[g.level];
        // A1: one thread per sample, raw taps straight into the bin's list slots
        if (tid < NB * 4) {
            const int b = tid >> 2, q = tid & 3;
            const int ph = b / 7, pw = b - ph * 7, iy = q >> 1, ix = q & 1;
            float x, y;
            sample_xy(g, L.version, ph, pw, iy, ix, x, y);
            const Taps t = make_taps(H, W, y, x);
#pragma unroll
            for (int k = 0; k < 4; k++) s_list[b * PITCH + q * 4 + k] = make_int2(t.o[k] * (C >> 2), __float_as_int(t.w[k]));
        }
        __syncthreads();
        // A2: one lane per bin, merge in registers, write back in place (same arithmetic and order as build_tap_lists)
        if (tid < NB) {
            const int b = tid;
            int o[16];
            float w[16];
#pragma unroll
            for (int j = 0; j < 16; j++) { const int2 e = s_list[b * PITCH + j]; o[j] = e.x; w[j] = __int_as_float(e.y); }
            int pos = 0;
#pragma unroll
            for (int j = 0; j < 16; j++) {
                float acc = w[j];
#pragma unroll
                for (int i = 0; i < 16; i++) {
                    if (i <= j) continue;
                    const bool same = o[i] == o[j] && w[j] != 0.f;
                    acc += same ? w[i] : 0.f;
                    w[i] = same ? 0.f : w[i];
                }
                if (w[j] != 0.f) s_list[b * PITCH + pos++] = make_int2(o[j], __float_as_int(acc));
            }
            s_list[b * PITCH + 16] = make_int2(pos, 0);
        }
        if (tid == THREADS - 1) {      // a thread without A1 / A2 work: the previous block must have left the staging area; next item
            if constexpr (!NHWC_OUT) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // returns at once when nothing is pending
            *s_next = (int)(atomicAdd(counter, 1u) + gridDim.x);
        }
        __syncthreads();
        if (tid < 3 && *s_next < items) {      // the next record: three 16-byte async copies, in flight during the gather
            const int nidx = *s_next;
            const int r = order ? __ldg(order + nidx / chunks) : nidx / chunks;
            if (tid == 0) *s_roi = r;
            asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(s_geom) + 16u * tid),
                         "l"(reinterpret_cast<const char*>(geoms + r) + 16 * tid) : "memory");
            asm volatile("cp.async.commit_group;" ::: "memory");
        }

        const typename Quad<T>::V* __restrict__ feat =
            reinterpret_cast<const typename Quad<T>::V*>(feat_base<T>(L, g.level) + (size_t)g.batch * H * W * C + chunk0) + lane;
        auto stage = [&](float4 a0, float4 a1, int b) {
            a0.x *= 0.25f; a0.y *= 0.25f; a0.z *= 0.25f; a0.w *= 0.25f;   // output_val /= count (:143), count = 4: exact
            a1.x *= 0.25f; a1.y *= 0.25f; a1.z *= 0.25f; a1.w *= 0.25f;
            if constexpr (NHWC_OUT) {
                O* const p = out + ((size_t)roi * NB + b) * C + chunk0 + lane * 4;
                st4_policy(p, a0, pol);
                st4_policy(p + 128, a1, pol);
                return;
            }
            const float4 r0 = rot4(a0, oct), r1 = rot4(a1, oct);
            O* const sb = sbase + b;
            O* const q0 = sb + ((0 + oct) & 3) * NB;
            O* const q1 = sb + ((1 + oct) & 3) * NB;
            O* const q2 = sb + ((2 + oct) & 3) * NB;
            O* const q3 = sb + ((3 + oct) & 3) * NB;
            q0[0] = from_f32<O>(r0.x); q1[0] = from_f32<O>(r0.y); q2[0] = from_f32<O>(r0.z); q3[0] = from_f32<O>(r0.w);
            q0[128 * NB] = from_f32<O>(r1.x); q1[128 * NB] = from_f32<O>(r1.y); q2[128 * NB] = from_f32<O>(r1.z); q3[128 * NB] = from_f32<O>(r1.w);
        };
        const int2* lp = s_list + warp * PITCH;
        int4 en[TAPS / 2];
#pragma unroll
        for (int t = 0; t < TAPS / 2; t++) en[t] = reinterpret_cast<const int4*>(lp)[t];
        int cnt = lp[16].x;
#pragma unroll 1
        for (int b = warp; b < NB; b += WARPS) {
            float4 acc0 = make_float4(0.f, 0.f, 0.f, 0.f), acc1 = acc0;
            const int nbin = min(b + WARPS, NB - 1);
            int ncnt = cnt;
            int e = 0;
#pragma unroll 1
            do {
                typename Quad<T>::V va[TAPS], vb[TAPS];   // raw: 2-byte values convert right before their FMAs
                float wt[TAPS];
#pragma unroll
                for (int t = 0; t < TAPS; t++) {
                    const int off = (t & 1) ? en[t >> 1].z : en[t >> 1].x;
                    wt[t] = __int_as_float((t & 1) ? en[t >> 1].w : en[t >> 1].y);
                    if (e + t < cnt) { const T* q = quad_ptr<T>(feat, (unsigned)off); va[t] = ldg4_raw(q); vb[t] = ldg4_raw(q + 128); }
                }
                const int e0 = e;
                e += TAPS;
                const bool more = e < cnt;
                const int2* np = more ? lp + e : s_list + nbin * PITCH;
                if (!more) ncnt = s_list[nbin * PITCH + 16].x;
#pragma unroll
                for (int t = 0; t < TAPS / 2; t++) en[t] = reinterpret_cast<const int4*>(np)[t];
#pragma unroll
                for (int t = 0; t < TAPS; t++)
                    if (e0 + t < cnt) {
                        const auto& a = quad_f32<T>(va[t]);
                        const auto& c = quad_f32<T>(vb[t]);
                        acc0.x = fmaf(wt[t], a.x, acc0.x); acc0.y = fmaf(wt[t], a.y, acc0.y); acc0.z = fmaf(wt[t], a.z, acc0.z); acc0.w = fmaf(wt[t], a.w, acc0.w);
                        acc1.x = fmaf(wt[t], c.x, acc1.x); acc1.y = fmaf(wt[t], c.y, acc1.y); acc1.z = fmaf(wt[t], c.z, acc1.z); acc1.w = fmaf(wt[t], c.w, acc1.w);
                    }
            } while (e < cnt);
            stage(acc0, acc1, b);
            lp = s_list + nbin * PITCH;
            cnt = ncnt;
        }
        if (tid < 3) asm volatile("cp.async.wait_all;" ::: "memory");
        if constexpr (NHWC_OUT) {
            __syncthreads();           // the record has landed, every warp is done with the lists
            idx = *s_next;
            continue;
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncthreads();
        if (tid == THREADS - 1) {      // the thread that will wait for it
            unsigned long long pol;
            asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;"
                         ::"l"(out + ((size_t)roi * C + chunk0) * NB), "r"((unsigned)__cvta_generic_to_shared(s_stage)), "r"(256u * NB * (unsigned)sizeof(O)), "l"(pol) : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
        idx = *s_next;
    }
    if constexpr (!NHWC_OUT)
        if (tid == THREADS - 1) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}

// cudaFuncSetAttribute is per device: remember what was set for each one (a process may drive several GPUs)
static void set_dyn_smem(const void* func, size_t bytes) {
    struct Slot { const void* f; size_t b; };
    static Slot slots[64][16];
    static std::mutex mu;
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> lk(mu);
    if (dev < 0 || dev >= 64) { cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes); return; }
    for (int i = 0; i < 16; i++) {
        Slot& s = slots[dev][i];
        if (s.f == func || s.f == nullptr) {
            if (s.f == func && s.b >= bytes) return;
            s.f = func; s.b = bytes;
            cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
            return;
        }
    }
    cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

// measurement aid (rsdet_roi_align_profile_events): events recorded around the gather kernel of the next forward call
static thread_local cudaEvent_t t_prof_start = nullptr, t_prof_stop = nullptr;
struct GatherTimer {       // records on construction / destruction when armed; disarms itself
    cudaStream_t st;
    cudaEvent_t stop;
    explicit GatherTimer(cudaStream_t s) : st(s), stop(t_prof_stop) {
        if (t_prof_start && t_prof_stop) cudaEventRecord(t_prof_start, st); else stop = nullptr;
        t_prof_start = t_prof_stop = nullptr;
    }
    ~GatherTimer() { if (stop) cudaEventRecord(stop, st); }
};

static bool fwd77_ok(const rsdet_roi_align_cfg* c) {
    return c->pooled_h == 7 && c->pooled_w == 7 && c->sampling_ratio == 2 && c->channels % 256 == 0;
}

// ---------------------------------------------------------------------------------- backward (fast)
// Same CTA shape and tap lists.  The RoI's (C,7,7) gradient block is copied into shared memory as it
// lies in memory (coalesced 16-byte loads); every merged tap becomes ONE 16-byte vector reduction per
// channel quad (red.global.add.v4.f32) into the channels-last accumulator.
// NHWC_IN: grad_out is (K, PH, PW, C); a thread reads its channel quads of a bin straight from global memory (vector loads
// when grad_out's base is aligned to four elements, scalar loads otherwise) and nothing is staged.
template <int QPT, typename G = float, bool NHWC_IN = false>   // G: grad_out elements (staged as fp32); the accumulators are always fp32
__global__ void __launch_bounds__(kRoiThreads, 4)
roi_align_bwd_kernel(LevelSet L, const int* __restrict__ order, const RoiGeom* __restrict__ geoms, int K,
                     const G* __restrict__ grad_out) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int roi = order ? order[blockIdx.x] : blockIdx.x;
    const int tid = threadIdx.x;
    const int nbins = L.PH * L.PW;
    const int spb = L.sampling_ratio * L.sampling_ratio;
    const int cap = 4 * spb;
    const int C = L.C;
    const int Q = quads_per_chunk(C);
    const int chunk0 = blockIdx.y * Q * 4;
    const int Qc = min(Q, (C - chunk0) / 4);
    int2* s_list = reinterpret_cast<int2*>(smem_raw);
    int* s_cnt = reinterpret_cast<int*>(smem_raw + list_bytes(nbins, cap));
    float* s_stage = reinterpret_cast<float*>(smem_raw + list_bytes(nbins, cap) + ((nbins * 4 + 15) & ~15));

    const RoiGeom g = geoms[roi];
    const int H = L.H[g.level], W = L.W[g.level];
    build_tap_lists(g, L, H, W, s_list, s_cnt, s_stage, C >> 2);

    if constexpr (!NHWC_IN) {
        // stage this chunk's gradient block [c_local][bin] (= memory order)
        const G* __restrict__ src = grad_out + ((size_t)roi * C + chunk0) * nbins;
        const int total = Qc * 4 * nbins;
        if ((((size_t)roi * C + chunk0) * nbins & 3) == 0 && (total & 3) == 0 && (((size_t)grad_out) & (4 * sizeof(G) - 1)) == 0) {
            float4* s4 = reinterpret_cast<float4*>(s_stage);
            for (int e = tid; e < total / 4; e += kRoiThreads) s4[e] = ldcs4(src + (size_t)e * 4);
        } else {
            for (int e = tid; e < total; e += kRoiThreads) s_stage[e] = to_f32(__ldg(src + e));
        }
        __syncthreads();
    }

    const int lanes = QPT == 2 ? 32 : Qc;
    const int groups = kRoiThreads / lanes;
    const int cq = tid % lanes, grp = tid / lanes;
    const int oct = (cq >> 3) & 3;
    float4* __restrict__ gfeat = reinterpret_cast<float4*>(L.grad[g.level] + (size_t)g.batch * H * W * C + chunk0) + cq;
    const bool pow2 = (spb & (spb - 1)) == 0;
    const float count = (float)spb, inv_count = 1.f / count;  // no max(.,1) in backward (:246)
    [[maybe_unused]] const bool g_vec = (((size_t)grad_out) & (4 * sizeof(G) - 1)) == 0;
    if (grp < groups) {
        for (int b = grp; b < nbins; b += groups) {
            float4 top[QPT];
#pragma unroll
            for (int u = 0; u < QPT; u++) {
                const int c0 = (cq + u * 32) * 4;
                if constexpr (NHWC_IN) {
                    const G* const p = grad_out + ((size_t)roi * nbins + b) * C + chunk0 + c0;
                    top[u] = g_vec ? ldcs4(p) : make_float4(to_f32(__ldg(p)), to_f32(__ldg(p + 1)), to_f32(__ldg(p + 2)), to_f32(__ldg(p + 3)));
                    continue;
                }
                float4 r;
                r.x = s_stage[(c0 + ((0 + oct) & 3)) * nbins + b];
                r.y = s_stage[(c0 + ((1 + oct) & 3)) * nbins + b];
                r.z = s_stage[(c0 + ((2 + oct) & 3)) * nbins + b];
                r.w = s_stage[(c0 + ((3 + oct) & 3)) * nbins + b];
                top[u] = unrot4(r, oct);
            }
            const int2* lp = s_list + b * (cap + 1);
            const int cnt = s_cnt[b];
            for (int e = 0; e < cnt; e++) {
                const int2 en = lp[e];
                const float wk = __int_as_float(en.y);
                float* dst = const_cast<float*>(tap_ptr(reinterpret_cast<const float4*>(gfeat), (unsigned)en.x));
#pragma unroll
                for (int u = 0; u < QPT; u++) {
                    // g = top * w / count (:280-283); exact reciprocal when count is a power of two
                    float4 gv;
                    if (pow2) gv = make_float4(top[u].x * wk * inv_count, top[u].y * wk * inv_count, top[u].z * wk * inv_count, top[u].w * wk * inv_count);
                    else gv = make_float4(top[u].x * wk / count, top[u].y * wk / count, top[u].z * wk / count, top[u].w * wk / count);
                    red_add_v4(dst + u * 128, gv);
                }
            }
        }
    }
}

// ---------------------------------------------------------------------------------- generic path
// Any pooled size / adaptive sampling grid / channel count; NCHW or NHWC directly.  One thread per
// output element like the reference, but with the level mapping fused.  Used only when the fast path's
// preconditions (C % 4 == 0, fixed sampling grid, <= kMaxSamples samples) do not hold.
struct GenericMaps {
    const float* feat[RSDET_MAX_LEVELS];   // element type: the kernel's T
    float* grad[RSDET_MAX_LEVELS];
    int channels_last;
};

__device__ __forceinline__ size_t feat_index(int cl, int n, int c, int pix, int C, int HW) {
    return cl ? ((size_t)n * HW + pix) * C + c : ((size_t)n * C + c) * HW + pix;
}

// T: feature elements (forward); O: output elements (forward) or grad_out elements (backward); gradients accumulate in
// fp32 maps (M.grad) in the caller's layout.  NHWC_ROIS: out / grad_out is (K, PH, PW, C), and consecutive threads take
// consecutive channels of it.
template <bool BACKWARD, typename T = float, typename O = float, bool NHWC_ROIS = false>
__global__ void roi_align_generic_kernel(LevelSet L, GenericMaps M, const float* __restrict__ rois, int K,
                                         O* __restrict__ out_or_gradout, int32_t* __restrict__ levels_out) {
    const int nbins = L.PH * L.PW;
    const long long total = (long long)K * L.C * nbins;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        int pw, ph, c, n;
        if constexpr (NHWC_ROIS) {
            c = (int)(idx % L.C);
            const int bin = (int)((idx / L.C) % nbins);
            n = (int)(idx / L.C / nbins);
            ph = bin / L.PW; pw = bin % L.PW;
        } else {
            pw = (int)(idx % L.PW); ph = (int)((idx / L.PW) % L.PH);
            c = (int)((idx / nbins) % L.C); n = (int)(idx / nbins / L.C);
        }
        RoiGeom g = roi_geometry(rois + (size_t)n * 6, L);
        if (!BACKWARD && levels_out && c == 0 && ph == 0 && pw == 0) levels_out[n] = g.level;
        const int H = L.H[g.level], W = L.W[g.level];
        if (!BACKWARD) {
            const float count = (float)max(g.gh * g.gw, 1);
            float acc = 0.f;
            for (int iy = 0; iy < g.gh; iy++)
                for (int ix = 0; ix < g.gw; ix++) {
                    float x, y;
                    sample_xy(g, L.version, ph, pw, iy, ix, x, y);
                    Taps t = make_taps(H, W, y, x);
                    const T* f = reinterpret_cast<const T*>(M.feat[g.level]);
                    float v = t.w[0] * to_f32(f[feat_index(M.channels_last, g.batch, c, t.o[0], L.C, H * W)]) +
                              t.w[1] * to_f32(f[feat_index(M.channels_last, g.batch, c, t.o[1], L.C, H * W)]) +
                              t.w[2] * to_f32(f[feat_index(M.channels_last, g.batch, c, t.o[2], L.C, H * W)]) +
                              t.w[3] * to_f32(f[feat_index(M.channels_last, g.batch, c, t.o[3], L.C, H * W)]);
                    acc += v;
                }
            out_or_gradout[idx] = from_f32<O>(acc / count);
        } else {
            const float count = (float)(g.gh * g.gw);
            const float top = to_f32(out_or_gradout[idx]);
            for (int iy = 0; iy < g.gh; iy++)
                for (int ix = 0; ix < g.gw; ix++) {
                    float x, y;
                    sample_xy(g, L.version, ph, pw, iy, ix, x, y);
                    Taps t = make_taps(H, W, y, x);
                    if (t.w[0] == 0.f && t.w[1] == 0.f && t.w[2] == 0.f && t.w[3] == 0.f) continue;
                    float* gf = M.grad[g.level];
#pragma unroll
                    for (int k = 0; k < 4; k++)
                        atomicAdd(gf + feat_index(M.channels_last, g.batch, c, t.o[k], L.C, H * W), top * t.w[k] / count);
                }
        }
    }
}

static bool fast_path_ok(const rsdet_roi_align_cfg* c) {
    for (int l = 0; l < c->num_levels; l++)  // tap offsets are 32-bit element offsets inside one image
        if ((long long)c->height[l] * c->width[l] * c->channels >= (1ll << 31)) return false;
    return c->channels % 4 == 0 && c->sampling_ratio > 0 &&
           c->pooled_h * c->pooled_w * c->sampling_ratio * c->sampling_ratio <= kMaxSamples;
}

// The fast kernels read (forward) or accumulate into (backward) a channels-last caller's maps with 4-channel vector
// accesses from each level's base pointer (16 bytes for fp32, 8 for half maps); a base that is not aligned to that goes
// to the scalar generic kernel, which addresses NHWC maps directly.  NCHW maps are only read by the transposes, which
// check alignment themselves.
// the layout bits of cfg.channels_last (include/rsdet.h)
static bool nhwc_maps(const rsdet_roi_align_cfg* c) { return (c->channels_last & RSDET_ROI_NHWC_MAPS) != 0; }
static bool nhwc_rois(const rsdet_roi_align_cfg* c) { return (c->channels_last & RSDET_ROI_NHWC_ROIS) != 0; }

template <typename P>
static bool nhwc_bases_aligned(const rsdet_roi_align_cfg* c, P const* maps, size_t align) {
    if (!nhwc_maps(c)) return true;
    for (int l = 0; l < c->num_levels; l++)
        if (((size_t)maps[l]) & (align - 1)) return false;
    return true;
}

static int check_cfg(const rsdet_roi_align_cfg* c) {
    if (!c) return RSDET_EINVAL;
    if (c->num_levels < 1 || c->num_levels > RSDET_MAX_LEVELS || c->batch < 1 || c->channels < 1) return RSDET_EINVAL;
    if (c->pooled_h < 1 || c->pooled_w < 1 || (c->version != 0 && c->version != 1)) return RSDET_EINVAL;
    if (c->channels_last & ~(RSDET_ROI_NHWC_MAPS | RSDET_ROI_NHWC_ROIS)) return RSDET_EINVAL;
    for (int l = 0; l < c->num_levels; l++)
        if (c->height[l] < 1 || c->width[l] < 1) return RSDET_EINVAL;
    return RSDET_OK;
}

static LevelSet make_levels(const rsdet_roi_align_cfg* c) {
    LevelSet L;
    L.num_levels = c->num_levels; L.batch = c->batch; L.C = c->channels;
    L.PH = c->pooled_h; L.PW = c->pooled_w; L.sampling_ratio = c->sampling_ratio; L.version = c->version;
    L.extend_w = c->extend_w; L.extend_h = c->extend_h; L.finest_scale = c->finest_scale;
    for (int l = 0; l < RSDET_MAX_LEVELS; l++) {
        L.feat[l] = nullptr; L.grad[l] = nullptr;
        L.H[l] = l < c->num_levels ? c->height[l] : 1;
        L.W[l] = l < c->num_levels ? c->width[l] : 1;
        L.scale[l] = l < c->num_levels ? c->spatial_scale[l] : 1.f;
    }
    return L;
}

static size_t fwd_smem_bytes(const rsdet_roi_align_cfg* c) {
    size_t nbins = (size_t)c->pooled_h * c->pooled_w;
    size_t ntaps = nbins * 4 * c->sampling_ratio * c->sampling_ratio;
    size_t stage = sizeof(float) * 4 * nbins * quads_per_chunk(c->channels), tmp = 12 * (ntaps + nbins);
    return list_bytes(nbins, ntaps / nbins) + ((nbins * 4 + 15) & ~(size_t)15) + (stage > tmp ? stage : tmp);
}

// roi_align_generic_kernel over the caller's maps (forward: feature maps, backward: fp32 gradient maps), one thread per
// output element, at most 16 CTAs per SM
template <bool BACKWARD, typename T, typename O, bool NHWC_ROIS, typename P>
static void launch_generic(const rsdet_roi_align_cfg* cfg, const LevelSet& L, P const* maps, const float* rois, int K,
                           O* out_or_gradout, int32_t* levels_out, cudaStream_t st) {
    GenericMaps M;
    M.channels_last = nhwc_maps(cfg);
    for (int l = 0; l < RSDET_MAX_LEVELS; l++) {
        M.feat[l] = nullptr;
        M.grad[l] = nullptr;
        if (l >= cfg->num_levels) continue;
        if constexpr (BACKWARD) M.grad[l] = maps[l];
        else M.feat[l] = reinterpret_cast<const float*>(maps[l]);
    }
    const long long blocks = ceil_div_ll((long long)K * cfg->channels * cfg->pooled_h * cfg->pooled_w, 256);
    roi_align_generic_kernel<BACKWARD, T, O, NHWC_ROIS><<<(int)(blocks < kNumSMs * 16 ? blocks : kNumSMs * 16), 256, 0, st>>>(
        L, M, rois, K, out_or_gradout, levels_out);
    count_launch();
}

}  // namespace rsdet

using namespace rsdet;

static bool dtype_ok(int dt) { return dt == RSDET_DTYPE_F32 || dt == RSDET_DTYPE_F16 || dt == RSDET_DTYPE_BF16; }

// elem: bytes of one feature-map element
static size_t roi_workspace_bytes(const rsdet_roi_align_cfg* cfg, int num_rois, int backward, size_t elem) {
    // order, geometry (+ forward: the work counter of the persistent kernel)
    size_t b = ws_bytes<int>(num_rois > 0 ? num_rois : 1) + ws_bytes<RoiGeom>(num_rois > 0 ? num_rois : 1) +
               (backward ? 0 : ws_bytes<unsigned>(1));
    if (backward && elem != sizeof(float)) {    // half gradient maps: fp32 accumulators on every path
        for (int l = 0; l < cfg->num_levels; l++)
            b += ws_bytes<float>((size_t)cfg->batch * cfg->channels * cfg->height[l] * cfg->width[l]);
        return b + 256;
    }
    if (nhwc_maps(cfg) || !fast_path_ok(cfg)) return b + 256;
    for (int l = 0; l < cfg->num_levels; l++)      // NHWC copy of the pyramid (forward) / fp32 NHWC accumulators (backward)
        b += align256(elem * cfg->batch * cfg->channels * cfg->height[l] * cfg->width[l]);
    return b + 256;
}

extern "C" size_t rsdet_roi_align_rotated_workspace_bytes_typed(const rsdet_roi_align_cfg* cfg, int num_rois, int backward,
                                                                 int feat_dtype) {
    if (!dtype_ok(feat_dtype) || check_cfg(cfg) != RSDET_OK) return 0;
    return roi_workspace_bytes(cfg, num_rois, backward, feat_dtype == RSDET_DTYPE_F32 ? sizeof(float) : 2);
}

extern "C" size_t rsdet_roi_align_rotated_workspace_bytes(const rsdet_roi_align_cfg* cfg, int num_rois, int backward) {
    return rsdet_roi_align_rotated_workspace_bytes_typed(cfg, num_rois, backward, RSDET_DTYPE_F32);
}

// T: feature elements, O: output elements (float or T), NHWC_OUT: out is (K, PH, PW, C).  Arguments are checked by the caller.
template <typename T, typename O, bool NHWC_OUT>
static int forward_impl(const rsdet_roi_align_cfg* cfg, const T* const* feats_host, const float* rois, int num_rois, O* out,
                        int32_t* levels_out, void* workspace, size_t workspace_bytes, cudaStream_t st) {
    int rc = RSDET_OK;
    LevelSet L = make_levels(cfg);
    if (!fast_path_ok(cfg) || !nhwc_bases_aligned(cfg, feats_host, 4 * sizeof(T))) {
        launch_generic<false, T, O, NHWC_OUT>(cfg, L, feats_host, rois, num_rois, out, levels_out, st);
        return cuda_status();
    }
    if (workspace_bytes < roi_workspace_bytes(cfg, num_rois, 0, sizeof(T))) return RSDET_EWORKSPACE;
    Workspace ws(workspace, workspace_bytes);
    int* order_ws = ws.take<int>(num_rois);
    RoiGeom* geoms = ws.take<RoiGeom>(num_rois);
    unsigned* counter = ws.take<unsigned>(1);
    if (nhwc_maps(cfg)) {
        for (int l = 0; l < cfg->num_levels; l++) L.feat[l] = reinterpret_cast<const float*>(feats_host[l]);
    } else {
        for (int l = 0; l < cfg->num_levels; l++)
            L.feat[l] = reinterpret_cast<const float*>(ws.take<T>((size_t)cfg->batch * cfg->channels * cfg->height[l] * cfg->width[l]));
        if (!ws.ok()) return RSDET_EWORKSPACE;
    }
    // locality order (needs the int[K] slot at the start of the workspace; skipped for tiny calls) and geometry records:
    // for NCHW callers with an order of at most kPrepMaxRois RoIs, order block and geometry blocks ride with the
    // pyramid transpose; every other call launches roi_prep_kernel (then NCHW callers the plain transpose)
    int* order = num_rois >= 256 && order_ws ? order_ws : nullptr;
    const bool ride = !nhwc_maps(cfg) && order && num_rois <= kPrepMaxRois;
    if (!ride) {
        roi_prep_kernel<<<(order ? 1 : 0) + ceil_div(num_rois, 1024), 1024, 0, st>>>(L, rois, num_rois, order, geoms, levels_out, counter);
        count_launch();
    }
    if (!nhwc_maps(cfg)) {
        PrepArgs prep = {&L, rois, num_rois, order, geoms, levels_out, counter};
        T* dst[RSDET_MAX_LEVELS];
        for (int l = 0; l < cfg->num_levels; l++) dst[l] = reinterpret_cast<T*>(const_cast<float*>(L.feat[l]));
        rc = launch_transpose(true, feats_host, dst, cfg->height, cfg->width, cfg->num_levels, cfg->batch, cfg->channels, st,
                              ride ? &prep : nullptr);
        if (rc != RSDET_OK) return rc;
    }
    // the persistent 7x7 kernel needs a 16-byte aligned output for its bulk stores (an NHWC output, stored from registers,
    // four-element alignment); everything else runs roi_align_fwd_kernel
    const bool persistent = fwd77_ok(cfg) && (((size_t)out) & (NHWC_OUT ? 4 * sizeof(O) - 1 : 15)) == 0;
    GatherTimer gather_timer(st);
    if (persistent) {
        const int chunks = cfg->channels / 256;
        const long long items = (long long)num_rois * chunks, ctas = kNumSMs * kFwd77pCtasPerSm;
        const size_t smp = kStage77pOffset + (NHWC_OUT ? 0 : sizeof(float) * 49 * 256);
        set_dyn_smem((const void*)roi_align_fwd77p_kernel<T, O, NHWC_OUT>, smp);
        roi_align_fwd77p_kernel<T, O, NHWC_OUT><<<(int)(items < ctas ? items : ctas), 32 * kFwd77pWarps, smp, st>>>(
            L, order, geoms, num_rois, chunks, out, counter);
        count_launch();
        return cuda_status();
    }
    const size_t smem = fwd_smem_bytes(cfg);
    const int Q = quads_per_chunk(cfg->channels);
    dim3 grid(num_rois, ceil_div(cfg->channels / 4, Q));
    if (cfg->channels % 256 == 0) {
        set_dyn_smem((const void*)roi_align_fwd_kernel<2, T, O, NHWC_OUT>, smem);
        roi_align_fwd_kernel<2, T, O, NHWC_OUT><<<grid, kRoiThreads, smem, st>>>(L, order, geoms, num_rois, out);
    } else {
        set_dyn_smem((const void*)roi_align_fwd_kernel<1, T, O, NHWC_OUT>, smem);
        roi_align_fwd_kernel<1, T, O, NHWC_OUT><<<grid, kRoiThreads, smem, st>>>(L, order, geoms, num_rois, out);
    }
    count_launch();
    return cuda_status();
}

extern "C" int rsdet_roi_align_rotated_forward_typed(const rsdet_roi_align_cfg* cfg, int feat_dtype, const void* const* feats_host,
                                                     const float* rois, int num_rois, int out_dtype, void* out,
                                                     int32_t* levels_out, void* workspace, size_t workspace_bytes, void* stream) {
    if (!dtype_ok(feat_dtype) || (out_dtype != RSDET_DTYPE_F32 && out_dtype != feat_dtype)) return RSDET_EINVAL;
    int rc = check_cfg(cfg);
    if (rc != RSDET_OK) return rc;
    if (num_rois < 0) return RSDET_EINVAL;
    if (num_rois == 0) return RSDET_OK;
    if (!feats_host || !rois || !out) return RSDET_EINVAL;
    for (int l = 0; l < cfg->num_levels; l++)
        if (!feats_host[l]) return RSDET_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    const bool half_out = out_dtype != RSDET_DTYPE_F32;
#define RSDET_FWD(T_, O_)                                                                                                      \
    (nhwc_rois(cfg) ? forward_impl<T_, O_, true>(cfg, reinterpret_cast<const T_* const*>(feats_host), rois, num_rois,             \
                                                 static_cast<O_*>(out), levels_out, workspace, workspace_bytes, st)              \
                    : forward_impl<T_, O_, false>(cfg, reinterpret_cast<const T_* const*>(feats_host), rois, num_rois,            \
                                                  static_cast<O_*>(out), levels_out, workspace, workspace_bytes, st))
    if (feat_dtype == RSDET_DTYPE_F16) return half_out ? RSDET_FWD(__half, __half) : RSDET_FWD(__half, float);
    if (feat_dtype == RSDET_DTYPE_BF16) return half_out ? RSDET_FWD(__nv_bfloat16, __nv_bfloat16) : RSDET_FWD(__nv_bfloat16, float);
    return RSDET_FWD(float, float);
#undef RSDET_FWD
}

extern "C" int rsdet_roi_align_rotated_forward(const rsdet_roi_align_cfg* cfg, const float* const* feats_host, const float* rois,
                                               int num_rois, float* out, int32_t* levels_out, void* workspace,
                                               size_t workspace_bytes, void* stream) {
    return rsdet_roi_align_rotated_forward_typed(cfg, RSDET_DTYPE_F32, reinterpret_cast<const void* const*>(feats_host), rois,
                                                 num_rois, RSDET_DTYPE_F32, out, levels_out, workspace, workspace_bytes, stream);
}

// the fp32 accumulators of half gradient maps -> the caller's maps, same layout (see backward_impl)
template <typename D>
static int launch_convert(const rsdet_roi_align_cfg* cfg, float* const* acc, D* const* dst, cudaStream_t st) {
    ConvertJob job;
    size_t most = 0;
    for (int l = 0; l < cfg->num_levels; l++) {
        job.src[l] = acc[l]; job.dst[l] = dst[l];
        job.n[l] = (size_t)cfg->batch * cfg->channels * cfg->height[l] * cfg->width[l];
        most = job.n[l] > most ? job.n[l] : most;
    }
    const long long blocks = ceil_div_ll(ceil_div_ll((long long)most, 4), 256);
    convert_maps_kernel<D><<<dim3((unsigned)(blocks < kNumSMs * 16 ? blocks : kNumSMs * 16), cfg->num_levels), 256, 0, st>>>(job);
    count_launch();
    return cuda_status();
}

// G: grad_out elements (float or T), T: gradient-map elements.  fp32 maps: channels-last maps and generic-kernel calls
// accumulate straight into the caller's maps, NCHW maps through fp32 NHWC accumulators and the NHWC->NCHW transpose.
// Half maps always accumulate into fp32 workspace maps -- channels-last for the fast kernels, the caller's layout for the
// generic kernel -- and ONE pass writes the caller's maps from them, rounding to nearest-even: the NHWC->NCHW transpose,
// or a conversion that keeps the layout.  The fast kernels then never touch the caller's maps, so their alignment does
// not matter.
template <typename G, typename T, bool NHWC_IN>   // NHWC_IN: grad_out is (K, PH, PW, C)
static int backward_impl(const rsdet_roi_align_cfg* cfg, const G* grad_out, const float* rois, int num_rois, T* const* grad_feats_host,
                         void* workspace, size_t workspace_bytes, cudaStream_t st) {
    int rc = RSDET_OK;
    LevelSet L = make_levels(cfg);
    const bool fast = fast_path_ok(cfg) && (!kIsF32<T> || nhwc_bases_aligned(cfg, grad_feats_host, 16));
    const bool direct = kIsF32<T> && (nhwc_maps(cfg) || !fast);  // accumulate straight into the caller's buffers
    float* acc[RSDET_MAX_LEVELS];
    if (workspace_bytes < roi_workspace_bytes(cfg, num_rois, 1, sizeof(T))) return RSDET_EWORKSPACE;
    Workspace ws(workspace, workspace_bytes);
    int* order_ws = ws.take<int>(num_rois > 0 ? num_rois : 1);
    RoiGeom* geoms = ws.take<RoiGeom>(num_rois > 0 ? num_rois : 1);
    if (direct) {
        for (int l = 0; l < cfg->num_levels; l++) acc[l] = reinterpret_cast<float*>(grad_feats_host[l]);
    } else {
        for (int l = 0; l < cfg->num_levels; l++)
            acc[l] = ws.take<float>((size_t)cfg->batch * cfg->channels * cfg->height[l] * cfg->width[l]);
        if (!ws.ok()) return RSDET_EWORKSPACE;
    }
    for (int l = 0; l < cfg->num_levels; l++) {
        cudaMemsetAsync(acc[l], 0, sizeof(float) * (size_t)cfg->batch * cfg->channels * cfg->height[l] * cfg->width[l], st);
        L.grad[l] = acc[l];
    }
    count_launch(cfg->num_levels);
    if (num_rois > 0) {
        if (!grad_out || !rois) return RSDET_EINVAL;
        if (!fast) {
            launch_generic<true, float, G, NHWC_IN>(cfg, L, acc, rois, num_rois, const_cast<G*>(grad_out), nullptr, st);
        } else {
            size_t smem = fwd_smem_bytes(cfg);
            set_dyn_smem((const void*)roi_align_bwd_kernel<1, G, NHWC_IN>, smem);
            set_dyn_smem((const void*)roi_align_bwd_kernel<2, G, NHWC_IN>, smem);
            int* order = num_rois >= 256 ? order_ws : nullptr;
            roi_prep_kernel<<<(order ? 1 : 0) + ceil_div(num_rois, 1024), 1024, 0, st>>>(L, rois, num_rois, order, geoms, nullptr, nullptr);
            int Q = quads_per_chunk(cfg->channels);
            dim3 grid(num_rois, ceil_div(cfg->channels / 4, Q));
            if (cfg->channels % 256 == 0) roi_align_bwd_kernel<2, G, NHWC_IN><<<grid, kRoiThreads, smem, st>>>(L, order, geoms, num_rois, grad_out);
            else roi_align_bwd_kernel<1, G, NHWC_IN><<<grid, kRoiThreads, smem, st>>>(L, order, geoms, num_rois, grad_out);
            count_launch(2);
        }
    }
    if (!direct) {
        if constexpr (!kIsF32<T>) {
            if (!fast || nhwc_maps(cfg)) return launch_convert(cfg, acc, grad_feats_host, st);
        }
        rc = launch_transpose(false, acc, grad_feats_host, cfg->height, cfg->width, cfg->num_levels, cfg->batch, cfg->channels, st);
        if (rc != RSDET_OK) return rc;
    }
    return cuda_status();
}

extern "C" int rsdet_roi_align_rotated_backward_typed(const rsdet_roi_align_cfg* cfg, int grad_out_dtype, const void* grad_out,
                                                      const float* rois, int num_rois, int feat_dtype, void* const* grad_feats_host,
                                                      void* workspace, size_t workspace_bytes, void* stream) {
    if (!dtype_ok(feat_dtype) || (grad_out_dtype != RSDET_DTYPE_F32 && grad_out_dtype != feat_dtype)) return RSDET_EINVAL;
    int rc = check_cfg(cfg);
    if (rc != RSDET_OK) return rc;
    if (num_rois < 0 || !grad_feats_host) return RSDET_EINVAL;
    for (int l = 0; l < cfg->num_levels; l++)
        if (!grad_feats_host[l]) return RSDET_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    const bool half_g = grad_out_dtype != RSDET_DTYPE_F32;
#define RSDET_BWD(G_, T_)                                                                                                      \
    (nhwc_rois(cfg) ? backward_impl<G_, T_, true>(cfg, static_cast<const G_*>(grad_out), rois, num_rois,                         \
                                                  reinterpret_cast<T_* const*>(grad_feats_host), workspace, workspace_bytes, st) \
                    : backward_impl<G_, T_, false>(cfg, static_cast<const G_*>(grad_out), rois, num_rois,                        \
                                                   reinterpret_cast<T_* const*>(grad_feats_host), workspace, workspace_bytes, st))
    if (feat_dtype == RSDET_DTYPE_F16) return half_g ? RSDET_BWD(__half, __half) : RSDET_BWD(float, __half);
    if (feat_dtype == RSDET_DTYPE_BF16) return half_g ? RSDET_BWD(__nv_bfloat16, __nv_bfloat16) : RSDET_BWD(float, __nv_bfloat16);
    return RSDET_BWD(float, float);
#undef RSDET_BWD
}

extern "C" int rsdet_roi_align_rotated_backward(const rsdet_roi_align_cfg* cfg, const float* grad_out, const float* rois,
                                                int num_rois, float* const* grad_feats_host, void* workspace,
                                                size_t workspace_bytes, void* stream) {
    return rsdet_roi_align_rotated_backward_typed(cfg, RSDET_DTYPE_F32, grad_out, rois, num_rois, RSDET_DTYPE_F32,
                                                  reinterpret_cast<void* const*>(grad_feats_host), workspace, workspace_bytes, stream);
}

// ---------------------------------------------------------------------------------- backward (deterministic)
// The reference (roi_align_rotated_v1.py:193-298) accumulates every gradient element as one sequential fp32 sum: for a
// fixed (level, image, channel, pixel) the terms (top * w) / count arrive in the order RoI, bin row, bin column, sample
// row, sample column, tap (lt, rt, lb, rb).  Entry e = ((roi * nbins + bin) * spb + sample) * 4 + tap enumerates every
// term in exactly that order, so
//   1. roi_bwd_det_entries_kernel: one thread per (RoI, bin, sample) writes the sample's four entries: a 32-bit pixel
//      key over (level, image, y, x) (all ones when the sample is out of range or the weight is 0: such terms add
//      nothing to a sum that starts at +0), the entry index and the weight;
//   2. a stable LSD radix sort of (key, entry index) over the key's bits groups the entries by pixel and keeps the
//      reference's order inside each pixel;
//   3. grad_out (K, C, bins) is copied bin-major to (K, bins, C), so that a term reads C contiguous values (a (K, bins, C)
//      grad_out is read in place when fp32 and widened to fp32 when half);
//   4. roi_bwd_det_gather_kernel: one warp per touched pixel, lanes over channels, adds the pixel's terms in sorted
//      order with separately rounded multiply, divide and add, and stores the C sums once (plain stores, no atomics).
// Untouched pixels keep the zero fill that precedes step 4; NCHW and fp32-accumulated half maps reuse the output passes
// of the atomic backward.  Results do not depend on the stream, the launch configuration, the layout or the alignment.
namespace rsdet {

constexpr long long kDetMaxEntries = 1ll << 28;   // K * PH * PW * sr^2 * 4 (include/rsdet.h)
constexpr int kDetChannelsPerLane = 8;            // a warp covers 256 channels per walk of a pixel's entries

// radix_sort.cu: stable sort of (key, value) pairs on the key's low `key_bits` bits (CUB, in a unit of its own)
int sort_pairs_u32(void* tmp, size_t* tmp_bytes, uint32_t* key_a, uint32_t* key_b, int* val_a, int* val_b, int n, int key_bits,
                   bool* in_b, cudaStream_t st);

struct DetJob {
    LevelSet L;                                   // geometry only (feat / grad unused)
    unsigned pix_base[RSDET_MAX_LEVELS + 1];      // key of (level l, image 0, pixel 0): prefix of batch * H * W
    void* out[RSDET_MAX_LEVELS];                  // channels-last destinations (fp32 accumulators or the caller's maps)
    unsigned sentinel;                            // key of a term that is dropped; sorts after every pixel
};

__global__ void __launch_bounds__(256) roi_bwd_det_entries_kernel(DetJob J, const float* __restrict__ rois, int K,
                                                                  uint32_t* __restrict__ keys, int* __restrict__ idx,
                                                                  float* __restrict__ wts) {
    const LevelSet& L = J.L;
    const int spb = L.sampling_ratio * L.sampling_ratio, per_roi = L.PH * L.PW * spb;
    const long long total = (long long)K * per_roi;
    for (long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x; s < total; s += (long long)gridDim.x * blockDim.x) {
        const int roi = (int)(s / per_roi), r = (int)(s % per_roi);
        const int bin = r / spb, smp = r % spb;
        const RoiGeom g = roi_geometry(rois + (size_t)roi * 6, L);
        float x, y;
        sample_xy(g, L.version, bin / L.PW, bin % L.PW, smp / L.sampling_ratio, smp % L.sampling_ratio, x, y);
        const int H = L.H[g.level], W = L.W[g.level];
        const Taps t = make_taps(H, W, y, x);
        const bool image_ok = g.batch >= 0 && g.batch < L.batch;
        const unsigned base = J.pix_base[g.level] + (unsigned)g.batch * (unsigned)(H * W);
        uint4 k, e;
        k.x = image_ok && t.w[0] != 0.f ? base + t.o[0] : J.sentinel;
        k.y = image_ok && t.w[1] != 0.f ? base + t.o[1] : J.sentinel;
        k.z = image_ok && t.w[2] != 0.f ? base + t.o[2] : J.sentinel;
        k.w = image_ok && t.w[3] != 0.f ? base + t.o[3] : J.sentinel;
        const unsigned e0 = (unsigned)(4 * s);
        e.x = e0; e.y = e0 + 1; e.z = e0 + 2; e.w = e0 + 3;
        reinterpret_cast<uint4*>(keys)[s] = k;
        reinterpret_cast<uint4*>(idx)[s] = e;
        reinterpret_cast<float4*>(wts)[s] = make_float4(t.w[0], t.w[1], t.w[2], t.w[3]);
    }
}

// (p / count) rounded once to fp32, without the subroutine call of the fp32 division (whose calling convention costs the
// gather kernel spills): the fp64 product with rd = 1/count rounded, one exact-remainder correction (fp64 fma) that
// makes it p / count rounded to fp64, then the rounding to fp32.  fp64 carries more than 2 * 24 + 2 bits, so rounding
// a quotient twice equals rounding it once; p is finite here and p / count stays far inside the fp64 range.
__device__ __forceinline__ float div_by_count(float p, double count, double rcp) {
    const double q = __dmul_rn((double)p, rcp);
    const double r = __fma_rn(-q, count, (double)p);
    return p == 0.f ? p : __double2float_rn(__fma_rn(r, rcp, q));
}

// top: (K, bins, C) fp32.  Warp w scans the sorted keys in chunks of 32 positions (grid-stride) and takes every run that
// starts in its chunk; a run is walked in batches of 32 entries whose (entry, weight) pairs the lanes load together.
template <typename O, bool POW2>
__global__ void __launch_bounds__(256) roi_bwd_det_gather_kernel(DetJob J, const uint32_t* __restrict__ keys,
                                                                 const int* __restrict__ idx, const float* __restrict__ wts,
                                                                 const float* __restrict__ top, int E) {
    const int lane = threadIdx.x & 31;
    const int warp = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), nwarps = (int)((gridDim.x * blockDim.x) >> 5);
    const int C = J.L.C, spb = J.L.sampling_ratio * J.L.sampling_ratio;
    const float inv_count = 1.f / (float)spb;   // POW2: x * 2^-k is x / 2^k rounded once, the same bits as the division
    const double count_d = (double)spb, rcp_d = 1.0 / count_d;
    for (long long c0 = 32ll * warp; c0 < E; c0 += 32ll * nwarps) {
        const int p = (int)c0 + lane;
        const unsigned k = p < E ? __ldg(keys + p) : J.sentinel;
        if (__shfl_sync(~0u, k, 0) == J.sentinel) break;          // sorted: only dropped terms from here on
        const unsigned prev = p > 0 && p < E ? __ldg(keys + p - 1) : ~k;
        unsigned starts = __ballot_sync(~0u, k != J.sentinel && prev != k);
        while (starts) {
            const int s = (int)c0 + __ffs(starts) - 1;
            const unsigned key = __shfl_sync(~0u, k, __ffs(starts) - 1);
            starts &= starts - 1;
            unsigned base = J.pix_base[0];     // the key's level, with constant indices only (no local copy of J)
            void* out = J.out[0];
#pragma unroll
            for (int l = 1; l < RSDET_MAX_LEVELS; l++)
                if (l < J.L.num_levels && key >= J.pix_base[l]) { base = J.pix_base[l]; out = J.out[l]; }
            O* __restrict__ dst = static_cast<O*>(out) + (size_t)(key - base) * C;
            for (int cb = 0; cb < C; cb += 32 * kDetChannelsPerLane) {
                float acc[kDetChannelsPerLane];
#pragma unroll
                for (int u = 0; u < kDetChannelsPerLane; u++) acc[u] = 0.f;
                for (int j0 = s;; j0 += 32) {
                    const int j = j0 + lane;
                    const bool in = j < E && __ldg(keys + j) == key;
                    const unsigned m = __ballot_sync(~0u, in);     // the run is a prefix of the batch
                    int rb = 0;
                    float w = 0.f;
                    if (in) {
                        const int e = __ldg(idx + j);
                        rb = e / (4 * spb);                         // roi * bins + bin
                        w = __ldg(wts + e);
                    }
                    const int n = __popc(m);
#pragma unroll 4
                    for (int t = 0; t < n; t++) {
                        const int rbt = __shfl_sync(~0u, rb, t);
                        const float wt = __shfl_sync(~0u, w, t);
                        const float* __restrict__ src = top + (size_t)rbt * C + cb + lane;
#pragma unroll
                        for (int u = 0; u < kDetChannelsPerLane; u++) {
                            if (cb + lane + 32 * u < C) {
                                const float pr = __fmul_rn(__ldg(src + 32 * u), wt);
                                acc[u] = __fadd_rn(acc[u], POW2 ? __fmul_rn(pr, inv_count) : div_by_count(pr, count_d, rcp_d));
                            }
                        }
                    }
                    if (n < 32) break;
                }
#pragma unroll
                for (int u = 0; u < kDetChannelsPerLane; u++)
                    if (cb + lane + 32 * u < C) dst[cb + lane + 32 * u] = from_f32<O>(acc[u]);
            }
        }
    }
}

// a (K, PH, PW, C) half grad_out -> the fp32 bin-major array the gather reads (exact conversion, same layout)
template <typename G>
__global__ void __launch_bounds__(256) widen_kernel(const G* __restrict__ src, float* __restrict__ dst, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        dst[i] = to_f32(__ldg(src + i));
}

// Sizes of one call; false when the call is outside the contract (adaptive grid, entry or pixel count too large).
struct DetPlan {
    long long entries;      // K * bins * sr^2 * 4
    long long pixels;       // batch * sum of H * W: the key space
    int key_bits;
    size_t cub_bytes;       // bound on the radix sort's temporary storage
};
static bool det_plan(const rsdet_roi_align_cfg* c, int num_rois, DetPlan* p) {
    if (c->sampling_ratio <= 0 || num_rois < 0) return false;
    const long long bins = (long long)c->pooled_h * c->pooled_w;
    if (c->sampling_ratio > 1 << 14 || bins > kDetMaxEntries) return false;       // no overflow below
    const long long per_roi = bins * c->sampling_ratio * c->sampling_ratio * 4;
    if (per_roi > kDetMaxEntries) return false;
    p->entries = per_roi * num_rois;
    if (p->entries > kDetMaxEntries) return false;
    // tiles of the bin-major copy of grad_out (one launch, int tile indices)
    if ((long long)num_rois * ((bins + 63) / 64) * ((c->channels + 63) / 64) > 0x7fffffffll) return false;
    p->pixels = 0;
    for (int l = 0; l < c->num_levels; l++) p->pixels += (long long)c->batch * c->height[l] * c->width[l];
    if (p->pixels > 0xfffffffell) return false;     // every key below the all-ones sentinel
    p->key_bits = 1;
    while (p->key_bits < 32 && (1ll << p->key_bits) <= p->pixels) p->key_bits++;
    // onesweep: a few KB of bins and counters plus one 256-digit lookback row per tile of thousands of items
    p->cub_bytes = ((size_t)1 << 20) + 2 * (size_t)p->entries;
    return true;
}

static size_t det_workspace_bytes(const rsdet_roi_align_cfg* c, int num_rois, const DetPlan& p, bool f32) {
    const size_t E = (size_t)(p.entries > 0 ? p.entries : 1);
    size_t b = 4 * ws_bytes<uint32_t>(E) + ws_bytes<float>(E);        // keys x2, entry indices x2, weights
    // the fp32 bin-major copy of grad_out.  An NHWC fp32 grad_out is that array already; the query does not know the
    // grad_out dtype, so it reserves the copy unless the maps -- and hence grad_out -- are fp32.
    if (!nhwc_rois(c) || !f32)
        b += ws_bytes<float>((size_t)(num_rois > 0 ? num_rois : 1) * c->pooled_h * c->pooled_w * c->channels);
    if (!nhwc_maps(c))                                                 // fp32 NHWC accumulators
        for (int l = 0; l < c->num_levels; l++) b += ws_bytes<float>((size_t)c->batch * c->channels * c->height[l] * c->width[l]);
    return b + align256(p.cub_bytes) + 256;
}

template <typename G, typename T>
static int backward_det_impl(const rsdet_roi_align_cfg* cfg, const DetPlan& plan, const G* grad_out, const float* rois,
                             int num_rois, T* const* grad_feats_host, void* workspace, size_t workspace_bytes, cudaStream_t st) {
    auto map_bytes = [&](int l) { return sizeof(T) * (size_t)cfg->batch * cfg->channels * cfg->height[l] * cfg->width[l]; };
    if (num_rois == 0) {     // nothing to sum: zero maps
        for (int l = 0; l < cfg->num_levels; l++) cudaMemsetAsync(grad_feats_host[l], 0, map_bytes(l), st);
        count_launch(cfg->num_levels);
        return cuda_status();
    }
    if (workspace_bytes < det_workspace_bytes(cfg, num_rois, plan, kIsF32<T>)) return RSDET_EWORKSPACE;
    const int E = (int)plan.entries, nbins = cfg->pooled_h * cfg->pooled_w;
    Workspace ws(workspace, workspace_bytes);
    uint32_t* keyA = ws.take<uint32_t>(E);
    uint32_t* keyB = ws.take<uint32_t>(E);
    int* idxA = ws.take<int>(E);
    int* idxB = ws.take<int>(E);
    float* wts = ws.take<float>(E);
    // an fp32 (K, PH, PW, C) grad_out already is the bin-major array the gather reads
    const float* top = nullptr;
    float* top_ws = nullptr;
    if constexpr (kIsF32<G>) { if (nhwc_rois(cfg)) top = grad_out; }
    if (!top) top = top_ws = ws.take<float>((size_t)num_rois * nbins * cfg->channels);
    float* acc[RSDET_MAX_LEVELS];
    if (!nhwc_maps(cfg))
        for (int l = 0; l < cfg->num_levels; l++) acc[l] = ws.take<float>((size_t)cfg->batch * cfg->channels * cfg->height[l] * cfg->width[l]);
    void* cub_tmp = ws.take<char>(plan.cub_bytes);
    if (!ws.ok()) return RSDET_EWORKSPACE;
    size_t need = 0;
    int rc = sort_pairs_u32(nullptr, &need, keyA, keyB, idxA, idxB, E, plan.key_bits, nullptr, st);
    if (rc != RSDET_OK) return rc;
    if (need > plan.cub_bytes) return RSDET_EWORKSPACE;

    DetJob J;
    J.L = make_levels(cfg);
    J.sentinel = plan.key_bits == 32 ? 0xffffffffu : (1u << plan.key_bits) - 1;
    unsigned base = 0;
    for (int l = 0; l <= RSDET_MAX_LEVELS; l++) {
        J.pix_base[l] = base;
        if (l < cfg->num_levels) base += (unsigned)((size_t)cfg->batch * cfg->height[l] * cfg->width[l]);
        if (l < RSDET_MAX_LEVELS) J.out[l] = l < cfg->num_levels ? (nhwc_maps(cfg) ? (void*)grad_feats_host[l] : (void*)acc[l]) : nullptr;
    }
    // zero fill of whatever the gather writes into; an NCHW caller's maps are written whole by the transpose
    for (int l = 0; l < cfg->num_levels; l++) {
        if (nhwc_maps(cfg)) cudaMemsetAsync(grad_feats_host[l], 0, map_bytes(l), st);
        else cudaMemsetAsync(acc[l], 0, sizeof(float) * (size_t)cfg->batch * cfg->channels * cfg->height[l] * cfg->width[l], st);
    }
    count_launch(cfg->num_levels);
    const long long samples = plan.entries / 4;
    roi_bwd_det_entries_kernel<<<(unsigned)(ceil_div_ll(samples, 256) < kNumSMs * 16 ? ceil_div_ll(samples, 256) : kNumSMs * 16),
                                 256, 0, st>>>(J, rois, num_rois, keyA, idxA, wts);
    count_launch();
    if (nhwc_rois(cfg) && top_ws) {
        if constexpr (!kIsF32<G>) {   // half (K, PH, PW, C) grad_out: already bin-major, widened exactly to fp32
            const size_t n = (size_t)num_rois * nbins * cfg->channels;
            const long long blocks = ceil_div_ll((long long)n, 256);
            widen_kernel<G><<<(unsigned)(blocks < kNumSMs * 16 ? blocks : kNumSMs * 16), 256, 0, st>>>(grad_out, top_ws, n);
            count_launch();
        }
    } else if (!nhwc_rois(cfg)) {
        // bin-major copy of grad_out: the NCHW -> NHWC transpose with K images of PH x PW pixels
        TransposeJob tj;
        tj.num_levels = 1; tj.N = num_rois; tj.C = cfg->channels;
        tj.src[0] = grad_out; tj.dst[0] = top_ws; tj.HW[0] = nbins;
        tj.tile_begin[0] = 0;
        tj.tile_begin[1] = num_rois * ceil_div(nbins, 64) * ceil_div(cfg->channels, 64);
        transpose_kernel<G, float, true><<<tj.tile_begin[1], 256, 0, st>>>(tj);
        count_launch();
    }
    bool in_b = false;
    rc = sort_pairs_u32(cub_tmp, &need, keyA, keyB, idxA, idxB, E, plan.key_bits, &in_b, st);
    if (rc != RSDET_OK) return rc;
    count_launch(2 + ceil_div(plan.key_bits, 8));
    const uint32_t* keys = in_b ? keyB : keyA;
    const int* idx = in_b ? idxB : idxA;
    const long long chunks = ceil_div_ll(E, 32);
    const unsigned blocks = (unsigned)(ceil_div_ll(chunks, 8) < kNumSMs * 8 ? ceil_div_ll(chunks, 8) : kNumSMs * 8);
    const int spb = cfg->sampling_ratio * cfg->sampling_ratio;
    const bool pow2 = (spb & (spb - 1)) == 0;
    if (nhwc_maps(cfg) && pow2) roi_bwd_det_gather_kernel<T, true><<<blocks, 256, 0, st>>>(J, keys, idx, wts, top, E);
    else if (nhwc_maps(cfg)) roi_bwd_det_gather_kernel<T, false><<<blocks, 256, 0, st>>>(J, keys, idx, wts, top, E);
    else if (pow2) roi_bwd_det_gather_kernel<float, true><<<blocks, 256, 0, st>>>(J, keys, idx, wts, top, E);
    else roi_bwd_det_gather_kernel<float, false><<<blocks, 256, 0, st>>>(J, keys, idx, wts, top, E);
    count_launch();
    if (!nhwc_maps(cfg)) {
        rc = launch_transpose(false, acc, grad_feats_host, cfg->height, cfg->width, cfg->num_levels, cfg->batch,
                                        cfg->channels, st);
        if (rc != RSDET_OK) return rc;
    }
    return cuda_status();
}

}  // namespace rsdet

extern "C" size_t rsdet_roi_align_rotated_backward_deterministic_workspace_bytes(const rsdet_roi_align_cfg* cfg, int num_rois,
                                                                                 int feat_dtype) {
    DetPlan plan;
    if (!dtype_ok(feat_dtype) || check_cfg(cfg) != RSDET_OK || !det_plan(cfg, num_rois, &plan)) return 0;
    return det_workspace_bytes(cfg, num_rois, plan, feat_dtype == RSDET_DTYPE_F32);
}

extern "C" int rsdet_roi_align_rotated_backward_deterministic(const rsdet_roi_align_cfg* cfg, int grad_out_dtype,
                                                              const void* grad_out, const float* rois, int num_rois,
                                                              int feat_dtype, void* const* grad_feats_host, void* workspace,
                                                              size_t workspace_bytes, void* stream) {
    if (!dtype_ok(feat_dtype) || (grad_out_dtype != RSDET_DTYPE_F32 && grad_out_dtype != feat_dtype)) return RSDET_EINVAL;
    int rc = check_cfg(cfg);
    if (rc != RSDET_OK) return rc;
    if (cfg->sampling_ratio <= 0 || num_rois < 0 || !grad_feats_host) return RSDET_EINVAL;
    for (int l = 0; l < cfg->num_levels; l++)
        if (!grad_feats_host[l]) return RSDET_EINVAL;
    DetPlan plan;
    if (!det_plan(cfg, num_rois, &plan)) return RSDET_ELIMIT;
    if (num_rois > 0 && (!grad_out || !rois)) return RSDET_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    const bool half_g = grad_out_dtype != RSDET_DTYPE_F32;
#define RSDET_BWD_DET(G_, T_) backward_det_impl<G_, T_>(cfg, plan, static_cast<const G_*>(grad_out), rois, num_rois, \
                                                        reinterpret_cast<T_* const*>(grad_feats_host), workspace, workspace_bytes, st)
    if (feat_dtype == RSDET_DTYPE_F16) return half_g ? RSDET_BWD_DET(__half, __half) : RSDET_BWD_DET(float, __half);
    if (feat_dtype == RSDET_DTYPE_BF16) return half_g ? RSDET_BWD_DET(__nv_bfloat16, __nv_bfloat16) : RSDET_BWD_DET(float, __nv_bfloat16);
    return RSDET_BWD_DET(float, float);
#undef RSDET_BWD_DET
}

extern "C" int rsdet_roi_align_profile_events(void* start_event, void* stop_event) {
    t_prof_start = (cudaEvent_t)start_event;
    t_prof_stop = (cudaEvent_t)stop_event;
    return RSDET_OK;
}

extern "C" int rsdet_nchw_to_nhwc(const float* src, int n, int c, int h, int w, float* dst, void* stream) {
    if (!src || !dst || n < 1 || c < 1 || h < 1 || w < 1) return RSDET_EINVAL;
    const float* s[1] = {src};
    float* d[1] = {dst};
    return launch_transpose(true, s, d, &h, &w, 1, n, c, (cudaStream_t)stream);
}

extern "C" int rsdet_nhwc_to_nchw(const float* src, int n, int c, int h, int w, float* dst, void* stream) {
    if (!src || !dst || n < 1 || c < 1 || h < 1 || w < 1) return RSDET_EINVAL;
    const float* s[1] = {src};
    float* d[1] = {dst};
    return launch_transpose(false, s, d, &h, &w, 1, n, c, (cudaStream_t)stream);
}
