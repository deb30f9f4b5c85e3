// transforms.cu -- box format conversions on the hot path + library bookkeeping.
//
// obb2poly / obb2hbb / poly2hbb: python/jdet/ops/bbox_transforms.py:612-623, 626-632, 602-609 (each is
// ~10 tiny elementwise Jittor kernels in the reference; one fused kernel here, op order preserved).
// poly2origpoly: python/jdet/data/devkits/result_merge.py:196-203.
// poly2obb: cv2.minAreaRect + le90, python/jdet/ops/bbox_transforms.py:549-575 (one thread per quad).
// Compile with -fmad=false so a*b+c stays two IEEE operations like the reference's separate kernels.
#include <cfloat>

#include "common.cuh"

namespace rsdet {

unsigned long long g_launches = 0;

__global__ void obb2poly_kernel(const float* __restrict__ obb, int n, float* __restrict__ poly) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* o = obb + (size_t)i * 5;
    float cx = o[0], cy = o[1], w = o[2], h = o[3], t = o[4];
    float Cos = cosf(t), Sin = sinf(t);
    float v1x = w / 2 * Cos, v1y = -w / 2 * Sin;
    float v2x = -h / 2 * Sin, v2y = -h / 2 * Cos;
    float* p = poly + (size_t)i * 8;
    p[0] = cx + v1x + v2x; p[1] = cy + v1y + v2y;
    p[2] = cx + v1x - v2x; p[3] = cy + v1y - v2y;
    p[4] = cx - v1x - v2x; p[5] = cy - v1y - v2y;
    p[6] = cx - v1x + v2x; p[7] = cy - v1y + v2y;
}

__global__ void obb2hbb_kernel(const float* __restrict__ obb, int n, float* __restrict__ hbb) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* o = obb + (size_t)i * 5;
    float cx = o[0], cy = o[1], w = o[2], h = o[3], t = o[4];
    float Cos = cosf(t), Sin = sinf(t);
    float xb = fabsf(w / 2 * Cos) + fabsf(h / 2 * Sin);
    float yb = fabsf(w / 2 * Sin) + fabsf(h / 2 * Cos);
    float* p = hbb + (size_t)i * 4;
    p[0] = cx - xb; p[1] = cy - yb; p[2] = cx + xb; p[3] = cy + yb;
}

__global__ void poly2hbb_kernel(const float* __restrict__ poly, int n, int np, float* __restrict__ hbb) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* q = poly + (size_t)i * np * 2;
    float x1 = q[0], x2 = q[0], y1 = q[1], y2 = q[1];
    for (int k = 1; k < np; k++) {
        x1 = fminf(x1, q[2 * k]); x2 = fmaxf(x2, q[2 * k]);
        y1 = fminf(y1, q[2 * k + 1]); y2 = fmaxf(y2, q[2 * k + 1]);
    }
    float* p = hbb + (size_t)i * 4;
    p[0] = x1; p[1] = y1; p[2] = x2; p[3] = y2;
}

__global__ void poly2origpoly_kernel(const double* __restrict__ polys, const double* __restrict__ offs, int n,
                                     double* __restrict__ out) {
    int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n * 8) return;
    int i = e >> 3, k = e & 7;
    const double* o = offs + (size_t)i * 3;
    out[e] = (polys[e] + ((k & 1) ? o[1] : o[0])) / o[2];
}

// ---------------------------------------------------------------------------------------------------------- poly2obb
// cv2.minAreaRect (OpenCV 4.13: imgproc/src/convhull.cpp, rotcalipers.cpp) on the 4 float32 corners of a quad, then
// the le90 step of python/jdet/ops/bbox_transforms.py:549-575.  Every float and double operation is OpenCV's, in its
// order; the tests pin a host transcription of the same algorithm to cv2 bit for bit.
// sklansky, convex_hull4 and rotating_calipers stay out of line: inlined into the kernel, nvcc 12.9 -O3 produced a
// wrong hull for sm_100a (the upper and lower chains came back reversed), while the same source is right on the host
// and with -G.
struct P2f { float x, y; };

__device__ __forceinline__ int sign_f(float v) { return (v > 0) - (v < 0); }
__device__ __forceinline__ int sign_d(double v) { return (v > 0) - (v < 0); }

// Sklansky_<float, double> over ptr[start..end] (sorted indices into the quad); returns the stack size
__device__ __noinline__ int sklansky(const P2f* d, const int* ptr, int start, int end, int* stack, int nsign, int sign2) {
    int incr = end > start ? 1 : -1;
    int pprev = start, pcur = pprev + incr, pnext = pcur + incr;
    int stacksize = 3;
    if (start == end || (d[ptr[start]].x == d[ptr[end]].x && d[ptr[start]].y == d[ptr[end]].y)) {
        stack[0] = start;
        return 1;
    }
    stack[0] = pprev;
    stack[1] = pcur;
    stack[2] = pnext;
    end += incr;
    while (pnext != end) {
        float cury = d[ptr[pcur]].y, nexty = d[ptr[pnext]].y;
        float by = nexty - cury;
        if (sign_f(by) != nsign) {
            float ax = d[ptr[pcur]].x - d[ptr[pprev]].x;
            float bx = d[ptr[pnext]].x - d[ptr[pcur]].x;
            float ay = cury - d[ptr[pprev]].y;
            double convexity = (double)ay * bx - (double)ax * by;
            if (sign_d(convexity) == sign2 && (ax != 0 || ay != 0)) {
                pprev = pcur;
                pcur = pnext;
                pnext += incr;
                stack[stacksize++] = pnext;
            } else if (pprev == start) {
                pcur = pnext;
                stack[1] = pcur;
                pnext += incr;
                stack[2] = pnext;
            } else {
                stack[stacksize - 2] = pnext;
                pcur = pprev;
                pprev = stack[stacksize - 4];
                stacksize--;
            }
        } else {
            pnext += incr;
            stack[stacksize - 1] = pnext;
        }
    }
    return --stacksize;
}

// convexHull(points, hull, clockwise=false) of 4 points: hull[] gets indices into d, returns the hull size
__device__ __noinline__ int convex_hull4(const P2f* d, int* hull) {
    int ptr[4] = {0, 1, 2, 3};
    int stack[6];
    for (int i = 1; i < 4; i++) {  // std::sort of 4 elements: a stable insertion sort by (x, y)
        int v = ptr[i], j = i;
        while (j > 0 && (d[v].x < d[ptr[j - 1]].x || (d[v].x == d[ptr[j - 1]].x && d[v].y < d[ptr[j - 1]].y))) {
            ptr[j] = ptr[j - 1];
            j--;
        }
        ptr[j] = v;
    }
    int miny = 0, maxy = 0, nout = 0;
    for (int i = 1; i < 4; i++) {
        float y = d[ptr[i]].y;
        if (d[ptr[miny]].y > y) miny = i;
        if (d[ptr[maxy]].y < y) maxy = i;
    }
    if (d[ptr[0]].x == d[ptr[3]].x && d[ptr[0]].y == d[ptr[3]].y) {
        hull[0] = 0;  // all four points equal
        return 1;
    }
    // upper half; the counter-clockwise output swaps the two stacks
    int* tr = stack;
    int trc = sklansky(d, ptr, 0, maxy, tr, -1, 1);
    int* tl = stack + trc;
    int tlc = sklansky(d, ptr, 3, maxy, tl, -1, -1);
    for (int i = 0; i < tlc - 1; i++) hull[nout++] = ptr[tl[i]];
    for (int i = trc - 1; i > 0; i--) hull[nout++] = ptr[tr[i]];
    int stop = trc > 2 ? tr[1] : tlc > 2 ? tl[tlc - 2] : -1;
    // lower half
    int blc = sklansky(d, ptr, 0, miny, stack, 1, -1);
    int* bl = stack;
    int brc = sklansky(d, ptr, 3, miny, stack + blc, 1, 1);
    int* br = stack + blc;
    if (stop >= 0) {
        int check = blc > 2 ? bl[1] : blc + brc > 2 ? br[2 - blc] : -1;
        if (check == stop || (check >= 0 && d[ptr[check]].x == d[ptr[stop]].x && d[ptr[check]].y == d[ptr[stop]].y)) {
            blc = min(blc, 2);  // all points on one line: the lower part mirrors the upper part
            brc = min(brc, 2);
        }
    }
    for (int i = 0; i < blc - 1; i++) hull[nout++] = ptr[bl[i]];
    for (int i = brc - 1; i > 0; i--) hull[nout++] = ptr[br[i]];
    if (nout >= 3) {  // cyclic shift towards an ascending or descending index sequence
        int min_idx = 0, max_idx = 0, lt = 0, i;
        for (i = 1; i < nout; i++) {
            int idx = hull[i];
            lt += hull[i - 1] < idx;
            if (lt > 1 && lt <= i - 2) break;
            if (idx < hull[min_idx]) min_idx = i;
            if (idx > hull[max_idx]) max_idx = i;
        }
        int mmdist = abs(max_idx - min_idx);
        if ((mmdist == 1 || mmdist == nout - 1) && (lt <= 1 || lt >= nout - 2)) {
            int ascending = (max_idx + 1) % nout == min_idx;
            int j = ascending ? min_idx : max_idx;
            if (j > 0) {
                int tmp[4];
                for (i = 0; i < nout; i++) {
                    int cur = tmp[i] = hull[j];
                    int nj = j + 1 < nout ? j + 1 : 0;
                    if (i < nout - 1 && (ascending != (cur < hull[nj]))) break;
                    j = nj;
                }
                if (i == nout)
                    for (i = 0; i < nout; i++) hull[i] = tmp[i];
            }
        }
    }
    return nout;
}

// rotatingCalipers(points, n, CALIPERS_MINAREARECT, out) for 3 <= n <= 4
__device__ __noinline__ void rotating_calipers(const P2f* pts, int n, float* out) {
    float minarea = FLT_MAX;
    float b_base_a = 0, b_width = 0, b_base_b = 0, b_height = 0;
    int b_left = 0, b_bottom = 0;
    float inv_len[4];
    P2f vect[4];
    int left = 0, bottom = 0, right = 0, top = 0;
    int seq[4];
    P2f pt0 = pts[0];
    float left_x = pt0.x, right_x = pt0.x, top_y = pt0.y, bottom_y = pt0.y;
    for (int i = 0; i < n; i++) {
        // OpenCV tests the previous point while it records index i; kept as is
        if (pt0.x < left_x) left_x = pt0.x, left = i;
        if (pt0.x > right_x) right_x = pt0.x, right = i;
        if (pt0.y > top_y) top_y = pt0.y, top = i;
        if (pt0.y < bottom_y) bottom_y = pt0.y, bottom = i;
        P2f pt = pts[i + 1 < n ? i + 1 : 0];
        double dx = pt.x - pt0.x, dy = pt.y - pt0.y;
        vect[i].x = (float)dx;
        vect[i].y = (float)dy;
        inv_len[i] = (float)(1. / sqrt(dx * dx + dy * dy));
        pt0 = pt;
    }
    float orientation = 0;
    {
        double ax = vect[n - 1].x, ay = vect[n - 1].y;
        for (int i = 0; i < n; i++) {
            double bx = vect[i].x, by = vect[i].y;
            double convexity = ax * by - ay * bx;
            if (convexity != 0) {
                orientation = convexity > 0 ? 1.f : -1.f;
                break;
            }
            ax = bx;
            ay = by;
        }
    }
    float base_a = orientation, base_b = 0;
    seq[0] = bottom;
    seq[1] = right;
    seq[2] = top;
    seq[3] = left;
    for (int k = 0; k < n; k++) {
        P2f rv[4];  // the edge each caliper rests on, turned into caliper 0's frame
        rv[0] = vect[seq[0]];
        rv[1].x = vect[seq[1]].y;  rv[1].y = -vect[seq[1]].x;
        rv[2].x = -vect[seq[2]].x; rv[2].y = -vect[seq[2]].y;
        rv[3].x = -vect[seq[3]].y; rv[3].y = vect[seq[3]].x;
        int main_element = 0;
        for (int i = 1; i < 4; i++) {  // firstVecIsRight(rv[i], rv[main_element])
            float tx = rv[i].y, ty = -rv[i].x;
            if (tx * rv[main_element].x + ty * rv[main_element].y < 0) main_element = i;
        }
        int pindex = seq[main_element];
        float lead_x = vect[pindex].x * inv_len[pindex];
        float lead_y = vect[pindex].y * inv_len[pindex];
        switch (main_element) {
            case 0: base_a = lead_x;  base_b = lead_y;  break;
            case 1: base_a = lead_y;  base_b = -lead_x; break;
            case 2: base_a = -lead_x; base_b = -lead_y; break;
            default: base_a = -lead_y; base_b = lead_x; break;
        }
        seq[main_element] += 1;
        if (seq[main_element] == n) seq[main_element] = 0;
        float dx = pts[seq[1]].x - pts[seq[3]].x;
        float dy = pts[seq[1]].y - pts[seq[3]].y;
        float width = dx * base_a + dy * base_b;
        dx = pts[seq[2]].x - pts[seq[0]].x;
        dy = pts[seq[2]].y - pts[seq[0]].y;
        float height = -dx * base_b + dy * base_a;
        float area = width * height;
        if (area <= minarea) {  // the last minimum wins
            minarea = area;
            b_left = seq[3];
            b_base_a = base_a;
            b_width = width;
            b_base_b = base_b;
            b_height = height;
            b_bottom = seq[0];
        }
    }
    float A1 = b_base_a, B1 = b_base_b, A2 = -b_base_b, B2 = b_base_a;
    float C1 = A1 * pts[b_left].x + pts[b_left].y * B1;
    float C2 = A2 * pts[b_bottom].x + pts[b_bottom].y * B2;
    float idet = 1.f / (A1 * B2 - A2 * B1);
    out[0] = (C1 * B2 - C2 * B1) * idet;
    out[1] = (A1 * C2 - A2 * C1) * idet;
    out[2] = A1 * b_width;
    out[3] = B1 * b_width;
    out[4] = A2 * b_height;
    out[5] = B2 * b_height;
}

__global__ void poly2obb_kernel(const double* __restrict__ polys, int n, double* __restrict__ obb) {
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    const double* p = polys + (size_t)r * 8;
    P2f d[4];
    for (int i = 0; i < 4; i++) {
        d[i].x = (float)p[2 * i];
        d[i].y = (float)p[2 * i + 1];
    }
    int idx[4];
    int nh = convex_hull4(d, idx);
    P2f h[4];
    for (int i = 0; i < nh; i++) h[i] = d[idx[i]];
    float cx, cy, w = 0, hh = 0;
    double angle = 0;
    if (nh > 2) {
        float out[6];
        rotating_calipers(h, nh, out);
        cx = out[0] + (out[2] + out[4]) * 0.5f;
        cy = out[1] + (out[3] + out[5]) * 0.5f;
        w = (float)sqrt((double)out[2] * out[2] + (double)out[3] * out[3]);
        hh = (float)sqrt((double)out[4] * out[4] + (double)out[5] * out[5]);
        angle = atan2((double)out[3], (double)out[2]) * 180 / 3.14159265358979323846;
    } else if (nh == 2) {
        cx = (h[0].x + h[1].x) * 0.5f;
        cy = (h[0].y + h[1].y) * 0.5f;
        double dx = h[1].x - h[0].x, dy = h[1].y - h[0].y;
        w = (float)sqrt(dx * dx + dy * dy);
        angle = atan2(dy, dx) * 180 / 3.14159265358979323846;
    } else {
        cx = h[0].x;
        cy = h[0].y;
    }
    // OpenCV >= 4.5.1 brings the angle into [-90, 0) in double, swapping the sides at each 90-degree step
    while (angle >= 0) { float t = w; w = hh; hh = t; angle -= 90; }
    while (angle < -90) { float t = w; w = hh; hh = t; angle += 90; }
    float a = (float)angle;
    // le90 (bbox_transforms.py:563-574), float64 on the float32 rectangle
    double W = w, H = hh, A;
    if (W >= H) {
        A = -(double)a;
    } else {
        W = hh;
        H = w;
        A = -90 - (double)a;
    }
    double* o = obb + (size_t)r * 5;
    o[0] = cx;
    o[1] = cy;
    o[2] = W;
    o[3] = H;
    o[4] = A / 180 * 3.14159265358979323846;
}

}  // namespace rsdet

using namespace rsdet;

extern "C" int rsdet_version(void) { return 100; }

extern "C" unsigned long long rsdet_launch_count(void) { return g_launches; }

extern "C" const char* rsdet_error_string(int code) {
    switch (code) {
        case RSDET_OK: return "ok";
        case RSDET_EINVAL: return "invalid argument";
        case RSDET_EWORKSPACE: return "workspace too small";
        case RSDET_ELIMIT: return "size above the documented limit";
        default: return code > 0 ? cudaGetErrorString((cudaError_t)code) : "unknown error";
    }
}

extern "C" int rsdet_obb2poly(const float* obb, int n, float* poly, void* stream) {
    if (n < 0) return RSDET_EINVAL;
    if (n == 0) return RSDET_OK;
    if (!obb || !poly) return RSDET_EINVAL;
    obb2poly_kernel<<<ceil_div(n, 256), 256, 0, (cudaStream_t)stream>>>(obb, n, poly);
    count_launch();
    return cuda_status();
}

extern "C" int rsdet_obb2hbb(const float* obb, int n, float* hbb, void* stream) {
    if (n < 0) return RSDET_EINVAL;
    if (n == 0) return RSDET_OK;
    if (!obb || !hbb) return RSDET_EINVAL;
    obb2hbb_kernel<<<ceil_div(n, 256), 256, 0, (cudaStream_t)stream>>>(obb, n, hbb);
    count_launch();
    return cuda_status();
}

extern "C" int rsdet_poly2hbb(const float* poly, int n, int num_points, float* hbb, void* stream) {
    if (n < 0 || num_points < 1) return RSDET_EINVAL;
    if (n == 0) return RSDET_OK;
    if (!poly || !hbb) return RSDET_EINVAL;
    poly2hbb_kernel<<<ceil_div(n, 256), 256, 0, (cudaStream_t)stream>>>(poly, n, num_points, hbb);
    count_launch();
    return cuda_status();
}

extern "C" int rsdet_poly2obb(const double* polys, int n, double* obb, void* stream) {
    if (n < 0) return RSDET_EINVAL;
    if (n == 0) return RSDET_OK;
    if (!polys || !obb) return RSDET_EINVAL;
    poly2obb_kernel<<<ceil_div(n, 128), 128, 0, (cudaStream_t)stream>>>(polys, n, obb);
    count_launch();
    return cuda_status();
}

extern "C" int rsdet_poly2origpoly(const double* polys, const double* offs, int n, double* out, void* stream) {
    if (n < 0) return RSDET_EINVAL;
    if (n == 0) return RSDET_OK;
    if (!polys || !offs || !out) return RSDET_EINVAL;
    poly2origpoly_kernel<<<ceil_div(n * 8, 256), 256, 0, (cudaStream_t)stream>>>(polys, offs, n, out);
    count_launch();
    return cuda_status();
}
