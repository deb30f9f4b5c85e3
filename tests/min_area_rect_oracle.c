/*
 * min_area_rect_oracle.c -- CPU restatement of OpenCV's cv::minAreaRect for 4-point polygons, and of the mirror's
 * le90 step on top of it (python/jdet/ops/bbox_transforms.py:549-575, merge.py:73-100).
 *
 * TEST INFRASTRUCTURE ONLY: the checker for rsdet_poly2obb (csrc/transforms.cu).  Pinned bit for bit against
 * cv2.minAreaRect of OpenCV 4.13 as installed (tests/test_poly2obb_host.py); agreement with 4.5.5, which the reference
 * pins, is unverified.
 *
 * OpenCV's routine, restated in its own operation order (modules/imgproc/src/convhull.cpp, rotcalipers.cpp):
 *   1. convexHull(points, clockwise=false): points sorted by (x, y), Sklansky scans of the upper and lower halves
 *      (float differences, double convexity), then the cyclic shift that makes the hull indices ascending or
 *      descending where it can.
 *   2. rotatingCalipers on the hull (float32 edge vectors, double inverse lengths rounded to float).  The extreme-point
 *      scan compares the previous point's coordinates while it records the current index; that quirk is kept.  The
 *      caliper that turns next is picked by the sign of a float dot product (OpenCV >= 4.5.1); `area <= minarea`
 *      keeps the last minimum; the corner is solved in float32.
 *   3. centre = out[0] + (out[1] + out[2]) * 0.5f; width = |out[1]|, height = |out[2]| (double sqrt rounded to
 *      float); angle = atan2(out[1].y, out[1].x) * 180 / pi in double.  A two-point hull gives its midpoint, its
 *      length as width, 0 as height and the direction of its edge; a one-point hull gives that point, 0, 0 and 0.
 *   4. The angle is brought into [-90, 0) in steps of 90 degrees, each step swapping width and height, still in
 *      double; only then is it rounded to float.
 * Compile with `gcc -O2 -ffp-contract=off -fno-fast-math`: no FMA contraction.
 */
#include <float.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

typedef struct { float x, y; } P2;

static int sign_f(float v) { return (v > 0) - (v < 0); }
static int sign_d(double v) { return (v > 0) - (v < 0); }

/* convhull.cpp Sklansky_<float, double> */
static int sklansky(const P2** a, int start, int end, int* stack, int nsign, int sign2)
{
    int incr = end > start ? 1 : -1;
    int pprev = start, pcur = pprev + incr, pnext = pcur + incr;
    int stacksize = 3;
    if (start == end || (a[start]->x == a[end]->x && a[start]->y == a[end]->y)) {
        stack[0] = start;
        return 1;
    }
    stack[0] = pprev;
    stack[1] = pcur;
    stack[2] = pnext;
    end += incr;
    while (pnext != end) {
        float cury = a[pcur]->y, nexty = a[pnext]->y;
        float by = nexty - cury;
        if (sign_f(by) != nsign) {
            float ax = a[pcur]->x - a[pprev]->x;
            float bx = a[pnext]->x - a[pcur]->x;
            float ay = cury - a[pprev]->y;
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

static int pt_less(const P2* p, const P2* q) { return p->x < q->x || (p->x == q->x && p->y < q->y); }

/* convhull.cpp convexHull(points, hull, clockwise=false, returnPoints) for 4 points: hull indices into d, returns n */
static int convex_hull4(const P2* d, int* hull)
{
    const int total = 4;
    const P2* ptr[4];
    int stack[6];
    int i, nout = 0, miny = 0, maxy = 0;
    for (i = 0; i < total; i++) ptr[i] = &d[i];
    for (i = 1; i < total; i++) { /* std::sort of 4 elements is an insertion sort: stable */
        const P2* v = ptr[i];
        int j = i;
        while (j > 0 && pt_less(v, ptr[j - 1])) { ptr[j] = ptr[j - 1]; j--; }
        ptr[j] = v;
    }
    for (i = 1; i < total; i++) {
        float y = ptr[i]->y;
        if (ptr[miny]->y > y) miny = i;
        if (ptr[maxy]->y < y) maxy = i;
    }
    if (ptr[0]->x == ptr[total - 1]->x && ptr[0]->y == ptr[total - 1]->y) {
        hull[nout++] = 0;
        return nout;
    }
    /* upper half; clockwise == false swaps the two stacks */
    int* tl = stack;
    int tlc = sklansky(ptr, 0, maxy, tl, -1, 1);
    int* tr = stack + tlc;
    int trc = sklansky(ptr, total - 1, maxy, tr, -1, -1);
    { int* t = tl; tl = tr; tr = t; int c = tlc; tlc = trc; trc = c; }
    for (i = 0; i < tlc - 1; i++) hull[nout++] = (int)(ptr[tl[i]] - d);
    for (i = trc - 1; i > 0; i--) hull[nout++] = (int)(ptr[tr[i]] - d);
    int stop = trc > 2 ? tr[1] : tlc > 2 ? tl[tlc - 2] : -1;
    /* lower half */
    int* bl = stack;
    int blc = sklansky(ptr, 0, miny, bl, 1, -1);
    int* br = stack + blc;
    int brc = sklansky(ptr, total - 1, miny, br, 1, 1);
    if (stop >= 0) {
        int check = blc > 2 ? bl[1] : blc + brc > 2 ? br[2 - blc] : -1;
        if (check == stop || (check >= 0 && ptr[check]->x == ptr[stop]->x && ptr[check]->y == ptr[stop]->y)) {
            if (blc > 2) blc = 2; /* all points on one line: the lower part mirrors the upper part */
            if (brc > 2) brc = 2;
        }
    }
    for (i = 0; i < blc - 1; i++) hull[nout++] = (int)(ptr[bl[i]] - d);
    for (i = brc - 1; i > 0; i--) hull[nout++] = (int)(ptr[br[i]] - d);
    if (nout >= 3) { /* cyclic shift towards an ascending or descending index sequence */
        int min_idx = 0, max_idx = 0, lt = 0;
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
            int i0 = ascending ? min_idx : max_idx, j = i0;
            if (i0 > 0) {
                int tmp[4];
                for (i = 0; i < nout; i++) {
                    int cur = tmp[i] = hull[j];
                    int nj = j + 1 < nout ? j + 1 : 0;
                    if (i < nout - 1 && (ascending != (cur < hull[nj]))) break;
                    j = nj;
                }
                if (i == nout) memcpy(hull, tmp, (size_t)nout * sizeof(int));
            }
        }
    }
    return nout;
}

/* rotcalipers.cpp rotatingCalipers(points, n, CALIPERS_MINAREARECT, out) for 3 <= n <= 4 */
static void rotating_calipers(const P2* pts, int n, float out[6])
{
    float minarea = FLT_MAX;
    float b_base_a = 0, b_width = 0, b_base_b = 0, b_height = 0;
    int b_left = 0, b_bottom = 0;
    float inv_len[4];
    P2 vect[4];
    int left = 0, bottom = 0, right = 0, top = 0;
    int seq[4];
    float orientation = 0, base_a, base_b = 0;
    P2 pt0 = pts[0];
    float left_x = pt0.x, right_x = pt0.x, top_y = pt0.y, bottom_y = pt0.y;
    int i, k;
    for (i = 0; i < n; i++) {
        if (pt0.x < left_x) left_x = pt0.x, left = i;
        if (pt0.x > right_x) right_x = pt0.x, right = i;
        if (pt0.y > top_y) top_y = pt0.y, top = i;
        if (pt0.y < bottom_y) bottom_y = pt0.y, bottom = i;
        P2 pt = pts[i + 1 < n ? i + 1 : 0];
        double dx = pt.x - pt0.x, dy = pt.y - pt0.y;
        vect[i].x = (float)dx;
        vect[i].y = (float)dy;
        inv_len[i] = (float)(1. / sqrt(dx * dx + dy * dy));
        pt0 = pt;
    }
    {
        double ax = vect[n - 1].x, ay = vect[n - 1].y;
        for (i = 0; i < n; i++) {
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
    base_a = orientation;
    seq[0] = bottom;
    seq[1] = right;
    seq[2] = top;
    seq[3] = left;
    for (k = 0; k < n; k++) {
        /* rot_vect: the edge each caliper rests on, turned into the frame of caliper 0 */
        P2 rv[4];
        rv[0] = vect[seq[0]];
        rv[1].x = vect[seq[1]].y;  rv[1].y = -vect[seq[1]].x;
        rv[2].x = -vect[seq[2]].x; rv[2].y = -vect[seq[2]].y;
        rv[3].x = -vect[seq[3]].y; rv[3].y = vect[seq[3]].x;
        int main_element = 0;
        for (i = 1; i < 4; i++) { /* firstVecIsRight(rv[i], rv[main_element]) */
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
        if (area <= minarea) {
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

/* cv2.minAreaRect(quad.astype(np.float32)) -> rect[5] = cx, cy, w, h, angle (degrees), all float */
static void min_area_rect4(const float q[8], float rect[5])
{
    P2 d[4], h[4];
    int idx[4];
    int i;
    for (i = 0; i < 4; i++) { d[i].x = q[2 * i]; d[i].y = q[2 * i + 1]; }
    int n = convex_hull4(d, idx);
    for (i = 0; i < n; i++) h[i] = d[idx[i]];
    float cx, cy, w = 0, hh = 0;
    double angle = 0;
    if (n > 2) {
        float out[6];
        rotating_calipers(h, n, out);
        cx = out[0] + (out[2] + out[4]) * 0.5f;
        cy = out[1] + (out[3] + out[5]) * 0.5f;
        w = (float)sqrt((double)out[2] * out[2] + (double)out[3] * out[3]);
        hh = (float)sqrt((double)out[4] * out[4] + (double)out[5] * out[5]);
        angle = atan2((double)out[3], (double)out[2]) * 180 / M_PI;
    } else if (n == 2) {
        cx = (h[0].x + h[1].x) * 0.5f;
        cy = (h[0].y + h[1].y) * 0.5f;
        double dx = h[1].x - h[0].x, dy = h[1].y - h[0].y;
        w = (float)sqrt(dx * dx + dy * dy);
        angle = atan2(dy, dx) * 180 / M_PI;
    } else {
        cx = h[0].x;
        cy = h[0].y;
    }
    while (angle >= 0) { float t = w; w = hh; hh = t; angle -= 90; }
    while (angle < -90) { float t = w; w = hh; hh = t; angle += 90; }
    rect[0] = cx;
    rect[1] = cy;
    rect[2] = w;
    rect[3] = hh;
    rect[4] = (float)angle;
}

/* polys (n, 8) fp64 -> rects (n, 5) fp32: cv2.minAreaRect of each row rounded to float32 */
void mar_min_area_rect(const double* polys, int n, float* rects)
{
    for (int r = 0; r < n; r++) {
        float q[8];
        for (int k = 0; k < 8; k++) q[k] = (float)polys[(size_t)r * 8 + k];
        min_area_rect4(q, rects + (size_t)r * 5);
    }
}

/* polys (n, 8) fp64 -> obb (n, 5) fp64: jdet.ops.bbox_transforms.poly2obb (bbox_transforms.py:549-575) */
void mar_poly2obb(const double* polys, int n, double* obb)
{
    for (int r = 0; r < n; r++) {
        float q[8], rect[5];
        for (int k = 0; k < 8; k++) q[k] = (float)polys[(size_t)r * 8 + k];
        min_area_rect4(q, rect);
        double w = rect[2], h = rect[3], a = rect[4];
        double* o = obb + (size_t)r * 5;
        if (w >= h) {
            a = -a;
        } else {
            double t = w; w = h; h = t;
            a = -90 - a;
        }
        o[0] = rect[0];
        o[1] = rect[1];
        o[2] = w;
        o[3] = h;
        o[4] = a / 180 * M_PI;
    }
}
