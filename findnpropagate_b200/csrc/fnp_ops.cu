// Op-level kernels behind the pcdet.ops API surface (see include/fnp.h for the symbol map).
//
//   points_in_boxes            roiaware_pool3d_kernel.cu:313-336 (first-match index)
//   rotated BEV overlap / IoU  iou3d_nms_kernel.cu:34-234        (convex polygon clipping)
//   rotated / normal NMS       iou3d_nms_kernel.cu:280-385 + iou3d_nms.cpp:113-209
//   recall counters            detectors/detector3d_template.py:315-399
//
// Arithmetic: every fma below is one the reference's sm_100a SASS contains; the library is
// compiled with -fmad=false so nothing else gets contracted.
#include "fnp_common.cuh"

namespace fnp {

// ======================================================================================
// points_in_boxes (API form)
// ======================================================================================
constexpr int kPibThreads = 256;

__global__ void __launch_bounds__(kPibThreads) points_in_boxes_kernel(const float *__restrict__ boxes,
                                                                      const float *__restrict__ pts,
                                                                      int32_t *__restrict__ out, int T, int M)
{
    __shared__ BoxPrep s_box[kPibThreads];
    const int b = blockIdx.y;
    const int i = blockIdx.x * kPibThreads + threadIdx.x;
    const bool live = i < M;
    float x = 0.f, y = 0.f, z = 0.f;
    if (live) {
        const float *p = pts + ((size_t)b * M + i) * 3;
        x = p[0]; y = p[1]; z = p[2];
    }
    int found = -1;
    for (int t0 = 0; t0 < T; t0 += kPibThreads) {
        const int nt = min(kPibThreads, T - t0);
        __syncthreads();
        if ((int)threadIdx.x < nt) s_box[threadIdx.x] = prep_box(boxes + ((size_t)b * T + t0 + threadIdx.x) * 7);
        __syncthreads();
        if (live && found < 0) {
            for (int k = 0; k < nt; k++)
                if (in_box(x, y, z, s_box[k])) { found = t0 + k; break; }
        }
        if (__syncthreads_and(!live || found >= 0)) break;
    }
    if (live) out[(size_t)b * M + i] = found;
}

// ======================================================================================
// count_in_boxes over packed segments (generic op; the fused pipeline uses score_kernel)
// ======================================================================================
constexpr int kCntThreads = 128;
constexpr int kCntTile = 1024;

__global__ void __launch_bounds__(kCntThreads) count_segments_kernel(const float4 *__restrict__ pts,
                                                                     const int32_t *__restrict__ pt_start,
                                                                     const float *__restrict__ boxes,
                                                                     const int32_t *__restrict__ box_start,
                                                                     int32_t *__restrict__ counts)
{
    __shared__ float4 s_pts[kCntTile];
    const int seg = blockIdx.x;
    const int b0 = box_start[seg], nb = box_start[seg + 1] - b0;
    const int p0 = pt_start[seg], np = pt_start[seg + 1] - p0;
    // the CTAs of a segment stride over its boxes, gridDim.y * kCntThreads at a time (the bound is uniform per CTA)
    for (int hb = blockIdx.y * kCntThreads; hb < nb; hb += gridDim.y * kCntThreads) {
        const int h = hb + threadIdx.x;
        BoxPrep bp;
        if (h < nb) bp = prep_box(boxes + (size_t)(b0 + h) * 7);
        else { bp.cx = bp.cy = bp.cz = 0.f; bp.hz = -1.f; bp.cosa = 1.f; bp.sina = 0.f; bp.tx = bp.ty = -1.f; }
        int cnt = 0;
        for (int t0 = 0; t0 < np; t0 += kCntTile) {
            const int m = min(kCntTile, np - t0);
            __syncthreads();
            for (int i = threadIdx.x; i < m; i += kCntThreads) s_pts[i] = pts[p0 + t0 + i];
            __syncthreads();
            for (int i = 0; i < m; i++) {
                const float4 q = s_pts[i];
                count_if(cnt, in_box(q.x, q.y, q.z, bp));
            }
        }
        if (h < nb) counts[b0 + h] = cnt;
    }
}

// ======================================================================================
// points_in_boxes_cpu semantics on the device: the (N, P) 0/1 matrix of the reference's CPU op
// (roiaware_pool3d.cpp:121-168).  Its predicate is NOT the GPU op's: MARGIN is 1e-2 (1 cm) instead of
// 1e-5, and the host compiler evaluates  lx = sx*cosa + sy*(-sina),  ly = sx*sina + sy*cosa  with every
// product rounded (no fma on x86-64 without -mfma), with glibc's cosf/sinf.  The per-box constants
// therefore come from the HOST (fnp_host_prep_boxes_cpu: glibc trig, the fp64 compares hoisted into fp32
// thresholds exactly as for the GPU predicate); this kernel only does the rounded fp32 arithmetic.
//   prep (N,8): cx, cy, cz, hz, cosa, sina, tx, ty   with  |l| < t  <=>  |l| <= t_prepared
// ======================================================================================
constexpr int kMatThreads = 256;
constexpr int kMatBoxes = 16;     // boxes per CTA (rows of the output a CTA writes)

// The CPU op's test of one point against one prepared box (q: the 8 floats of box_prep), every product rounded.
// pib_matrix_kernel and the every-box crop both call it, so the two give the same bits.
__device__ __forceinline__ bool in_box_cpu(float x, float y, float z, const float *q)
{
    const float sz = __fsub_rn(z, q[2]);
    const float sx = __fsub_rn(x, q[0]), sy = __fsub_rn(y, q[1]);
    const float lx = __fadd_rn(__fmul_rn(sx, q[4]), __fmul_rn(sy, -q[5]));
    const float ly = __fadd_rn(__fmul_rn(sx, q[5]), __fmul_rn(sy, q[4]));
    return !(fabsf(sz) > q[3]) && (fabsf(lx) <= q[6]) && (fabsf(ly) <= q[7]);
}

__global__ void __launch_bounds__(kMatThreads) pib_matrix_kernel(const float *__restrict__ prep, const float *__restrict__ pts,
                                                                 int32_t *__restrict__ out, int N, int P)
{
    __shared__ float s_box[kMatBoxes][8];
    const int n0 = blockIdx.y * kMatBoxes;
    const int nb = min(kMatBoxes, N - n0);
    for (int i = threadIdx.x; i < nb * 8; i += kMatThreads) s_box[i / 8][i % 8] = prep[(size_t)n0 * 8 + i];
    __syncthreads();
    const int j = blockIdx.x * kMatThreads + threadIdx.x;
    if (j >= P) return;
    const float x = pts[(size_t)j * 3], y = pts[(size_t)j * 3 + 1], z = pts[(size_t)j * 3 + 2];
    for (int k = 0; k < nb; k++)
        out[(size_t)(n0 + k) * P + j] = in_box_cpu(x, y, z, s_box[k]) ? 1 : 0;      // coalesced along the points
}

// ======================================================================================
// Rotated BEV overlap
// ======================================================================================
struct RBox {
    float px[4], py[4];  // rotated corners, order (x1,y1) (x2,y1) (x2,y2) (x1,y2)
    float cx, cy;        // centre
    float c, s;          // cos(-heading), sin(-heading)   (check_in_box2d)
    float tx, ty;        // dx/2 + 1e-2, dy/2 + 1e-2
    float area;          // dx * dy
    float pad;
};

__device__ __forceinline__ RBox prep_rbox(const float *__restrict__ b)
{
    RBox r;
    const float cx = b[0], cy = b[1], dx = b[3], dy = b[4], ang = b[6];
    const float x1 = __fmaf_rn(dx, -0.5f, cx), x2 = __fmaf_rn(dx, 0.5f, cx);
    const float y1 = __fmaf_rn(dy, -0.5f, cy), y2 = __fmaf_rn(dy, 0.5f, cy);
    const float ca = cosf(ang), sa = sinf(ang);
    const float rx[4] = {x1, x2, x2, x1}, ry[4] = {y1, y1, y2, y2};
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const float ddx = __fsub_rn(rx[k], cx), ddy = __fsub_rn(ry[k], cy);
        // rotate_around_center: first product fused, second rounded (both coordinates)
        r.px[k] = __fadd_rn(__fmaf_rn(ddx, ca, -__fmul_rn(ddy, sa)), cx);
        r.py[k] = __fadd_rn(__fmaf_rn(ddx, sa, __fmul_rn(ddy, ca)), cy);
    }
    r.cx = cx; r.cy = cy;
    r.c = cosf(-ang); r.s = sinf(-ang);
    r.tx = __fmaf_rn(dx, 0.5f, 1e-2f);
    r.ty = __fmaf_rn(dy, 0.5f, 1e-2f);
    r.area = __fmul_rn(dx, dy);
    r.pad = 0.f;
    return r;
}

// a*b - c*d with the first product fused and the second rounded
__device__ __forceinline__ float mulsub(float a, float b, float c, float d)
{
    return __fmaf_rn(a, b, -__fmul_rn(c, d));
}

__device__ __forceinline__ float cross3(float p1x, float p1y, float p2x, float p2y, float p0x, float p0y)
{
    return mulsub(__fsub_rn(p1x, p0x), __fsub_rn(p2y, p0y), __fsub_rn(p2x, p0x), __fsub_rn(p1y, p0y));
}

__device__ __forceinline__ bool seg_intersection(float p1x, float p1y, float p0x, float p0y, float q1x, float q1y,
                                                 float q0x, float q0y, float &ax, float &ay)
{
    if (!(fminf(p0x, p1x) <= fmaxf(q0x, q1x) && fminf(q0x, q1x) <= fmaxf(p0x, p1x) &&
          fminf(p0y, p1y) <= fmaxf(q0y, q1y) && fminf(q0y, q1y) <= fmaxf(p0y, p1y)))
        return false;
    const float s1 = cross3(q0x, q0y, p1x, p1y, p0x, p0y);
    // cross(p1,q1,p0) and cross(q1,p1,p0) share both products: rounded products, plain subtract
    const float P = __fmul_rn(__fsub_rn(p1x, p0x), __fsub_rn(q1y, p0y));
    const float Q = __fmul_rn(__fsub_rn(q1x, p0x), __fsub_rn(p1y, p0y));
    const float s2 = __fsub_rn(P, Q);
    const float s3 = cross3(p0x, p0y, q1x, q1y, q0x, q0y);
    const float s4 = cross3(q1x, q1y, p1x, p1y, q0x, q0y);
    if (!(__fmul_rn(s1, s2) > 0.f && __fmul_rn(s3, s4) > 0.f)) return false;
    const float s5 = __fsub_rn(Q, P);
    const float den = __fsub_rn(s5, s1);
    if (fabsf(den) > 1e-8f) {
        ax = __fdiv_rn(mulsub(s5, q0x, s1, q1x), den);
        ay = __fdiv_rn(mulsub(s5, q0y, s1, q1y), den);
    } else {
        const float a0 = __fsub_rn(p0y, p1y), b0 = __fsub_rn(p1x, p0x), c0 = mulsub(p0x, p1y, p1x, p0y);
        const float a1 = __fsub_rn(q0y, q1y), b1 = __fsub_rn(q1x, q0x), c1 = mulsub(q0x, q1y, q1x, q0y);
        const float D = mulsub(a0, b1, a1, b0);
        ax = __fdiv_rn(mulsub(b0, c1, b1, c0), D);
        ay = __fdiv_rn(mulsub(a1, c0, a0, c1), D);
    }
    return true;
}

__device__ __forceinline__ bool in_box2d(const RBox &bx, float x, float y)
{
    const float ddx = __fsub_rn(x, bx.cx), ddy = __fsub_rn(y, bx.cy);
    const float rx = __fmaf_rn(ddx, bx.c, -__fmul_rn(ddy, bx.s));
    const float ry = __fmaf_rn(ddy, bx.c, __fmul_rn(ddx, bx.s));
    return fabsf(rx) < bx.tx && fabsf(ry) < bx.ty;
}

__device__ float box_overlap(const RBox &A, const RBox &B)
{
    float qx[16], qy[16], key[16];
    float sx = 0.f, sy = 0.f;
    int cnt = 0;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int i1 = (i + 1) & 3;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int j1 = (j + 1) & 3;
            float ax, ay;
            if (seg_intersection(A.px[i1], A.py[i1], A.px[i], A.py[i], B.px[j1], B.py[j1], B.px[j], B.py[j], ax, ay)) {
                if (cnt < 16) { qx[cnt] = ax; qy[cnt] = ay; }
                sx = __fadd_rn(sx, ax); sy = __fadd_rn(sy, ay);
                cnt++;
            }
        }
    }
#pragma unroll
    for (int k = 0; k < 4; k++) {
        if (in_box2d(A, B.px[k], B.py[k])) {
            sx = __fadd_rn(sx, B.px[k]); sy = __fadd_rn(sy, B.py[k]);
            if (cnt < 16) { qx[cnt] = B.px[k]; qy[cnt] = B.py[k]; }
            cnt++;
        }
        if (in_box2d(B, A.px[k], A.py[k])) {
            sx = __fadd_rn(sx, A.px[k]); sy = __fadd_rn(sy, A.py[k]);
            if (cnt < 16) { qx[cnt] = A.px[k]; qy[cnt] = A.py[k]; }
            cnt++;
        }
    }
    if (cnt > 16) cnt = 16;
    if (cnt < 2) return 0.f;  // area loop is empty (also for cnt == 0, where the centroid is 0/0)
    const float fc = (float)cnt;
    const float mx = __fdiv_rn(sx, fc), my = __fdiv_rn(sy, fc);
    for (int k = 0; k < cnt; k++) key[k] = atan2f(__fsub_rn(qy[k], my), __fsub_rn(qx[k], mx));
    // the reference bubble-sorts with `>` on the polar angle; same comparisons, same result
    for (int j = 0; j < cnt - 1; j++)
        for (int i = 0; i < cnt - j - 1; i++)
            if (key[i] > key[i + 1]) {
                float t = key[i]; key[i] = key[i + 1]; key[i + 1] = t;
                t = qx[i]; qx[i] = qx[i + 1]; qx[i + 1] = t;
                t = qy[i]; qy[i] = qy[i + 1]; qy[i + 1] = t;
            }
    float area = 0.f;
    for (int k = 0; k < cnt - 1; k++) {
        const float ax = __fsub_rn(qx[k], qx[0]), ay = __fsub_rn(qy[k], qy[0]);
        const float bx = __fsub_rn(qx[k + 1], qx[0]), by = __fsub_rn(qy[k + 1], qy[0]);
        area = __fadd_rn(area, mulsub(ax, by, ay, bx));
    }
    return __fmul_rn(fabsf(area), 0.5f);
}

// |d|/2 + 1e-2 of a box side d from t = fma(d, 0.5, 1e-2): t itself for d >= 0, and 2e-2 - t for d < 0,
// where t falls below 1e-2 (a negative size spans the same corners as its absolute value)
__device__ __forceinline__ float abs_half_side(float t)
{
    return t >= 1e-2f ? t : 2e-2f - t;
}

// True only when box_overlap(A, B) is exactly 0, for any finite box (a negative or zero size too): the
// centres are further apart than both half diagonals plus a slack that covers the 1e-2 corner margin of
// in_box2d and all rounding, so the polygon clipper would find no edge intersection and no contained
// corner (cnt == 0 -> area 0).  For sizes >= 0 the radius is tx + ty, bit for bit.
__device__ __forceinline__ bool surely_disjoint(const RBox &A, const RBox &B)
{
    const float ddx = A.cx - B.cx, ddy = A.cy - B.cy;
    // >= half diagonal + margin (L1 >= L2)
    const float ra = abs_half_side(A.tx) + abs_half_side(A.ty), rb = abs_half_side(B.tx) + abs_half_side(B.ty);
    const float r = ra + rb + 0.1f;
    return ddx * ddx + ddy * ddy > 1.0001f * r * r;
}

__device__ __forceinline__ float iou_bev(const RBox &A, const RBox &B)
{
    const float ov = box_overlap(A, B);
    return __fdiv_rn(ov, fmaxf(__fsub_rn(__fadd_rn(A.area, B.area), ov), 1e-8f));
}

template <bool IOU>
__global__ void __launch_bounds__(256) pairwise_kernel(const float *__restrict__ a, const float *__restrict__ b,
                                                       float *__restrict__ out, int N, int M)
{
    __shared__ RBox s_a[16], s_b[16];
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int a0 = blockIdx.y * 16, b0 = blockIdx.x * 16;
    if (threadIdx.x < 16) {
        if (a0 + (int)threadIdx.x < N) s_a[threadIdx.x] = prep_rbox(a + (size_t)(a0 + threadIdx.x) * 7);
    } else if (threadIdx.x < 32) {
        const int k = threadIdx.x - 16;
        if (b0 + k < M) s_b[k] = prep_rbox(b + (size_t)(b0 + k) * 7);
    }
    __syncthreads();
    const int ai = a0 + ty, bi = b0 + tx;
    if (ai >= N || bi >= M) return;
    out[(size_t)ai * M + bi] = IOU ? iou_bev(s_a[ty], s_b[tx]) : box_overlap(s_a[ty], s_b[tx]);
}

__global__ void __launch_bounds__(128) aligned_overlap_kernel(const float *__restrict__ a, const float *__restrict__ b,
                                                              float *__restrict__ out, int N)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const RBox A = prep_rbox(a + (size_t)i * 7), B = prep_rbox(b + (size_t)i * 7);
    out[i] = box_overlap(A, B);
}

// 3D IoU from a BEV overlap (iou3d_nms_utils.py:48-81 / :83-117): height overlap, volumes, clamp and
// division, every step one rounded fp32 operation in torch's order.
__device__ __forceinline__ float iou3d_from_overlap(const float *__restrict__ a, const float *__restrict__ b, const float ov_bev)
{
    const float a_hi = __fadd_rn(a[2], __fmul_rn(a[5], 0.5f)), a_lo = __fsub_rn(a[2], __fmul_rn(a[5], 0.5f));
    const float b_hi = __fadd_rn(b[2], __fmul_rn(b[5], 0.5f)), b_lo = __fsub_rn(b[2], __fmul_rn(b[5], 0.5f));
    const float ov_h = fmaxf(__fsub_rn(fminf(a_hi, b_hi), fmaxf(a_lo, b_lo)), 0.f);
    const float ov3 = __fmul_rn(ov_bev, ov_h);
    const float va = __fmul_rn(__fmul_rn(a[3], a[4]), a[5]);
    const float vb = __fmul_rn(__fmul_rn(b[3], b[4]), b[5]);
    return __fdiv_rn(ov3, fmaxf(__fsub_rn(__fadd_rn(va, vb), ov3), 1e-6f));
}

__global__ void __launch_bounds__(256) pairwise_iou3d_kernel(const float *__restrict__ a, const float *__restrict__ b,
                                                             float *__restrict__ out, int N, int M)
{
    __shared__ RBox s_a[16], s_b[16];
    __shared__ float s_ra[16][7], s_rb[16][7];
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int a0 = blockIdx.y * 16, b0 = blockIdx.x * 16;
    if (threadIdx.x < 16) {
        if (a0 + (int)threadIdx.x < N) {
            s_a[threadIdx.x] = prep_rbox(a + (size_t)(a0 + threadIdx.x) * 7);
            for (int k = 0; k < 7; k++) s_ra[threadIdx.x][k] = a[(size_t)(a0 + threadIdx.x) * 7 + k];
        }
    } else if (threadIdx.x < 32) {
        const int k = threadIdx.x - 16;
        if (b0 + k < M) {
            s_b[k] = prep_rbox(b + (size_t)(b0 + k) * 7);
            for (int c = 0; c < 7; c++) s_rb[k][c] = b[(size_t)(b0 + k) * 7 + c];
        }
    }
    __syncthreads();
    const int ai = a0 + ty, bi = b0 + tx;
    if (ai >= N || bi >= M) return;
    out[(size_t)ai * M + bi] = iou3d_from_overlap(s_ra[ty], s_rb[tx], box_overlap(s_a[ty], s_b[tx]));
}

__global__ void __launch_bounds__(128) aligned_iou3d_kernel(const float *__restrict__ a, const float *__restrict__ b,
                                                            float *__restrict__ out, int N)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const RBox A = prep_rbox(a + (size_t)i * 7), B = prep_rbox(b + (size_t)i * 7);
    out[i] = iou3d_from_overlap(a + (size_t)i * 7, b + (size_t)i * 7, box_overlap(A, B));
}

// ======================================================================================
// NMS: 64x64 bitmask tiles + on-device greedy scan
// ======================================================================================
__global__ void __launch_bounds__(128) prep_rbox_kernel(const float *__restrict__ boxes, RBox *__restrict__ out, int N)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N) out[i] = prep_rbox(boxes + (size_t)i * 7);
}

template <bool ROTATED>
__global__ void __launch_bounds__(64) nms_mask_kernel(const float *__restrict__ boxes, const RBox *__restrict__ rb,
                                                      int N, float thresh, unsigned long long *__restrict__ mask)
{
    const int row_blk = blockIdx.y, col_blk = blockIdx.x;
    if (col_blk < row_blk) return;  // the greedy scan never reads the lower triangle
    const int cb = divup(N, 64);
    const int row_n = min(N - row_blk * 64, 64), col_n = min(N - col_blk * 64, 64);
    __shared__ RBox s_rb[ROTATED ? 64 : 1];
    __shared__ float s_raw[64 * 7];
    const int t = threadIdx.x;
    if (t < col_n) {
        if (ROTATED) s_rb[t] = rb[col_blk * 64 + t];
        else
            for (int k = 0; k < 7; k++) s_raw[t * 7 + k] = boxes[(size_t)(col_blk * 64 + t) * 7 + k];
    }
    __syncthreads();
    if (t >= row_n) return;
    const int cur = row_blk * 64 + t;
    unsigned long long bits = 0;
    const int start = (row_blk == col_blk) ? t + 1 : 0;
    if (ROTATED) {
        const RBox me = rb[cur];
        for (int i = start; i < col_n; i++)
            if (iou_bev(me, s_rb[i]) > thresh) bits |= 1ULL << i;
    } else {
        float me[7];
        for (int k = 0; k < 7; k++) me[k] = boxes[(size_t)cur * 7 + k];
        for (int i = start; i < col_n; i++)
            if (iou_normal(me, s_raw + i * 7) > thresh) bits |= 1ULL << i;
    }
    mask[(size_t)cur * cb + col_blk] = bits;
}

// Greedy scan over the bitmask, one CTA.  Per 64-box block: warp 0 resolves the block's own 64 boxes in order
// (the only sequential part), then every thread ORs the kept rows' masks into one later block's "removed"
// word -- loads coalesced along the blocks, four independent accumulators per thread.  remv (cb words) lives
// in dynamic shared memory.
constexpr int kScanThreads = 256;
__global__ void __launch_bounds__(kScanThreads) nms_scan_kernel(const unsigned long long *__restrict__ mask, int N,
                                                                int64_t *__restrict__ keep, int32_t *__restrict__ num_keep)
{
    extern __shared__ unsigned long long s_remv[];
    __shared__ unsigned long long s_kept;
    __shared__ int s_nkeep;
    const int tid = threadIdx.x, lane = tid & 31;
    const int cb = divup(N, 64);
    for (int j = tid; j < cb; j += kScanThreads) s_remv[j] = 0ULL;
    if (tid == 0) s_nkeep = 0;
    __syncthreads();
    for (int b = 0; b < cb; b++) {
        const int n_in = min(64, N - b * 64);
        if (tid < 32) {
            const unsigned long long d0 = (lane < n_in) ? mask[(size_t)(b * 64 + lane) * cb + b] : 0ULL;
            const unsigned long long d1 = (lane + 32 < n_in) ? mask[(size_t)(b * 64 + lane + 32) * cb + b] : 0ULL;
            unsigned long long cur = s_remv[b];
            unsigned long long kept = 0ULL;
            for (int r = 0; r < n_in; r++) {
                const unsigned long long d = __shfl_sync(0xffffffffu, (r < 32) ? d0 : d1, r & 31);
                if (!((cur >> r) & 1ULL)) { kept |= 1ULL << r; cur |= d; }
            }
            const int nkeep = s_nkeep;
            for (int r = lane; r < n_in; r += 32)      // emit kept indices in order
                if ((kept >> r) & 1ULL) keep[nkeep + __popcll(kept & ((1ULL << r) - 1ULL))] = (int64_t)b * 64 + r;
            __syncwarp();
            if (lane == 0) { s_kept = kept; s_nkeep = nkeep + __popcll(kept); }
        }
        __syncthreads();
        const unsigned long long kept = s_kept;
        for (int j = b + 1 + tid; j < cb; j += kScanThreads) {     // propagate the kept rows' masks to later blocks
            unsigned long long a0 = 0ULL, a1 = 0ULL, a2 = 0ULL, a3 = 0ULL, k2 = kept;
            const unsigned long long *col = mask + (size_t)(b * 64) * cb + j;
            while (k2) {
                int r = __ffsll((long long)k2) - 1; k2 &= k2 - 1;
                a0 |= col[(size_t)r * cb];
                if (!k2) break;
                r = __ffsll((long long)k2) - 1; k2 &= k2 - 1;
                a1 |= col[(size_t)r * cb];
                if (!k2) break;
                r = __ffsll((long long)k2) - 1; k2 &= k2 - 1;
                a2 |= col[(size_t)r * cb];
                if (!k2) break;
                r = __ffsll((long long)k2) - 1; k2 &= k2 - 1;
                a3 |= col[(size_t)r * cb];
            }
            s_remv[j] |= (a0 | a1) | (a2 | a3);
        }
        __syncthreads();
    }
    if (tid == 0) *num_keep = s_nkeep;
}

// ======================================================================================
// Stage 4: batched per-segment rotated NMS entirely in shared memory
// ======================================================================================
__global__ void __launch_bounds__(256) seg_nms_kernel(const float *__restrict__ boxes, const int32_t *__restrict__ label,
                                                      const int32_t *__restrict__ order,
                                                      const int32_t *__restrict__ valid,
                                                      const int32_t *__restrict__ seg_start, float thresh,
                                                      uint8_t *__restrict__ keep_mask)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int seg = blockIdx.x;
    const int s0 = seg_start[seg], n = seg_start[seg + 1] - s0;
    if (n <= 0) return;
    const int cb = divup(n, 64);
    RBox *s_rb = reinterpret_cast<RBox *>(smem);
    unsigned long long *s_mask = reinterpret_cast<unsigned long long *>(s_rb + n);
    int *s_lab = reinterpret_cast<int *>(s_mask + (size_t)n * cb);
    unsigned long long *s_remv = reinterpret_cast<unsigned long long *>(s_lab + ((n + 1) & ~1));
    // entry i of the segment is box src(i) = order ? order[s0+i] : s0+i; label -1 = not a box
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const int src = order ? order[s0 + i] : s0 + i;
        s_rb[i] = prep_rbox(boxes + (size_t)src * 7);
        const bool ok = !valid || valid[src] >= 0;
        s_lab[i] = ok ? (label ? label[src] : 0) : -1;
    }
    for (int i = threadIdx.x; i < cb; i += blockDim.x) s_remv[i] = 0ULL;
    __syncthreads();
    for (int w = threadIdx.x; w < n * cb; w += blockDim.x) s_mask[w] = 0ULL;
    __syncthreads();
    // bitmask, one (i, j) pair per thread iteration (the upper triangle of an n x n grid);
    // far-apart pairs are dismissed without running the polygon clipper
    const bool prefilter = thresh >= 0.f;
    for (int p = threadIdx.x; p < n * n; p += blockDim.x) {
        const int i = p / n, j = p - i * n;
        if (j <= i || s_lab[i] < 0 || s_lab[i] != s_lab[j]) continue;
        if (prefilter && surely_disjoint(s_rb[i], s_rb[j])) continue;
        if (iou_bev(s_rb[i], s_rb[j]) > thresh) atomicOr(&s_mask[(size_t)i * cb + (j >> 6)], 1ULL << (j & 63));
    }
    __syncthreads();
    if (threadIdx.x < 32) {
        const int lane = threadIdx.x;
        for (int i = 0; i < n; i++) {
            const bool dead = ((s_remv[i >> 6] >> (i & 63)) & 1ULL) || s_lab[i] < 0;
            if (!dead)
                for (int j = (i >> 6) + lane; j < cb; j += 32) s_remv[j] |= s_mask[(size_t)i * cb + j];
            __syncwarp();
            if (lane == 0) keep_mask[order ? order[s0 + i] : s0 + i] = dead ? 0 : 1;
        }
    }
}

// ======================================================================================
// Recall counters
// ======================================================================================
__global__ void __launch_bounds__(256) recall_kernel(const float *__restrict__ pred, const int32_t *__restrict__ pred_valid,
                                                     const int32_t *__restrict__ pred_start,
                                                     const float *__restrict__ gt, const int32_t *__restrict__ gt_start,
                                                     int n_thresh, float t0, float t1, float t2, float t3, float t4,
                                                     float t5, float t6, float t7, long long *__restrict__ counters)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const float thr[8] = {t0, t1, t2, t3, t4, t5, t6, t7};
    const int fr = blockIdx.x;
    const int p0 = pred_start[fr], K = pred_start[fr + 1] - p0;
    const int g0 = gt_start[fr];
    int G = gt_start[fr + 1] - g0;
    // strip trailing all-zero GT rows (detector3d_template.py:342-346)
    while (G > 0) {
        const float *g = gt + (size_t)(g0 + G - 1) * 8;
        float s = 0.f;
        for (int k = 0; k < 8; k++) s += g[k];
        if (s != 0.f) break;
        G--;
    }
    if (G == 0) return;
    RBox *s_g = reinterpret_cast<RBox *>(smem);          // [G]
    RBox *s_p = s_g + G;                                  // [K]
    int *s_best = reinterpret_cast<int *>(s_p + K);       // [G] float bits; IoU >= 0 orders like int
    for (int i = threadIdx.x; i < G; i += blockDim.x) {
        s_g[i] = prep_rbox(gt + (size_t)(g0 + i) * 8);
        s_best[i] = __float_as_int(-1.f);
    }
    for (int i = threadIdx.x; i < K; i += blockDim.x) {
        s_p[i] = prep_rbox(pred + (size_t)(p0 + i) * 7);
        if (pred_valid && pred_valid[p0 + i] < 0) s_p[i].pad = -1.f;   // not a proposal
    }
    __syncthreads();
    // one (gt, proposal) pair per thread iteration: boxes_iou3d_gpu (iou3d_nms_utils.py:48-81),
    // elementwise fp32 like torch; pairs whose BEV overlap is provably 0 have IoU 0
    for (int q = threadIdx.x; q < G * K; q += blockDim.x) {
        const int gi = q / K, k = q - gi * K;
        if (s_p[k].pad < 0.f) continue;
        float iou = 0.f;
        if (!surely_disjoint(s_p[k], s_g[gi])) {
            const float *g = gt + (size_t)(g0 + gi) * 8;
            const float *p = pred + (size_t)(p0 + k) * 7;
            const float ov_bev = box_overlap(s_p[k], s_g[gi]);
            const float g_hi = __fadd_rn(g[2], __fmul_rn(g[5], 0.5f)), g_lo = __fsub_rn(g[2], __fmul_rn(g[5], 0.5f));
            const float p_hi = __fadd_rn(p[2], __fmul_rn(p[5], 0.5f)), p_lo = __fsub_rn(p[2], __fmul_rn(p[5], 0.5f));
            const float ov_h = fmaxf(__fsub_rn(fminf(p_hi, g_hi), fmaxf(p_lo, g_lo)), 0.f);
            const float ov3 = __fmul_rn(ov_bev, ov_h);
            const float vg = __fmul_rn(__fmul_rn(g[3], g[4]), g[5]);
            const float vp = __fmul_rn(__fmul_rn(p[3], p[4]), p[5]);
            iou = __fdiv_rn(ov3, fmaxf(__fsub_rn(__fadd_rn(vp, vg), ov3), 1e-6f));
        }
        if (iou >= 0.f) atomicMax(&s_best[gi], __float_as_int(iou));
    }
    __syncthreads();
    long long local[5 + 5 * 8];
    for (int i = 0; i < 5 + 5 * 8; i++) local[i] = 0;
    for (int gi = threadIdx.x; gi < G; gi += blockDim.x) {
        const int lab = (int)gt[(size_t)(g0 + gi) * 8 + 7];
        const bool k3 = (lab == 1 || lab == 8 || lab == 9);
        const bool k6 = k3 || lab == 3 || lab == 5 || lab == 6;
        local[0]++;
        local[1] += k3; local[2] += k6; local[3] += !k6; local[4] += !k3;
        const float best = __int_as_float(s_best[gi]);
        for (int t = 0; t < n_thresh; t++)
            if (best > thr[t]) {
                local[5 + 5 * t]++;
                local[5 + 5 * t + 1] += k3; local[5 + 5 * t + 2] += k6;
                local[5 + 5 * t + 3] += !k6; local[5 + 5 * t + 4] += !k3;
            }
    }
    for (int i = 0; i < 5 + 5 * n_thresh; i++) {
        long long v = local[i];
        for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if ((threadIdx.x & 31) == 0 && v) atomicAdd(reinterpret_cast<unsigned long long *>(counters + i), (unsigned long long)v);
    }
}

// Precision counters: per valid proposal the largest IoU3D over its frame's GT boxes (the IoU of recall_kernel),
// thresholded.  One CTA per frame.
__global__ void __launch_bounds__(256) precision_kernel(const float *__restrict__ pred, const int32_t *__restrict__ pred_valid,
                                                        const int32_t *__restrict__ pred_start,
                                                        const float *__restrict__ gt, const int32_t *__restrict__ gt_start,
                                                        int n_thresh, float t0, float t1, float t2, float t3, float t4,
                                                        float t5, float t6, float t7, long long *__restrict__ counters)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const float thr[8] = {t0, t1, t2, t3, t4, t5, t6, t7};
    const int fr = blockIdx.x;
    const int p0 = pred_start[fr], K = pred_start[fr + 1] - p0;
    const int g0 = gt_start[fr], G = gt_start[fr + 1] - g0;
    if (K <= 0) return;
    RBox *s_g = reinterpret_cast<RBox *>(smem);          // [G]
    RBox *s_p = s_g + G;                                  // [K]
    int *s_best = reinterpret_cast<int *>(s_p + K);       // [K] float bits; IoU >= 0 orders like int
    for (int i = threadIdx.x; i < G; i += blockDim.x) s_g[i] = prep_rbox(gt + (size_t)(g0 + i) * 8);
    for (int i = threadIdx.x; i < K; i += blockDim.x) {
        s_p[i] = prep_rbox(pred + (size_t)(p0 + i) * 7);
        if (pred_valid && pred_valid[p0 + i] < 0) s_p[i].pad = -1.f;   // not a proposal
        s_best[i] = __float_as_int(-1.f);
    }
    __syncthreads();
    for (int q = threadIdx.x; q < G * K; q += blockDim.x) {
        const int k = q / G, gi = q - k * G;
        if (s_p[k].pad < 0.f) continue;
        float iou = 0.f;
        if (!surely_disjoint(s_p[k], s_g[gi]))
            iou = iou3d_from_overlap(pred + (size_t)(p0 + k) * 7, gt + (size_t)(g0 + gi) * 8, box_overlap(s_p[k], s_g[gi]));
        if (iou >= 0.f) atomicMax(&s_best[k], __float_as_int(iou));
    }
    __syncthreads();
    long long local[1 + 8];
    for (int i = 0; i < 1 + 8; i++) local[i] = 0;
    for (int k = threadIdx.x; k < K; k += blockDim.x) {
        if (s_p[k].pad < 0.f) continue;
        local[0]++;
        const float best = __int_as_float(s_best[k]);
        for (int t = 0; t < n_thresh; t++) local[1 + t] += best > thr[t];
    }
    for (int i = 0; i < 1 + n_thresh; i++) {
        long long v = local[i];
        for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if ((threadIdx.x & 31) == 0 && v) atomicAdd(reinterpret_cast<unsigned long long *>(counters + i), (unsigned long long)v);
    }
}

// Quality counters: recall and precision per (class, BEV range bin), for many settings of proposals over the same
// frames and GT.  One CTA per (frame, chunk of kQualitySettingsPerCta settings): the frame's GT is staged once, then
// per setting the proposals are staged and every (GT, proposal) pair is computed once; its IoU feeds the four
// per-box maxima (GT: over all / same-label proposals, proposal: over all / same-class GT).  The counters are
// gathered in shared memory and flushed once per setting.
constexpr int kQualitySettingsPerCta = 8;
constexpr int kQualityMaxThresh = 8, kQualityMaxBins = 8, kQualityMaxClasses = 32;

struct QualityParams {
    float thr[kQualityMaxThresh];
    float edges[kQualityMaxBins - 1];
    int n_thresh, n_edges, n_classes;
};

// Range bin of a box centre: the number of edges <= sqrt(x*x + y*y), each operation rounded on its own
__device__ __forceinline__ int range_bin(const float *__restrict__ b, const QualityParams &q)
{
    const float r = __fsqrt_rn(__fadd_rn(__fmul_rn(b[0], b[0]), __fmul_rn(b[1], b[1])));
    int bin = 0;
    for (int e = 0; e < q.n_edges; e++) bin += q.edges[e] <= r;
    return bin;
}

__global__ void __launch_bounds__(256) quality_kernel(const float *__restrict__ pred, long long pred_setting_stride,
                                                      const int32_t *__restrict__ pred_valid, long long valid_setting_stride,
                                                      const int32_t *__restrict__ pred_label,
                                                      const int32_t *__restrict__ pred_start, int n_settings,
                                                      const float *__restrict__ gt, const int32_t *__restrict__ gt_start,
                                                      const QualityParams q, long long *__restrict__ counters)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int fr = blockIdx.x;
    const int s_begin = blockIdx.y * kQualitySettingsPerCta;
    const int s_end = min(n_settings, s_begin + kQualitySettingsPerCta);
    const int p0 = pred_start[fr], K = pred_start[fr + 1] - p0;
    const int g0 = gt_start[fr];
    int G = gt_start[fr + 1] - g0;
    // strip trailing all-zero GT rows (recall_kernel's rule)
    while (G > 0) {
        const float *g = gt + (size_t)(g0 + G - 1) * 8;
        float s = 0.f;
        for (int k = 0; k < 8; k++) s += g[k];
        if (s != 0.f) break;
        G--;
    }
    if (K <= 0 && G == 0) return;
    const int R = q.n_edges + 1, W = 1 + 2 * q.n_thresh;      // counters per (class, bin)
    const int n_block = q.n_classes * R * W;                  // one block: recall, then one: precision
    RBox *s_g = reinterpret_cast<RBox *>(smem);               // [G]
    RBox *s_p = s_g + G;                                      // [K]
    int *s_gbest = reinterpret_cast<int *>(s_p + K);          // [2G]: best IoU (float bits) over all / same-label
    int *s_pbest = s_gbest + 2 * G;                           // [2K]
    int *s_gcell = s_pbest + 2 * K;                           // [G] (class - 1) * R + bin, -1: not counted
    int *s_plab = s_gcell + G;                                // [K] label
    int *s_pcell = s_plab + K;                                // [K] (label - 1) * R + bin, -1: not a proposal
    int *s_cnt = s_pcell + K;                                 // [2 n_block]
    for (int i = threadIdx.x; i < G; i += blockDim.x) {
        const float *g = gt + (size_t)(g0 + i) * 8;
        s_g[i] = prep_rbox(g);
        const int lab = (int)g[7];
        s_gcell[i] = (lab >= 1 && lab <= q.n_classes) ? (lab - 1) * R + range_bin(g, q) : -1;
    }
    for (int k = threadIdx.x; k < K; k += blockDim.x) s_plab[k] = pred_label[p0 + k];
    for (int s = s_begin; s < s_end; s++) {
        const float *P = pred + (size_t)s * pred_setting_stride * 7;
        const int32_t *V = pred_valid ? pred_valid + (size_t)s * valid_setting_stride : nullptr;
        for (int i = threadIdx.x; i < G; i += blockDim.x) s_gbest[2 * i] = s_gbest[2 * i + 1] = __float_as_int(-1.f);
        for (int k = threadIdx.x; k < K; k += blockDim.x) {
            const float *p = P + (size_t)(p0 + k) * 7;
            s_p[k] = prep_rbox(p);
            s_pbest[2 * k] = s_pbest[2 * k + 1] = __float_as_int(-1.f);
            const int lab = s_plab[k];
            const bool ok = (!V || V[p0 + k] >= 0) && lab >= 1 && lab <= q.n_classes;
            if (!ok) s_p[k].pad = -1.f;                       // not a proposal
            s_pcell[k] = ok ? (lab - 1) * R + range_bin(p, q) : -1;
        }
        for (int i = threadIdx.x; i < 2 * n_block; i += blockDim.x) s_cnt[i] = 0;
        __syncthreads();
        // the IoU of recall_kernel / precision_kernel, bit for bit
        for (int w = threadIdx.x; w < G * K; w += blockDim.x) {
            const int gi = w / K, k = w - gi * K;
            if (s_p[k].pad < 0.f) continue;
            float iou = 0.f;
            if (!surely_disjoint(s_p[k], s_g[gi]))
                iou = iou3d_from_overlap(P + (size_t)(p0 + k) * 7, gt + (size_t)(g0 + gi) * 8, box_overlap(s_p[k], s_g[gi]));
            if (!(iou >= 0.f)) continue;
            const int bits = __float_as_int(iou);
            atomicMax(&s_gbest[2 * gi], bits);
            atomicMax(&s_pbest[2 * k], bits);
            if (s_plab[k] == (int)gt[(size_t)(g0 + gi) * 8 + 7]) {
                atomicMax(&s_gbest[2 * gi + 1], bits);
                atomicMax(&s_pbest[2 * k + 1], bits);
            }
        }
        __syncthreads();
        for (int i = threadIdx.x; i < G; i += blockDim.x) {
            if (s_gcell[i] < 0) continue;
            int *c = s_cnt + s_gcell[i] * W;
            const float ba = __int_as_float(s_gbest[2 * i]), bl = __int_as_float(s_gbest[2 * i + 1]);
            atomicAdd(c, 1);
            for (int t = 0; t < q.n_thresh; t++) {
                if (ba > q.thr[t]) atomicAdd(c + 1 + t, 1);
                if (bl > q.thr[t]) atomicAdd(c + 1 + q.n_thresh + t, 1);
            }
        }
        for (int k = threadIdx.x; k < K; k += blockDim.x) {
            if (s_pcell[k] < 0) continue;
            int *c = s_cnt + n_block + s_pcell[k] * W;
            const float ba = __int_as_float(s_pbest[2 * k]), bl = __int_as_float(s_pbest[2 * k + 1]);
            atomicAdd(c, 1);
            for (int t = 0; t < q.n_thresh; t++) {
                if (ba > q.thr[t]) atomicAdd(c + 1 + t, 1);
                if (bl > q.thr[t]) atomicAdd(c + 1 + q.n_thresh + t, 1);
            }
        }
        __syncthreads();
        long long *out = counters + (size_t)s * 2 * n_block;
        for (int i = threadIdx.x; i < 2 * n_block; i += blockDim.x)
            if (s_cnt[i]) atomicAdd(reinterpret_cast<unsigned long long *>(out + i), (unsigned long long)s_cnt[i]);
        __syncthreads();
    }
}

// Small host->device upload executed by SMs: `src` is pinned (page-locked, UVA-mapped) host
// memory.  Used for the per-batch metadata so that it does not queue behind a large point
// copy in the H2D copy engine (copies of different streams are not served in issue order).
__global__ void __launch_bounds__(256) upload_kernel(uint4 *__restrict__ dst, const uint4 *__restrict__ src, size_t n16)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x)
        dst[i] = src[i];
}

// ======================================================================================
// Crop points in boxes: each point to the first box of its frame that contains it (the
// predicate of points_in_boxes_kernel), then every box's points copied out contiguously, in
// input order, with the box centre subtracted from x, y, z.
//
// A frame's points are cut into tiles of kCropTile rows.  Per frame the workspace holds a
// tiles x boxes int32 matrix: crop_assign_kernel counts each tile's points per box in it,
// crop_prefix_kernel turns every box's column into exclusive offsets over the tiles (and
// writes the box's count), crop_starts_kernel scans the counts into row starts, and
// crop_scatter_kernel copies each tile's points in order, one warp per tile, ranking points
// of the same box within 32 rows with __match_any_sync.  Counting atomics only add; no
// atomic decides a position, so the output is the same on every run.
// ======================================================================================
constexpr int kCropTile = 1024;
constexpr int kCropThreads = 256;
constexpr int kCropPerThread = kCropTile / kCropThreads;
constexpr int kCropScanThreads = 1024;

struct CropWs {                 // the workspace, carved as fnp_crop_workspace_bytes sizes it
    int64_t *mat_start;         // (n_frames + 1): frame f's matrix at mat + mat_start[f]
    int64_t *tile_start;        // (n_frames + 1): frame f's tiles are tile_start[f] ..
    int32_t *box_of_pt;         // (n_points): box index within the frame, or -1
    int32_t *mat;               // (mat_cap)
    long long mat_cap, n_points, n_boxes;
};

// The starts end at the sizes the call was given and the matrix fits: otherwise no kernel
// touches the outputs past counts (all zero), so a wrong call cannot write out of bounds.
__device__ __forceinline__ bool crop_ok(const int64_t *__restrict__ row_start, const int64_t *__restrict__ box_start,
                                        int n_frames, const CropWs &ws)
{
    return ws.mat_start[n_frames] <= ws.mat_cap && row_start[0] == 0 && box_start[0] == 0 &&
           row_start[n_frames] == ws.n_points && box_start[n_frames] == ws.n_boxes;
}

__device__ __forceinline__ int crop_frame_of(const int64_t *__restrict__ start, int n_frames, long long v)
{
    int lo = 0, hi = n_frames - 1;      // last f with start[f] <= v
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (start[mid] <= v) lo = mid; else hi = mid - 1;
    }
    return lo;
}

__global__ void __launch_bounds__(kCropScanThreads) crop_plan_kernel(const int64_t *__restrict__ row_start,
                                                                     const int64_t *__restrict__ box_start, int n_frames,
                                                                     CropWs ws)
{
    __shared__ long long s_carry[2];
    __shared__ long long s_warp[2][kCropScanThreads / 32];
    if (threadIdx.x == 0) { s_carry[0] = 0; s_carry[1] = 0; }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int f0 = 0; f0 <= n_frames; f0 += kCropScanThreads) {
        const int f = f0 + threadIdx.x;
        long long v[2] = {0, 0};
        if (f < n_frames) {
            const long long tiles = (row_start[f + 1] - row_start[f] + kCropTile - 1) / kCropTile;
            v[0] = tiles * (long long)(box_start[f + 1] - box_start[f]);
            v[1] = tiles;
        }
        __syncthreads();
        long long incl[2];
        for (int k = 0; k < 2; k++) {
            incl[k] = v[k];
            for (int o = 1; o < 32; o <<= 1) {
                const long long u = __shfl_up_sync(0xffffffffu, incl[k], o);
                if (lane >= o) incl[k] += u;
            }
            if (lane == 31) s_warp[k][warp] = incl[k];
        }
        __syncthreads();
        for (int k = 0; k < 2; k++) {
            long long before = s_carry[k];
            for (int w = 0; w < warp; w++) before += s_warp[k][w];
            if (f <= n_frames) (k ? ws.tile_start : ws.mat_start)[f] = before + incl[k] - v[k];
        }
        __syncthreads();
        if (threadIdx.x == 0)
            for (int k = 0; k < 2; k++)
                for (int w = 0; w < kCropScanThreads / 32; w++) s_carry[k] += s_warp[k][w];
    }
}

// Tile -> (frame, first row, rows); false for a grid slot past the last tile or a matrix that
// does not fit the workspace.
__device__ __forceinline__ bool crop_tile(const int64_t *__restrict__ row_start, const int64_t *__restrict__ box_start,
                                          int n_frames, const CropWs &ws, long long tile, int &f, long long &r0, int &n)
{
    if (n_frames == 0 || tile >= ws.tile_start[n_frames] || !crop_ok(row_start, box_start, n_frames, ws)) return false;
    f = crop_frame_of(ws.tile_start, n_frames, tile);
    const long long t = tile - ws.tile_start[f];
    r0 = row_start[f] + t * kCropTile;
    n = (int)min((long long)kCropTile, row_start[f + 1] - r0);
    return true;
}

__global__ void __launch_bounds__(kCropThreads) crop_assign_kernel(const float *__restrict__ pts, int n_cols,
                                                                   const int64_t *__restrict__ row_start,
                                                                   const float *__restrict__ boxes,
                                                                   const int64_t *__restrict__ box_start, int n_frames,
                                                                   CropWs ws)
{
    __shared__ BoxPrep s_box[kCropThreads];
    int f, n;
    long long r0;
    if (!crop_tile(row_start, box_start, n_frames, ws, blockIdx.x, f, r0, n)) return;
    const long long b0 = box_start[f];
    const int T = (int)(box_start[f + 1] - b0);
    float x[kCropPerThread], y[kCropPerThread], z[kCropPerThread];
    int found[kCropPerThread];
#pragma unroll
    for (int j = 0; j < kCropPerThread; j++) {
        const int i = j * kCropThreads + threadIdx.x;
        found[j] = i < n ? -1 : 0;          // 0: a slot past the tile's end, never tested
        x[j] = y[j] = z[j] = 0.f;
        if (i < n) {
            const float *p = pts + (size_t)(r0 + i) * n_cols;
            x[j] = p[0]; y[j] = p[1]; z[j] = p[2];
        }
    }
    for (int t0 = 0; t0 < T; t0 += kCropThreads) {
        const int nt = min(kCropThreads, T - t0);
        __syncthreads();
        if ((int)threadIdx.x < nt) s_box[threadIdx.x] = prep_box(boxes + (size_t)(b0 + t0 + threadIdx.x) * 7);
        __syncthreads();
        bool done = true;
#pragma unroll
        for (int j = 0; j < kCropPerThread; j++) {
            if (found[j] < 0)
                for (int k = 0; k < nt; k++)
                    if (in_box(x[j], y[j], z[j], s_box[k])) { found[j] = t0 + k; break; }
            done = done && found[j] >= 0;
        }
        if (__syncthreads_and(done)) break;
    }
    int32_t *row = ws.mat + ws.mat_start[f] + (blockIdx.x - ws.tile_start[f]) * (long long)T;
#pragma unroll
    for (int j = 0; j < kCropPerThread; j++) {
        const int i = j * kCropThreads + threadIdx.x;
        if (i < n) {
            ws.box_of_pt[r0 + i] = found[j];
            if (found[j] >= 0) atomicAdd(row + found[j], 1);
        }
    }
}

// One thread per box: its column of the frame's matrix becomes exclusive offsets over the tiles.
__global__ void __launch_bounds__(128) crop_prefix_kernel(const int64_t *__restrict__ row_start,
                                                          const int64_t *__restrict__ box_start, int n_frames,
                                                          int n_boxes, CropWs ws, int32_t *__restrict__ counts)
{
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n_boxes) return;
    if (!crop_ok(row_start, box_start, n_frames, ws)) { counts[g] = 0; return; }
    const int f = crop_frame_of(box_start, n_frames, g);
    const long long T = box_start[f + 1] - box_start[f];
    const long long tiles = ws.tile_start[f + 1] - ws.tile_start[f];
    int32_t *col = ws.mat + ws.mat_start[f] + (g - box_start[f]);
    int run = 0;
    long long t = 0;
    for (; t + 8 <= tiles; t += 8) {
        int v[8];
#pragma unroll
        for (int k = 0; k < 8; k++) v[k] = col[(t + k) * T];
#pragma unroll
        for (int k = 0; k < 8; k++) { col[(t + k) * T] = run; run += v[k]; }
    }
    for (; t < tiles; t++) {
        const int v = col[t * T];
        col[t * T] = run;
        run += v;
    }
    counts[g] = run;
}

// starts[g] = counts[0] + ... + counts[g-1] for g = 0 .. n_boxes (one CTA).
__global__ void __launch_bounds__(kCropScanThreads) crop_starts_kernel(const int32_t *__restrict__ counts, int n_boxes,
                                                                       int64_t *__restrict__ starts)
{
    __shared__ long long s_warp[kCropScanThreads / 32];
    __shared__ long long s_carry;
    if (threadIdx.x == 0) s_carry = 0;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int g0 = 0; g0 <= n_boxes; g0 += kCropScanThreads) {
        const int g = g0 + threadIdx.x;
        const long long v = g < n_boxes ? counts[g] : 0;
        long long incl = v;
        for (int o = 1; o < 32; o <<= 1) {
            const long long u = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += u;
        }
        __syncthreads();
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        long long before = s_carry;
        for (int w = 0; w < warp; w++) before += s_warp[w];
        if (g <= n_boxes) starts[g] = before + incl - v;
        __syncthreads();
        if (threadIdx.x == 0)
            for (int w = 0; w < kCropScanThreads / 32; w++) s_carry += s_warp[w];
    }
}

// One warp per tile, 32 rows at a time in input order.  The tile's matrix row holds, per box,
// where its next point goes within the box; only this warp touches it.
__global__ void __launch_bounds__(32) crop_scatter_kernel(const float *__restrict__ pts, int n_cols,
                                                          const int64_t *__restrict__ row_start,
                                                          const double *__restrict__ centres,
                                                          const int64_t *__restrict__ box_start, int n_frames,
                                                          CropWs ws, const int64_t *__restrict__ starts,
                                                          float *__restrict__ rows)
{
    int f, n;
    long long r0;
    if (!crop_tile(row_start, box_start, n_frames, ws, blockIdx.x, f, r0, n)) return;
    const long long b0 = box_start[f];
    const long long T = box_start[f + 1] - b0;
    int32_t *next = ws.mat + ws.mat_start[f] + (blockIdx.x - ws.tile_start[f]) * T;
    const unsigned lane = threadIdx.x;
    for (int i0 = 0; i0 < n; i0 += 32) {
        const int i = i0 + (int)lane;
        const int b = i < n ? ws.box_of_pt[r0 + i] : -1;
        const unsigned same = __match_any_sync(0xffffffffu, b);
        int base = 0;
        if (b >= 0) base = next[b];
        __syncwarp();
        if (b >= 0 && lane == (unsigned)(__ffs(same) - 1)) next[b] = base + __popc(same);
        __syncwarp();
        if (b < 0) continue;
        const long long g = b0 + b;
        const long long out = starts[g] + base + __popc(same & ((1u << lane) - 1u));
        const float *p = pts + (size_t)(r0 + i) * n_cols;
        float *o = rows + (size_t)out * n_cols;
#pragma unroll
        for (int c = 0; c < 3; c++) o[c] = __double2float_rn(__dsub_rn((double)p[c], centres[g * 3 + c]));
        for (int c = 3; c < n_cols; c++) o[c] = p[c];
    }
}

// --------------------------------------------------------------------------------------
// Every-box crop (points_in_boxes_cpu + points[mask[i] > 0], KittiDataset.create_groundtruth_database): a point is
// written once for every box of its frame that contains it, by in_box_cpu on fnp_host_prep_boxes_cpu's constants.
// The plan, the per-(tile, box) matrix, crop_prefix_kernel and crop_starts_kernel are the first-match crop's; only
// the count and the scatter differ.  crop_all_count_kernel writes each (tile, box) count, summed from warp ballots
// (no atomic); crop_all_scatter_kernel gives each box of a tile to one warp, which walks the tile's points in row
// order and ranks the ones in the box with a ballot.
// --------------------------------------------------------------------------------------
constexpr int kCropWarps = kCropThreads / 32;

__global__ void __launch_bounds__(kCropThreads) crop_all_count_kernel(const float *__restrict__ pts, int n_cols,
                                                                      const int64_t *__restrict__ row_start,
                                                                      const float *__restrict__ box_prep,
                                                                      const int64_t *__restrict__ box_start,
                                                                      int n_frames, CropWs ws)
{
    __shared__ float s_box[kCropThreads][8];
    __shared__ int s_cnt[kCropWarps][kCropThreads];
    int f, n;
    long long r0;
    if (!crop_tile(row_start, box_start, n_frames, ws, blockIdx.x, f, r0, n)) return;
    const long long b0 = box_start[f];
    const int T = (int)(box_start[f + 1] - b0);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float x[kCropPerThread], y[kCropPerThread], z[kCropPerThread];
#pragma unroll
    for (int j = 0; j < kCropPerThread; j++) {
        const int i = j * kCropThreads + threadIdx.x;
        x[j] = y[j] = z[j] = 0.f;
        if (i < n) {
            const float *p = pts + (size_t)(r0 + i) * n_cols;
            x[j] = p[0]; y[j] = p[1]; z[j] = p[2];
        }
    }
    int32_t *row = ws.mat + ws.mat_start[f] + (blockIdx.x - ws.tile_start[f]) * (long long)T;
    for (int t0 = 0; t0 < T; t0 += kCropThreads) {
        const int nt = min(kCropThreads, T - t0);
        __syncthreads();
        if ((int)threadIdx.x < nt)
#pragma unroll
            for (int c = 0; c < 8; c++) s_box[threadIdx.x][c] = box_prep[(size_t)(b0 + t0 + threadIdx.x) * 8 + c];
        __syncthreads();
        for (int k = 0; k < nt; k++) {
            int c = 0;
#pragma unroll
            for (int j = 0; j < kCropPerThread; j++) {
                const bool in = j * kCropThreads + (int)threadIdx.x < n && in_box_cpu(x[j], y[j], z[j], s_box[k]);
                c += __popc(__ballot_sync(0xffffffffu, in));
            }
            if (lane == 0) s_cnt[warp][k] = c;
        }
        __syncthreads();
        if ((int)threadIdx.x < nt) {
            int c = 0;
#pragma unroll
            for (int w = 0; w < kCropWarps; w++) c += s_cnt[w][threadIdx.x];
            row[t0 + threadIdx.x] = c;
        }
    }
}

// After crop_prefix_kernel the tile's matrix row holds each box's offset within the box, and the next tile's row (or
// the box's count, for the last tile) where this tile's points of the box end.  A warp stops a box once it has
// written them all, skips a box with none in the tile, and never writes at or past rows_cap.
__global__ void __launch_bounds__(kCropThreads) crop_all_scatter_kernel(const float *__restrict__ pts, int n_cols,
                                                                        const int64_t *__restrict__ row_start,
                                                                        const float *__restrict__ box_prep,
                                                                        const double *__restrict__ centres,
                                                                        const int64_t *__restrict__ box_start,
                                                                        int n_frames, CropWs ws,
                                                                        const int64_t *__restrict__ starts,
                                                                        float *__restrict__ rows, long long rows_cap)
{
    __shared__ float s_xyz[3][kCropTile];
    int f, n;
    long long r0;
    if (!crop_tile(row_start, box_start, n_frames, ws, blockIdx.x, f, r0, n)) return;
    const long long b0 = box_start[f];
    const int T = (int)(box_start[f + 1] - b0);
    if (T == 0) return;
    for (int i = threadIdx.x; i < n; i += kCropThreads) {
        const float *p = pts + (size_t)(r0 + i) * n_cols;
        s_xyz[0][i] = p[0]; s_xyz[1][i] = p[1]; s_xyz[2][i] = p[2];
    }
    __syncthreads();
    const unsigned lane = threadIdx.x & 31;
    const long long t = blockIdx.x - ws.tile_start[f], tiles = ws.tile_start[f + 1] - ws.tile_start[f];
    const int32_t *off = ws.mat + ws.mat_start[f] + t * T;
    for (int k = threadIdx.x >> 5; k < T; k += kCropWarps) {
        const long long g = b0 + k;
        const long long end = t + 1 < tiles ? (long long)off[k + T] : starts[g + 1] - starts[g];
        long long left = end - off[k];
        if (left <= 0) continue;
        float q[8];
#pragma unroll
        for (int c = 0; c < 8; c++) q[c] = box_prep[(size_t)g * 8 + c];
        long long out = starts[g] + off[k];
        for (int i0 = 0; i0 < n && left > 0; i0 += 32) {
            const int i = i0 + (int)lane;
            const bool in = i < n && in_box_cpu(s_xyz[0][i], s_xyz[1][i], s_xyz[2][i], q);
            const unsigned m = __ballot_sync(0xffffffffu, in);
            const long long r = out + __popc(m & ((1u << lane) - 1u));
            if (in && r >= 0 && r < rows_cap) {
                const float *p = pts + (size_t)(r0 + i) * n_cols;
                float *o = rows + (size_t)r * n_cols;
#pragma unroll
                for (int c = 0; c < 3; c++) o[c] = __double2float_rn(__dsub_rn((double)p[c], centres[g * 3 + c]));
                for (int c = 3; c < n_cols; c++) o[c] = p[c];
            }
            out += __popc(m);
            left -= __popc(m);
        }
    }
}

// test hook: the device math routines exactly as this library's kernels see them
__global__ void dbg_math_kernel(const float *__restrict__ x, const float *__restrict__ y, float *__restrict__ out, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    out[i] = sinf(x[i]);
    out[n + i] = cosf(x[i]);
    out[2 * n + i] = atan2f(y[i], x[i]);
    out[3 * n + i] = fnp_exp(x[i]);
}

}  // namespace fnp

using namespace fnp;

extern "C" int fnp_dbg_math(const float *x, const float *y, float *out, int n, void *stream)
{
    if (n <= 0) return FNP_OK;
    dbg_math_kernel<<<divup(n, 256), 256, 0, (cudaStream_t)stream>>>(x, y, out, n);
    FNP_LAUNCH_CHECK();
    return FNP_OK;
}

extern "C" int fnp_upload_from_pinned(void *dst, const void *src_pinned_host, size_t bytes, void *stream)
{
    if (bytes == 0) return FNP_OK;
    if (!dst || !src_pinned_host || (bytes & 15) || (reinterpret_cast<uintptr_t>(dst) & 15) ||
        (reinterpret_cast<uintptr_t>(src_pinned_host) & 15))
        return FNP_EINVAL;
    const size_t n16 = bytes >> 4;
    const int grid = (int)((n16 + 255) / 256 < 296 ? (n16 + 255) / 256 : 296);
    upload_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<uint4 *>(dst),
                                                          reinterpret_cast<const uint4 *>(src_pinned_host), n16);
    FNP_LAUNCH_CHECK();
    return FNP_OK;
}

extern "C" const char *fnp_version(void) { return "fnp-sm100a 0.1"; }

extern "C" int fnp_points_in_boxes(const float *boxes, const float *pts, int32_t *out, int B, int T, int M, void *stream)
{
    if (B < 0 || T < 0 || M < 0) return FNP_EINVAL;
    if (B == 0 || M == 0) return FNP_OK;
    if (!pts || !out || (T > 0 && !boxes)) return FNP_EINVAL;
    if (B > 65535) return FNP_EINVAL;
    dim3 grid(divup(M, kPibThreads), B);
    points_in_boxes_kernel<<<grid, kPibThreads, 0, (cudaStream_t)stream>>>(boxes, pts, out, T, M);
    FNP_LAUNCH_CHECK();
    return FNP_OK;
}

static size_t crop_head_bytes(long long n_points, int n_frames)
{
    return (size_t)2 * (n_frames + 1) * 8 + ((size_t)n_points * 4 + 15) / 16 * 16;
}

extern "C" size_t fnp_crop_workspace_bytes(const int64_t *row_start_host, const int64_t *box_start_host, int n_frames)
{
    if (n_frames < 0 || (n_frames > 0 && (!row_start_host || !box_start_host))) return 0;
    size_t mat = 0;
    for (int f = 0; f < n_frames; f++) {
        const long long n = row_start_host[f + 1] - row_start_host[f], g = box_start_host[f + 1] - box_start_host[f];
        if (n > 0 && g > 0) mat += (size_t)((n + kCropTile - 1) / kCropTile) * (size_t)g;
    }
    return crop_head_bytes(n_frames ? row_start_host[n_frames] : 0, n_frames) + mat * 4 + 16;
}

// The workspace as fnp_crop_workspace_bytes sizes it (the caller has checked it holds the head).
static CropWs crop_carve(void *workspace, size_t workspace_bytes, long long n_points, int n_boxes, int n_frames)
{
    const size_t head = crop_head_bytes(n_points, n_frames);
    char *w = static_cast<char *>(workspace);
    CropWs ws;
    ws.mat_start = reinterpret_cast<int64_t *>(w);
    ws.tile_start = ws.mat_start + n_frames + 1;
    ws.box_of_pt = reinterpret_cast<int32_t *>(ws.tile_start + n_frames + 1);
    ws.mat = reinterpret_cast<int32_t *>(w + head);
    ws.mat_cap = (long long)((workspace_bytes - head) / 4);
    ws.n_points = n_points;
    ws.n_boxes = n_boxes;
    return ws;
}

// The size and pointer checks the crop entries share: FNP_OK, FNP_EINVAL or FNP_EWORKSPACE.
static int crop_check(const float *pts, int n_cols, const int64_t *row_start, long long n_points,
                      const int64_t *box_start, int n_boxes, int n_frames, const int64_t *starts,
                      const void *workspace, size_t workspace_bytes)
{
    if (n_cols < 3 || n_points < 0 || n_boxes < 0 || n_frames < 0 || n_frames > 65535 * 1024) return FNP_EINVAL;
    if (n_frames == 0 && (n_points || n_boxes)) return FNP_EINVAL;
    if (!row_start || !box_start || !starts || !workspace || (n_points && !pts) ||
        (reinterpret_cast<uintptr_t>(workspace) & 15))
        return FNP_EINVAL;
    if (n_points / kCropTile + n_frames > 0x7fffffffLL || divup(n_boxes, 128) > 0x7fffffff) return FNP_EINVAL;
    if (workspace_bytes < crop_head_bytes(n_points, n_frames) + 16) return FNP_EWORKSPACE;
    return FNP_OK;
}

extern "C" int fnp_crop_all_count(const float *pts, int n_cols, const int64_t *row_start, long long n_points,
                                  const float *box_prep, const int64_t *box_start, int n_boxes, int n_frames,
                                  int32_t *counts, int64_t *starts, void *workspace, size_t workspace_bytes,
                                  void *stream)
{
    if (n_boxes > 0 && (!box_prep || !counts)) return FNP_EINVAL;
    const int rc = crop_check(pts, n_cols, row_start, n_points, box_start, n_boxes, n_frames, starts, workspace,
                              workspace_bytes);
    if (rc != FNP_OK) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    const CropWs ws = crop_carve(workspace, workspace_bytes, n_points, n_boxes, n_frames);
    const long long n_tiles = n_points / kCropTile + n_frames;
    const cudaError_t e = cudaMemsetAsync(ws.mat, 0, workspace_bytes - crop_head_bytes(n_points, n_frames), s);
    if (e != cudaSuccess) return (int)e;
    crop_plan_kernel<<<1, kCropScanThreads, 0, s>>>(row_start, box_start, n_frames, ws);
    FNP_LAUNCH_CHECK();
    if (n_tiles > 0 && n_boxes > 0)
        crop_all_count_kernel<<<(unsigned)n_tiles, kCropThreads, 0, s>>>(pts, n_cols, row_start, box_prep, box_start,
                                                                         n_frames, ws);
    FNP_LAUNCH_CHECK();
    if (n_boxes > 0)
        crop_prefix_kernel<<<divup(n_boxes, 128), 128, 0, s>>>(row_start, box_start, n_frames, n_boxes, ws, counts);
    FNP_LAUNCH_CHECK();
    crop_starts_kernel<<<1, kCropScanThreads, 0, s>>>(counts, n_boxes, starts);
    FNP_LAUNCH_CHECK();
    return FNP_OK;
}

extern "C" int fnp_crop_all_scatter(const float *pts, int n_cols, const int64_t *row_start, long long n_points,
                                    const float *box_prep, const double *centres, const int64_t *box_start,
                                    int n_boxes, int n_frames, const int64_t *starts, float *rows, long long rows_cap,
                                    void *workspace, size_t workspace_bytes, void *stream)
{
    if ((n_boxes > 0 && (!box_prep || !centres)) || rows_cap < 0 || (rows_cap > 0 && !rows)) return FNP_EINVAL;
    const int rc = crop_check(pts, n_cols, row_start, n_points, box_start, n_boxes, n_frames, starts, workspace,
                              workspace_bytes);
    if (rc != FNP_OK) return rc;
    const CropWs ws = crop_carve(workspace, workspace_bytes, n_points, n_boxes, n_frames);
    const long long n_tiles = n_points / kCropTile + n_frames;
    if (n_tiles > 0 && n_boxes > 0 && rows_cap > 0)
        crop_all_scatter_kernel<<<(unsigned)n_tiles, kCropThreads, 0, (cudaStream_t)stream>>>(
            pts, n_cols, row_start, box_prep, centres, box_start, n_frames, ws, starts, rows, rows_cap);
    FNP_LAUNCH_CHECK();
    return FNP_OK;
}

extern "C" int fnp_crop_points_in_boxes(const float *pts, int n_cols, const int64_t *row_start, long long n_points,
                                        const float *boxes, const double *centres, const int64_t *box_start,
                                        int n_boxes, int n_frames, int32_t *counts, int64_t *starts, float *rows,
                                        void *workspace, size_t workspace_bytes, void *stream)
{
    if ((n_boxes > 0 && (!boxes || !centres || !counts)) || (n_points > 0 && n_boxes > 0 && !rows)) return FNP_EINVAL;
    const int rc = crop_check(pts, n_cols, row_start, n_points, box_start, n_boxes, n_frames, starts, workspace,
                              workspace_bytes);
    if (rc != FNP_OK) return rc;
    const long long n_tiles = n_points / kCropTile + n_frames;
    const size_t head = crop_head_bytes(n_points, n_frames);
    cudaStream_t s = (cudaStream_t)stream;
    const CropWs ws = crop_carve(workspace, workspace_bytes, n_points, n_boxes, n_frames);
    const cudaError_t e = cudaMemsetAsync(ws.mat, 0, workspace_bytes - head, s);
    if (e != cudaSuccess) return (int)e;
    crop_plan_kernel<<<1, kCropScanThreads, 0, s>>>(row_start, box_start, n_frames, ws);
    FNP_LAUNCH_CHECK();
    if (n_tiles > 0 && n_boxes > 0)
        crop_assign_kernel<<<(unsigned)n_tiles, kCropThreads, 0, s>>>(pts, n_cols, row_start, boxes, box_start,
                                                                      n_frames, ws);
    FNP_LAUNCH_CHECK();
    if (n_boxes > 0)
        crop_prefix_kernel<<<divup(n_boxes, 128), 128, 0, s>>>(row_start, box_start, n_frames, n_boxes, ws, counts);
    FNP_LAUNCH_CHECK();
    crop_starts_kernel<<<1, kCropScanThreads, 0, s>>>(counts, n_boxes, starts);
    FNP_LAUNCH_CHECK();
    if (n_tiles > 0 && n_boxes > 0)
        crop_scatter_kernel<<<(unsigned)n_tiles, 32, 0, s>>>(pts, n_cols, row_start, centres, box_start, n_frames, ws,
                                                             starts, rows);
    FNP_LAUNCH_CHECK();
    return FNP_OK;
}

extern "C" int fnp_count_in_boxes(const float *pts4, const int32_t *pt_start, const float *boxes,
                                  const int32_t *box_start, int n_segments, int32_t *counts, void *stream)
{
    if (n_segments < 0) return FNP_EINVAL;
    if (n_segments == 0) return FNP_OK;
    if (!pt_start || !box_start || !counts) return FNP_EINVAL;
    // boxes per segment are not known on the host: 32 CTAs per segment, each striding over the segment's boxes
    dim3 grid(n_segments, 32);
    count_segments_kernel<<<grid, kCntThreads, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const float4 *>(pts4), pt_start, boxes, box_start, counts);
    FNP_LAUNCH_CHECK();
    return FNP_OK;
}

template <bool IOU>
static int pairwise(const float *a, const float *b, float *out, int N, int M, void *stream)
{
    if (N < 0 || M < 0) return FNP_EINVAL;
    if (N == 0 || M == 0) return FNP_OK;
    if (!a || !b || !out) return FNP_EINVAL;
    if (divup(N, 16) > 65535) return FNP_EINVAL;
    dim3 grid(divup(M, 16), divup(N, 16));
    pairwise_kernel<IOU><<<grid, 256, 0, (cudaStream_t)stream>>>(a, b, out, N, M);
    FNP_LAUNCH_CHECK();
    return FNP_OK;
}

extern "C" int fnp_boxes_overlap_bev(const float *a, const float *b, float *out, int N, int M, void *stream)
{
    return pairwise<false>(a, b, out, N, M, stream);
}

extern "C" int fnp_boxes_iou_bev(const float *a, const float *b, float *out, int N, int M, void *stream)
{
    return pairwise<true>(a, b, out, N, M, stream);
}

extern "C" int fnp_boxes_aligned_overlap_bev(const float *a, const float *b, float *out, int N, void *stream)
{
    if (N < 0) return FNP_EINVAL;
    if (N == 0) return FNP_OK;
    if (!a || !b || !out) return FNP_EINVAL;
    aligned_overlap_kernel<<<divup(N, 128), 128, 0, (cudaStream_t)stream>>>(a, b, out, N);
    FNP_LAUNCH_CHECK();
    return FNP_OK;
}

extern "C" int fnp_points_in_boxes_matrix(const float *box_prep, const float *pts, int32_t *out, int N, int P, void *stream)
{
    if (N < 0 || P < 0) return FNP_EINVAL;
    if (N == 0 || P == 0) return FNP_OK;
    if (!box_prep || !pts || !out) return FNP_EINVAL;
    if (divup(N, kMatBoxes) > 65535) return FNP_EINVAL;
    dim3 grid(divup(P, kMatThreads), divup(N, kMatBoxes));
    pib_matrix_kernel<<<grid, kMatThreads, 0, (cudaStream_t)stream>>>(box_prep, pts, out, N, P);
    FNP_LAUNCH_CHECK();
    return FNP_OK;
}

extern "C" int fnp_boxes_iou3d(const float *a, const float *b, float *out, int N, int M, void *stream)
{
    if (N < 0 || M < 0) return FNP_EINVAL;
    if (N == 0 || M == 0) return FNP_OK;
    if (!a || !b || !out) return FNP_EINVAL;
    if (divup(N, 16) > 65535) return FNP_EINVAL;
    dim3 grid(divup(M, 16), divup(N, 16));
    pairwise_iou3d_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(a, b, out, N, M);
    FNP_LAUNCH_CHECK();
    return FNP_OK;
}

extern "C" int fnp_boxes_aligned_iou3d(const float *a, const float *b, float *out, int N, void *stream)
{
    if (N < 0) return FNP_EINVAL;
    if (N == 0) return FNP_OK;
    if (!a || !b || !out) return FNP_EINVAL;
    aligned_iou3d_kernel<<<divup(N, 128), 128, 0, (cudaStream_t)stream>>>(a, b, out, N);
    FNP_LAUNCH_CHECK();
    return FNP_OK;
}

extern "C" size_t fnp_nms_workspace_bytes(int N)
{
    if (N <= 0) return 16;
    const size_t cb = (size_t)divup(N, 64);
    return (size_t)N * cb * 8 + (size_t)N * sizeof(RBox) + 64;
}

template <bool ROTATED>
static int nms_impl(const float *boxes, int N, float thresh, int64_t *keep, int32_t *num_keep, void *ws,
                    size_t ws_bytes, void *stream)
{
    if (N < 0 || !num_keep) return FNP_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    if (N == 0) {
        cudaMemsetAsync(num_keep, 0, sizeof(int32_t), st);
        FNP_LAUNCH_CHECK();
        return FNP_OK;
    }
    if (!boxes || !keep || !ws) return FNP_EINVAL;
    if (ws_bytes < fnp_nms_workspace_bytes(N)) return FNP_EWORKSPACE;
    if ((reinterpret_cast<uintptr_t>(ws) & 7) != 0) return FNP_EINVAL;
    const int cb = divup(N, 64);
    if (cb > 65535 || (size_t)cb * 8 > 160 * 1024) return FNP_EINVAL;
    unsigned long long *mask = reinterpret_cast<unsigned long long *>(ws);
    RBox *rb = reinterpret_cast<RBox *>(mask + (size_t)N * cb);
    if (ROTATED) prep_rbox_kernel<<<divup(N, 128), 128, 0, st>>>(boxes, rb, N);
    dim3 grid(cb, cb);
    nms_mask_kernel<ROTATED><<<grid, 64, 0, st>>>(boxes, rb, N, thresh, mask);
    const size_t smem = (size_t)cb * 8;
    if (smem > 48 * 1024)
        cudaFuncSetAttribute(nms_scan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    nms_scan_kernel<<<1, kScanThreads, smem, st>>>(mask, N, keep, num_keep);
    FNP_LAUNCH_CHECK();
    return FNP_OK;
}

extern "C" int fnp_nms_rotated(const float *boxes_sorted, int N, float thresh, int64_t *keep, int32_t *num_keep,
                               void *workspace, size_t workspace_bytes, void *stream)
{
    return nms_impl<true>(boxes_sorted, N, thresh, keep, num_keep, workspace, workspace_bytes, stream);
}

extern "C" int fnp_nms_normal(const float *boxes_sorted, int N, float thresh, int64_t *keep, int32_t *num_keep,
                              void *workspace, size_t workspace_bytes, void *stream)
{
    return nms_impl<false>(boxes_sorted, N, thresh, keep, num_keep, workspace, workspace_bytes, stream);
}

extern "C" int fnp_seg_nms_rotated(const float *boxes, const int32_t *label, const int32_t *order,
                                   const int32_t *valid, const int32_t *seg_start, int n_segments,
                                   int max_seg_boxes, float thresh, uint8_t *keep_mask, void *stream)
{
    if (n_segments < 0 || max_seg_boxes < 0 || max_seg_boxes > FNP_SEG_NMS_MAX) return FNP_EINVAL;
    if (n_segments == 0 || max_seg_boxes == 0) return FNP_OK;
    if (!boxes || !seg_start || !keep_mask) return FNP_EINVAL;
    const int n = max_seg_boxes, cb = divup(n, 64);
    const size_t smem = (size_t)n * sizeof(RBox) + (size_t)n * cb * 8 + (size_t)(n + 2) * 4 + (size_t)cb * 8 + 16;
    cudaFuncSetAttribute(seg_nms_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    seg_nms_kernel<<<n_segments, 256, smem, (cudaStream_t)stream>>>(boxes, label, order, valid, seg_start, thresh, keep_mask);
    FNP_LAUNCH_CHECK();
    return FNP_OK;
}

extern "C" int fnp_recall_counters(const float *pred, const int32_t *pred_valid, const int32_t *pred_start, const float *gt,
                                   const int32_t *gt_start, int n_frames, int max_pred_per_frame, int max_gt_per_frame,
                                   const float *thresh_host, int n_thresh, long long *counters, void *stream)
{
    if (n_frames < 0 || n_thresh < 0 || n_thresh > 8 || max_pred_per_frame < 0 || max_gt_per_frame < 0) return FNP_EINVAL;
    if (n_frames == 0 || max_gt_per_frame == 0) return FNP_OK;
    if (!pred_start || !gt_start || !counters || (n_thresh && !thresh_host)) return FNP_EINVAL;
    float t[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int i = 0; i < n_thresh; i++) t[i] = thresh_host[i];
    const size_t smem = (size_t)(max_pred_per_frame + max_gt_per_frame) * sizeof(RBox) + (size_t)max_gt_per_frame * 4 + 16;
    if (smem > 200 * 1024) return FNP_EINVAL;
    cudaFuncSetAttribute(recall_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    recall_kernel<<<n_frames, 256, smem, (cudaStream_t)stream>>>(pred, pred_valid, pred_start, gt, gt_start, n_thresh, t[0], t[1],
                                                                 t[2], t[3], t[4], t[5], t[6], t[7], counters);
    FNP_LAUNCH_CHECK();
    return FNP_OK;
}

extern "C" int fnp_precision_counters(const float *pred, const int32_t *pred_valid, const int32_t *pred_start, const float *gt,
                                      const int32_t *gt_start, int n_frames, int max_pred_per_frame, int max_gt_per_frame,
                                      const float *thresh_host, int n_thresh, long long *counters, void *stream)
{
    if (n_frames < 0 || n_thresh < 0 || n_thresh > 8 || max_pred_per_frame < 0 || max_gt_per_frame < 0) return FNP_EINVAL;
    if (n_frames == 0 || max_pred_per_frame == 0) return FNP_OK;
    if (!pred || !pred_start || !gt_start || !counters || (n_thresh && !thresh_host) || (max_gt_per_frame && !gt))
        return FNP_EINVAL;
    float t[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int i = 0; i < n_thresh; i++) t[i] = thresh_host[i];
    const size_t smem = (size_t)(max_pred_per_frame + max_gt_per_frame) * sizeof(RBox) + (size_t)max_pred_per_frame * 4 + 16;
    if (smem > 200 * 1024) return FNP_EINVAL;
    cudaFuncSetAttribute(precision_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    precision_kernel<<<n_frames, 256, smem, (cudaStream_t)stream>>>(pred, pred_valid, pred_start, gt, gt_start, n_thresh, t[0],
                                                                    t[1], t[2], t[3], t[4], t[5], t[6], t[7], counters);
    FNP_LAUNCH_CHECK();
    return FNP_OK;
}

extern "C" size_t fnp_quality_smem_bytes(int max_pred_per_frame, int max_gt_per_frame, int n_classes, int n_edges, int n_thresh)
{
    const size_t n_block = (size_t)n_classes * (n_edges + 1) * (1 + 2 * n_thresh);
    return (size_t)max_pred_per_frame * (sizeof(RBox) + 16) + (size_t)max_gt_per_frame * (sizeof(RBox) + 12) + 8 * n_block + 16;
}

extern "C" int fnp_quality_counters(const float *pred, long long pred_setting_stride, const int32_t *pred_valid,
                                    long long valid_setting_stride, const int32_t *pred_label, const int32_t *pred_start,
                                    int n_settings, const float *gt, const int32_t *gt_start, int n_frames,
                                    int max_pred_per_frame, int max_gt_per_frame, int n_classes, const float *range_edges_host,
                                    int n_edges, const float *thresh_host, int n_thresh, long long *counters, void *stream)
{
    if (n_settings < 0 || n_frames < 0 || max_pred_per_frame < 0 || max_gt_per_frame < 0 || pred_setting_stride < 0 ||
        valid_setting_stride < 0)
        return FNP_EINVAL;
    if (n_thresh < 0 || n_thresh > kQualityMaxThresh || n_edges < 0 || n_edges > kQualityMaxBins - 1 || n_classes < 1 ||
        n_classes > kQualityMaxClasses)
        return FNP_EINVAL;
    if ((n_thresh && !thresh_host) || (n_edges && !range_edges_host)) return FNP_EINVAL;
    QualityParams q;
    q.n_thresh = n_thresh; q.n_edges = n_edges; q.n_classes = n_classes;
    for (int i = 0; i < kQualityMaxThresh; i++) q.thr[i] = i < n_thresh ? thresh_host[i] : 0.f;
    for (int i = 0; i < kQualityMaxBins - 1; i++) q.edges[i] = i < n_edges ? range_edges_host[i] : 0.f;
    for (int i = 0; i < n_edges; i++)
        if (!(q.edges[i] > 0.f) || (i && !(q.edges[i] > q.edges[i - 1]))) return FNP_EINVAL;
    const size_t smem = fnp_quality_smem_bytes(max_pred_per_frame, max_gt_per_frame, n_classes, n_edges, n_thresh);
    if (smem > 200 * 1024) return FNP_EINVAL;
    if (n_settings == 0 || n_frames == 0 || (max_pred_per_frame == 0 && max_gt_per_frame == 0)) return FNP_OK;
    if (!pred_start || !gt_start || !counters || (max_pred_per_frame && (!pred || !pred_label)) || (max_gt_per_frame && !gt))
        return FNP_EINVAL;
    const int chunks = divup(n_settings, kQualitySettingsPerCta);
    if (chunks > 65535) return FNP_EINVAL;
    cudaFuncSetAttribute(quality_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    quality_kernel<<<dim3(n_frames, chunks), 256, smem, (cudaStream_t)stream>>>(
        pred, pred_setting_stride, pred_valid, valid_setting_stride, pred_label, pred_start, n_settings, gt, gt_start, q,
        counters);
    FNP_LAUNCH_CHECK();
    return FNP_OK;
}
