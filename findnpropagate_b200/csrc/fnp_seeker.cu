// Fused Greedy Box Seeker stages for sm_100a (B200).  See include/fnp.h for the C ABI and
// DESIGN.md for the data layout and the roofline of each kernel.
//
// What these kernels replace (reference: pcdet/models/dense_heads/frustum_proposals_v1.py):
//   stage 1   :590-613,:812-815   project_to_camera x6 + boolean-mask compaction per 2D box
//   stage 1b  :616-662,:817-845   torch.quantile x3, get_cam_frustum, unprojection, clamp,
//                                 centre line
//   stage 2a  :851-911,:1392-1411 hypothesis grid, softmin front shift, distance/IoU filters
//   stage 2b  :930-932            one points_in_boxes_gpu launch + sum + D2H per hypothesis
//   stage 3   :994-1053           density+IoU score, sort, nms_normal(thresh 1), top-1
#include <cstring>
#include <string>

#include "fnp_common.cuh"

namespace fnp {

constexpr int kCullThreads = 256;                       // one point per thread per sub-tile
constexpr int kCullSubAll = FNP_CULL_TILE / kCullThreads;  // sub-tiles (256 rows) of one CTA tile
constexpr int kCullSub = 4;                                // sub-tiles a thread holds in registers at a time (one pass)
constexpr int kCullPasses = kCullSubAll / kCullSub;        // passes over the tile: all passes share one reservation round
constexpr int kStatsFloats = 40;
static_assert(FNP_CULL_TILE % (kCullThreads * kCullSub) == 0, "tile must be a whole number of passes");

// ======================================================================================
// Frustum point storage: pages.
//   A frustum's points live in pages of FNP_PAGE_POINTS (256) points, SoA inside the page:
//   x[256] | y[256] | z[256] | d[256] (| source row[256] with page_planes == 5), xyz of the *unprojected*
//   point and its camera depth.  Point i of frustum f is slot i & 255 of page page_tab[f][i >> 8].  Pages are
//   handed out from one pool by an atomic cursor while stage 1 runs, so stage 1 needs no counting pass, no
//   scan and no reordering pass: a tile reserves a range of the frustum's point indices with one atomic on
//   the frustum's fill counter and writes its members there.
//   The ORDER of a frustum's points is therefore whatever order the tiles got to it.  Nothing downstream
//   depends on it: the depth quantiles are exact order statistics, the AABB is min/max, the per-hypothesis
//   counts are integer sums -- every output is bit-identical whatever the order (the debug view sorts by
//   source row).  A page of one plane is 1 KB contiguous: x, y, z of a page are one 3 KB TMA bulk copy for
//   the scoring kernels, and (x0,x1) of neighbouring points are one 64-bit shared-memory word, the operand
//   of the packed fp32x2 instructions.
// ======================================================================================
constexpr int kPage = FNP_PAGE_POINTS;
static_assert(kPage == 256, "page = 256 points: the stats kernel's block size, the sweep kernel's chunk");

__device__ __forceinline__ int ld_volatile(const int *p)
{
    int v;
    asm volatile("ld.volatile.global.s32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}

// Page k of frustum f (nullptr: the pool overflowed).  Only for kernels that run AFTER stage 1.
__device__ __forceinline__ const float *page_of(const fnp_seeker_batch &b, int f, int k)
{
    const int pg = b.page_tab[(size_t)f * b.page_tab_stride + k];
    return b.frustum_pts + (size_t)(pg - 1) * (size_t)(b.page_planes * kPage);
}

__device__ __constant__ int kImageOrder[6] = {2, 0, 1, 5, 3, 4};   // frustum_proposals_v1.py:201

constexpr int kCellPx = 64;          // cell edge of the candidate lookup grid, pixels
constexpr float kCellInv = 1.0f / kCellPx;

__host__ __device__ inline int cell_cols(float img_w) { return (int)((img_w + kCellPx - 1) / kCellPx); }
__host__ __device__ inline int cell_rows(float img_h) { return (int)((img_h + kCellPx - 1) / kCellPx); }

// measured on 256 cfg2 frames (profiles/r02g_*): 5 CTAs/SM x 1280 entries 1.29 ms; 4 CTAs 1.49, 6 CTAs (40 registers,
// spills) 1.39, a 768-entry list 1.49 (more tiles take the direct pass), 6 CTAs x 768 entries 1.60
#ifndef FNP_CULL_LIST
#define FNP_CULL_LIST 1280
#endif
#ifndef FNP_CULL_MIN_CTAS
#define FNP_CULL_MIN_CTAS 5
#endif
constexpr int kCullList = FNP_CULL_LIST;      // member entries a tile can hold in shared memory (typical: ~300)

struct alignas(16) CullSmem {
    float cam[6][24];       // by camera index
    int cs[8];              // candidate range per camera RANK, local to the frame: [cs[r], cs[r+1])
    int n_list;             // entries pushed (may exceed kCullList: then the tile takes the direct pass)
    unsigned all_ranks;     // bit r: camera rank r has candidates in this frame
    int pad[2];
    unsigned sect[64];      // the frame's sector table: camera ranks that can see a point of the sector
};
static_assert(sizeof(CullSmem) % 16 == 0, "the float4 tables follow this struct in shared memory");

// --------------------------------------------------------------------------------------
// Azimuth sectors: which cameras can see a point at all.
//   The horizontal plane around the LiDAR is cut into 64 sectors (4 quadrants x 16 steps of the "diamond
//   angle" |y| / (|x| + |y|), which needs no atan).  Per frame a 64-entry table holds, for every sector, the
//   set of camera ranks that can possibly see a point of that sector; the membership pass then projects a
//   point into those cameras only (1-2 instead of 6).  The table is CONSERVATIVE: camera c is dropped from a
//   sector only if no point p of the sector's region
//        R = { rho >= kSecRho0, theta in the sector widened by kSecMargin, |z| <= kSecZ }
//   can pass the exact on-image test, proved with interval bounds on the linear forms wx, wy, wz of
//   lidar2image (in fp64, with a slack kSecSlack that is > 20x the fp32 rounding error of the forms):
//        front of the camera:  sup wx >= -slack, sup (W' wz - wx) >= -slack, sup wy >= -slack,
//                              sup (H' wz - wy) >= -slack, sup wz >= 0              (each is necessary)
//        behind it (depth clamps to 1e-5, so u = wx / 1e-5: a thin tube through the camera centre can still
//        land on the image):  |wx| <= slack, |wy| <= slack feasible and inf wz <= 1.
//   Points outside R (closer than kSecRho0, |z| > kSecZ, non-finite) take all cameras.  A wrong table could
//   only ADD work, never change a result, as long as it is a superset; tests/test_seeker_gpu.py runs stage 1
//   with and without the table on adversarial points (near the cameras, on the tubes, on sector borders).
// --------------------------------------------------------------------------------------
constexpr int kSectors = 64;
constexpr float kSecRho0 = 3.0f, kSecZ = 16.0f;
constexpr double kSecMargin = 0.02, kSecSlack = 1.0;

__device__ __forceinline__ int sector_of(const float x, const float y)
{
    const float ax = fabsf(x), ay = fabsf(y);
    const float q = __fdividef(ay, ax + ay);                      // in [0, 1]; any rounding is far inside kSecMargin
    const int iq = min((int)(q * 16.0f), 15);
    return ((x < 0.f) ? 32 : 0) | ((y < 0.f) ? 16 : 0) | iq;
}

__device__ bool angle_in(double a, double t0, double t1)
{
    const double two_pi = 6.283185307179586;
    double d = fmod(a - t0, two_pi);
    if (d < 0) d += two_pi;
    return d <= t1 - t0;
}

// sup / inf over the sector region of the linear form a x + b y + c z + e
__device__ void form_range(double a, double b, double c, double e, double t0, double t1, double &sup, double &inf)
{
    const double r = hypot(a, b), phi = atan2(b, a);
    const double h0 = a * cos(t0) + b * sin(t0), h1 = a * cos(t1) + b * sin(t1);
    double hmax = fmax(h0, h1), hmin = fmin(h0, h1);
    if (angle_in(phi, t0, t1)) hmax = r;
    if (angle_in(phi + 3.141592653589793, t0, t1)) hmin = -r;
    const double INF = 1e300;
    sup = (hmax > 0 ? INF : (double)kSecRho0 * hmax) + fabs(c) * (double)kSecZ + e;
    inf = (hmin < 0 ? -INF : (double)kSecRho0 * hmin) - fabs(c) * (double)kSecZ + e;
}

__device__ bool sector_sees(const float *__restrict__ L, const int s, const float img_w, const float img_h)
{
    const double PI = 3.141592653589793;
    const int iq = s & 15;
    const double q0 = iq / 16.0, q1 = (iq + 1) / 16.0;
    const double a0 = atan2(q0, 1.0 - q0), a1 = atan2(q1, 1.0 - q1);      // angles of (|x|, |y|), a0 < a1
    double t0, t1;
    switch (s >> 4) {
        case 0: t0 = a0; t1 = a1; break;                 // x >= 0, y >= 0
        case 1: t0 = -a1; t1 = -a0; break;               // x >= 0, y <  0
        case 2: t0 = PI - a1; t1 = PI - a0; break;       // x <  0, y >= 0
        default: t0 = -PI + a0; t1 = -PI + a1; break;    // x <  0, y <  0
    }
    t0 -= kSecMargin; t1 += kSecMargin;
    const double W = (double)img_w * 1.001, H = (double)img_h * 1.001;
    double sup[5], inf[5];
    // forms: wx, wy, wz, W wz - wx, H wz - wy
    const double f[5][4] = {
        {L[0], L[1], L[2], L[3]}, {L[4], L[5], L[6], L[7]}, {L[8], L[9], L[10], L[11]},
        {W * L[8] - L[0], W * L[9] - L[1], W * L[10] - L[2], W * L[11] - L[3]},
        {H * L[8] - L[4], H * L[9] - L[5], H * L[10] - L[6], H * L[11] - L[7]}};
    for (int k = 0; k < 5; k++) {
        if (!(isfinite(f[k][0]) && isfinite(f[k][1]) && isfinite(f[k][2]) && isfinite(f[k][3]))) return true;
        form_range(f[k][0], f[k][1], f[k][2], f[k][3], t0, t1, sup[k], inf[k]);
    }
    const bool front = sup[0] >= -kSecSlack && sup[1] >= -kSecSlack && sup[2] >= 0.0 && sup[3] >= -kSecSlack &&
                       sup[4] >= -kSecSlack;
    const bool back = inf[0] <= kSecSlack && sup[0] >= -kSecSlack && inf[1] <= kSecSlack && sup[1] >= -kSecSlack &&
                      inf[2] <= 1.0;
    return front || back;
}

// One CTA per (frame, camera rank): cell -> candidates of that rank whose box may contain a
// pixel of the cell.  Conservative (a superset); the exact test follows in cull_kernel.
__global__ void __launch_bounds__(128) cell_table_kernel(const fnp_seeker_batch b, const int n_cu, const int n_cv,
                                                         const float img_w, const float img_h, const int kitti)
{
    const int W = b.mask_words;
    extern __shared__ unsigned s_cells[];                 // [n_cu * n_cv][W]
    const int frame = blockIdx.x / 6, r = blockIdx.x % 6;
    const int n_cells = n_cu * n_cv;
    const int c0 = b.frame_cand_start[frame];
    const int lo = b.cam_cand_start[frame * 6 + r] - c0, hi = b.cam_cand_start[frame * 6 + r + 1] - c0;
    unsigned *out = b.cell_masks + ((size_t)frame * 6 + r) * n_cells * W;
    for (int i = threadIdx.x; i < n_cells * W; i += blockDim.x) s_cells[i] = 0u;
    __syncthreads();
    for (int j = lo + threadIdx.x; j < hi; j += blockDim.x) {
        const float4 bx = reinterpret_cast<const float4 *>(b.cand_box2d)[c0 + j];
        if (!(bx.z > bx.x) || !(bx.w > bx.y)) continue;   // empty (or NaN) box: no point can match
        // cell cu covers u in [64 cu, 64 cu + 64); a member has x1 <= u < x2
        int cu0 = max(0, (int)floorf(fmaxf(bx.x, 0.f) * kCellInv));
        int cu1 = min(n_cu - 1, (int)floorf(fminf(bx.z, 65536.f) * kCellInv));
        int cv0 = max(0, (int)floorf(fmaxf(bx.y, 0.f) * kCellInv));
        int cv1 = min(n_cv - 1, (int)floorf(fminf(bx.w, 65536.f) * kCellInv));
        if (kitti) {   // no on-image test in that head: a point beyond the grid looks up the nearest border cell
            cu0 = min(cu0, n_cu - 1); cv0 = min(cv0, n_cv - 1);
            cu1 = max(cu1, 0); cv1 = max(cv1, 0);
        }
        for (int cv = cv0; cv <= cv1; cv++)
            for (int cu = cu0; cu <= cu1; cu++) atomicOr(&s_cells[(cv * n_cu + cu) * W + (j >> 5)], 1u << (j & 31));
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n_cells * W; i += blockDim.x) out[i] = s_cells[i];
    // sector table of the frame (after the cell masks of all frames; zeroed by the host call): bit r of entry s
    if (hi > lo && (int)threadIdx.x < kSectors && !kitti) {
        unsigned *sect = b.cell_masks + (size_t)b.n_frames * 6 * n_cells * W + (size_t)frame * kSectors;
        const float *L = b.cam_mats + ((size_t)frame * 6 + kImageOrder[r]) * 24;
        if (sector_sees(L, threadIdx.x, img_w, img_h)) atomicOr(&sect[threadIdx.x], 1u << r);
    }
}

// wx, wy, wz of two points against one camera: the three rows of lidar2image, each
// fma(a2, z, fma(a1, y, a0 * x)) + a3 as in project(), evaluated on packed pairs (per-lane IEEE).
__device__ __forceinline__ unsigned long long pack2(float lo, float hi)
{
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack2(unsigned long long v, float &lo, float &hi)
{
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ unsigned long long row2(const float *__restrict__ a, unsigned long long x2,
                                                   unsigned long long y2, unsigned long long z2)
{
    unsigned long long t;
    const unsigned long long a0 = pack2(a[0], a[0]), a1 = pack2(a[1], a[1]), a2 = pack2(a[2], a[2]), a3 = pack2(a[3], a[3]);
    asm("{\n .reg .b64 t;\n mul.rn.f32x2 t, %1, %4;\n fma.rn.f32x2 t, %2, %5, t;\n fma.rn.f32x2 t, %3, %6, t;\n"
        " add.rn.f32x2 %0, t, %7;\n}\n"
        : "=l"(t)
        : "l"(a0), "l"(a1), "l"(a2), "l"(x2), "l"(y2), "l"(z2), "l"(a3));
    return t;
}

constexpr int kPtsPerThread = kCullSub;   // a thread owns row (sub * kCullThreads + tid) of every sub-tile

// Writes one member point to slot v of frustum f (global candidate index).  Spins (briefly) if the page
// that holds the slot is being handed out by another tile at this moment.
__device__ __forceinline__ void store_member(const fnp_seeker_batch &b, const int f, const int v, const float X,
                                             const float Y, const float Z, const float d, const int row)
{
    const int *slot_of_page = b.page_tab + (size_t)f * b.page_tab_stride + (v >> 8);
    int pg = ld_volatile(slot_of_page);
    while (pg == 0) pg = ld_volatile(slot_of_page);
    if (pg < 0) return;                       // pool exhausted: the batch is re-run with a larger pool
    float *base = b.frustum_pts + (size_t)(pg - 1) * (size_t)(b.page_planes * kPage) + (v & (kPage - 1));
    base[0] = X; base[kPage] = Y; base[2 * kPage] = Z; base[3 * kPage] = d;
    if (b.page_planes > 4) reinterpret_cast<int *>(base)[4 * kPage] = row;
}

// The membership pass of a tile.  Per camera a division-free "certainly off this image" test on packed
// point pairs, the reference's exact IEEE u, v only for the survivors, one lookup in the camera's cell
// table, exact half-open box tests for the few bits set there.  A member (point, candidate) pair gets its
// rank among the tile's members of that candidate from a shared-memory atomic and
//   DIRECT == false: is appended to the tile's member list (unprojected point, candidate, rank);
//   DIRECT == true : is written to its final place at once (s_base[] = the tile's reservation).
template <bool DIRECT, int W, bool KITTI>
__device__ __forceinline__ void cull_members(const fnp_seeker_batch &b, CullSmem &S, const float4 *s_box, int *s_cnt,
                                             const int *s_base, float4 *s_ent, int *s_key, int *s_row,
                                             const float (&x)[kPtsPerThread], const float (&y)[kPtsPerThread],
                                             const float (&z)[kPtsPerThread], const bool (&live)[kPtsPerThread],
                                             const int frame, const int c0, const int row0, const float img_w,
                                             const float img_h, const int n_cu, const int n_cv, const bool use_sectors,
                                             int *n_list, const int list_cap)
{
    const int tid = threadIdx.x;
    // conservative off-image bounds (see the exactness note in DESIGN.md, stage 1)
    const float w_hi = __fmul_rn(img_w, 1.0001f), h_hi = __fmul_rn(img_h, 1.0001f);
    const int n_cells = n_cu * n_cv;
#pragma unroll
    for (int s = 0; s < kPtsPerThread; s++) {
        // cameras (ranks) that can see this point at all: the frame's sector table, or every rank with candidates
        unsigned cams = 0u;
        if (live[s]) {
            const float rho2 = __fmaf_rn(y[s], y[s], __fmul_rn(x[s], x[s]));
            const bool in_region = use_sectors & (rho2 >= kSecRho0 * kSecRho0) & (rho2 < 1e12f) & (fabsf(z[s]) <= kSecZ);
            cams = in_region ? S.sect[sector_of(x[s], y[s])] : S.all_ranks;
        }
        // the 32 points of a warp's sub-tile are neighbours in the sweep: their camera sets nearly coincide
        unsigned todo = __reduce_or_sync(0xffffffffu, cams);
        while (todo) {
            const int r = __ffs(todo) - 1;
            todo &= todo - 1;
            const float *L = S.cam[kImageOrder[r]];
            float u, v, d;
            int cell;
            if (KITTI) {
                // FrustumProposerOGKITTI: the two-step calibration, no depth clamp, every point "on the image"
                if (!live[s]) continue;
                project_kitti(&S.cam[0][0], x[s], y[s], z[s], u, v, d);
                cell = min(max(__float2int_rz(v * kCellInv), 0), n_cv - 1) * n_cu + min(max(__float2int_rz(u * kCellInv), 0), n_cu - 1);
            } else {
                const float wx = __fadd_rn(dot3(L + 0, x[s], y[s], z[s]), L[3]);
                const float wy = __fadd_rn(dot3(L + 4, x[s], y[s], z[s]), L[7]);
                const float wz = __fadd_rn(dot3(L + 8, x[s], y[s], z[s]), L[11]);
                d = fminf(fmaxf(wz, 1e-5f), 1e5f);
                // cheap, division-free "certainly off this image" test
                const bool off = (wx < -1e-30f) | (wy < -1e-30f) | (wx > __fmul_rn(w_hi, d)) | (wy > __fmul_rn(h_hi, d));
                if (!live[s] | off) continue;
                // exact path: the reference's u, v (IEEE division) and on-image / in-box tests
                u = __fdiv_rn(wx, d); v = __fdiv_rn(wy, d);
                if (!((v < img_h) & (v >= 0.f) & (u < img_w) & (u >= 0.f))) continue;
                cell = min((int)(v * kCellInv), n_cv - 1) * n_cu + min((int)(u * kCellInv), n_cu - 1);
            }
            const unsigned *cm = b.cell_masks + (((size_t)frame * 6 + r) * n_cells + cell) * W;
            bool have = false;
            float X = 0.f, Y = 0.f, Z = 0.f;
#pragma unroll
            for (int w = 0; w < W; w++) {      // W words of the cell's candidate mask (W * 32 >= candidates of the busiest frame)
                unsigned m = __ldg(cm + w);
                while (m) {
                    const int jb = __ffs(m) - 1;
                    m &= m - 1;
                    const int j = 32 * w + jb;
                    const float4 bx = s_box[j];
                    if (!((v < bx.w) & (v >= bx.y) & (u < bx.z) & (u >= bx.x))) continue;
                    if (!have) {     // the reference tests unproject(project(p)) (:812-815): one per (point, camera)
                        if (KITTI) unproject_kitti(&S.cam[0][0], u, v, d, X, Y, Z);
                        else unproject(L + 12, L + 21, u, v, d, X, Y, Z);
                        have = true;
                    }
                    const int rank = atomicAdd(&s_cnt[j], 1);
                    const int row = row0 + s * kCullThreads + tid;
                    if (DIRECT) {
                        store_member(b, c0 + j, s_base[j] + rank, X, Y, Z, d, row);
                    } else {
                        const int e = atomicAdd(n_list, 1);
                        if (e < list_cap) {
                            s_ent[e] = make_float4(X, Y, Z, d);
                            s_key[e] = (j << 16) | rank;
                            s_row[e] = row;
                        }
                    }
                }
            }
        }
    }
}

__device__ __forceinline__ void reserve_range(const fnp_seeker_batch &b, const int f, const int c, int *base_out,
                                              const int n_pages_cap);

// Stage 1 proper: one CTA per 1024-point tile; reads every point ONCE.
//   1. membership pass -> member list in shared memory, per-candidate populations;
//   2. one atomic per (tile, candidate with members) on the frustum's fill counter reserves a range of its
//      point indices; the reservation that contains the first slot of a page takes that page from the pool;
//   3. the list is flushed to the reserved slots by full warps.
// A tile whose members do not fit the list (kCullList) repeats the membership pass with direct writes.
template <int W, bool KITTI>
__global__ void __launch_bounds__(kCullThreads, FNP_CULL_MIN_CTAS) cull_kernel(const fnp_seeker_batch b, const float img_w,
                                                            const float img_h, const int n_cu, const int n_cv,
                                                            const int use_sectors)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    CullSmem &S = *reinterpret_cast<CullSmem *>(smem_raw);
    const int Cmax = b.max_cands_per_frame;
    float4 *s_box = reinterpret_cast<float4 *>(smem_raw + sizeof(CullSmem));            // [Cmax]
    float4 *s_ent = s_box + Cmax;                                                        // [kCullList]
    int *s_key = reinterpret_cast<int *>(s_ent + kCullList);                             // [kCullList]
    int *s_row = s_key + kCullList;                                                      // [kCullList]
    int *s_cnt = s_row + kCullList;                                                      // [Cmax] members of a candidate in this tile
    int *s_base = s_cnt + Cmax;                                                          // [Cmax] first reserved slot

    const int tile = blockIdx.x;
    const int tid = threadIdx.x;
    const int frame = b.tile_frame[tile];
    const int row0 = b.tile_row0[tile];
    const int64_t frow = b.frame_row_start[frame];
    const int frame_rows = (int)(b.frame_row_start[frame + 1] - frow);
    const int c0 = b.frame_cand_start[frame];
    const int nc = b.frame_cand_start[frame + 1] - c0;
    if (nc == 0) return;

    // ---- my points of the first pass (issued first: the loads overlap the per-CTA setup)
    const int stride = b.point_stride;
    float x[kPtsPerThread], y[kPtsPerThread], z[kPtsPerThread];
    bool live[kPtsPerThread];
    auto load_pass = [&](const int pass) {
#pragma unroll
        for (int s = 0; s < kPtsPerThread; s++) {
            const int row = row0 + (pass * kCullSub + s) * kCullThreads + tid;
            live[s] = row < frame_rows;
            x[s] = y[s] = z[s] = 0.f;
            if (live[s]) {
                const float *p = b.points + (size_t)(frow + row) * stride + b.xyz_offset;
                x[s] = __ldg(p); y[s] = __ldg(p + 1); z[s] = __ldg(p + 2);
            }
        }
    };
    load_pass(0);
    // ---- per-CTA setup
    if (tid < 6 * 24) (&S.cam[0][0])[tid] = b.cam_mats[(size_t)frame * 144 + tid];
    for (int j = tid; j < nc; j += kCullThreads) { s_box[j] = reinterpret_cast<const float4 *>(b.cand_box2d)[c0 + j]; s_cnt[j] = 0; }
    if (tid < 7) S.cs[tid] = b.cam_cand_start[frame * 6 + tid] - c0;
    if (tid == 7) S.n_list = 0;
    if (tid >= 32 && tid < 32 + kSectors)
        S.sect[tid - 32] = b.cell_masks[(size_t)b.n_frames * 6 * n_cu * n_cv * W + (size_t)frame * kSectors + (tid - 32)];
    if (tid == 8) {
        unsigned all = 0u;
        for (int r = 0; r < 6; r++)
            if (b.cam_cand_start[frame * 6 + r + 1] > b.cam_cand_start[frame * 6 + r]) all |= 1u << r;
        S.all_ranks = all;
    }
    __syncthreads();

    for (int pass = 0; pass < kCullPasses; pass++) {      // all passes of the tile share one list and one reservation round
        if (pass) load_pass(pass);
        cull_members<false, W, KITTI>(b, S, s_box, s_cnt, s_base, s_ent, s_key, s_row, x, y, z, live, frame, c0,
                               row0 + pass * kCullSub * kCullThreads, img_w, img_h, n_cu, n_cv, use_sectors != 0, &S.n_list, kCullList);
    }
    __syncthreads();
    const int n_list = S.n_list;
    if (n_list == 0) return;

    // ---- reserve slots; hand out the pages whose first slot lies in the reservation
    const int n_pages_cap = (int)(b.pts_capacity / kPage);
    for (int j = tid; j < nc; j += kCullThreads) {
        const int c = s_cnt[j];
        if (c == 0) continue;
        reserve_range(b, c0 + j, c, &s_base[j], n_pages_cap);
    }
    __syncthreads();

    if (n_list <= kCullList) {
        // ---- flush the list: full warps, four 4-byte stores per member
        for (int e = tid; e < n_list; e += kCullThreads) {
            const int key = s_key[e];
            const int j = key >> 16;
            const float4 p = s_ent[e];
            store_member(b, c0 + j, s_base[j] + (key & 0xffff), p.x, p.y, p.z, p.w, s_row[e]);
        }
    } else {
        // ---- more members than the list holds (dense overlapping boxes): repeat the pass with direct writes;
        // the ranks are handed out again, any assignment of a candidate's members to its reserved slots will do
        for (int j = tid; j < nc; j += kCullThreads) s_cnt[j] = 0;
        __syncthreads();
        for (int pass = 0; pass < kCullPasses; pass++) {
            if (kCullPasses > 1) load_pass(pass);
            cull_members<true, W, KITTI>(b, S, s_box, s_cnt, s_base, s_ent, s_key, s_row, x, y, z, live, frame, c0,
                                  row0 + pass * kCullSub * kCullThreads, img_w, img_h, n_cu, n_cv, use_sectors != 0, &S.n_list, kCullList);
        }
    }
}

__device__ __forceinline__ void reserve_range(const fnp_seeker_batch &b, const int f, const int c, int *base_out,
                                              const int n_pages_cap)
{
    const int base = atomicAdd(&b.cand_npts[f], c);
    *base_out = base;
    int *tab = b.page_tab + (size_t)f * b.page_tab_stride;
    for (int k = (base + kPage - 1) / kPage; k * kPage < base + c; k++) {      // pages whose first slot is in the range
        const int pg = atomicAdd(&b.status[5], 1);
        int val = pg + 1;
        if (pg >= n_pages_cap || k >= b.page_tab_stride) { val = -1; atomicOr(&b.status[0], 1); }
        if (k < b.page_tab_stride) atomicExch(&tab[k], val);
    }
}

// After the tiles: pages needed (for the host's retry), overflow flag.
__global__ void cull_finish_kernel(const fnp_seeker_batch b)
{
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        const long long pages = b.status[5];
        b.status[1] = (int)min(pages * (long long)kPage, (long long)0x7fffffff);   // points of capacity needed
        if (pages * kPage > b.pts_capacity) b.status[0] |= 1;
    }
}

// ======================================================================================
// Stage 1b: per-frustum statistics and centre line
// ======================================================================================
__device__ __forceinline__ float warp_min(float v)
{
#pragma unroll
    for (int o = 16; o; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float warp_max(float v)
{
#pragma unroll
    for (int o = 16; o; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// k-th (0-based) and (k+1)-th smallest depth of a frustum, exactly.  Depths are >= 1e-5 > 0, so
// their bit patterns order like the values and everything below is integer arithmetic on
// rel = key - kmin.  Range-normalised MSD radix select: the first 11-bit digit already spreads the
// keys over [kmin, kmax] (2048 bins), a bin with few enough keys is finished by rank counting in
// shared memory, a crowded one is refined by the next 11 bits.  Typical frustum: one histogram
// pass + one collect pass, both from the shared-memory key cache when the frustum fits.
// All threads of the block call this; results are block-uniform.
constexpr int kSelBits = 11, kSelBins = 1 << kSelBits;
constexpr int kSelList = 512;      // keys finished by rank counting
constexpr int kStatsCache = 4096;  // depth keys cached in shared memory
constexpr int kStatsThreads = 256;
#ifndef FNP_STATS_MIN_CTAS
#define FNP_STATS_MIN_CTAS 4      // 64 registers: 4 CTAs per SM (3 at the natural 79 registers: 0.50 -> 0.43 ms per 256 cfg2 frames)
#endif

struct alignas(16) SelSmem {
    unsigned hist[kSelBins];
    unsigned list[kSelList];
    unsigned key[kStatsCache];
    unsigned warp_sum[kStatsThreads / 32];
    unsigned misc[8];   // 0 bin, 1 keys below it, 2 keys in it, 3 next non-empty bin, 4 list fill, 5 min key above, 6/7 results
};

// Calls f(key) for every depth key of the frustum.  Cached frustums (<= kStatsCache points) read the keys
// from shared memory; the few large ones, which set the duration of the whole kernel, stream the depth plane
// of their pages, one point per thread and page, four pages in flight.
struct FrustumPages {
    const int *tab;          // page table row of the frustum
    const float *pool;
    int page_floats;
    __device__ __forceinline__ const float *page(int k) const { return pool + (size_t)(tab[k] - 1) * (size_t)page_floats; }
};

template <typename F>
__device__ __forceinline__ void for_each_key(const FrustumPages &P, const SelSmem &S, bool cached, int n, F f)
{
    const int tid = threadIdx.x, nt = blockDim.x;
    if (cached) {
        for (int i = tid; i < n; i += nt) f(S.key[i]);
        return;
    }
    // thread t: 16-byte vector t & 63 of the depth plane of page k0 + (t >> 6); two such loads in flight
    const int n_pg = (n + kPage - 1) / kPage;
    const int sub = tid >> 6, i4 = (tid & 63) * 4;
    for (int k0 = 0; k0 < n_pg; k0 += 8) {
        float4 c[2];
#pragma unroll
        for (int u = 0; u < 2; u++) {
            const int k = k0 + 4 * u + sub;
            if (k < n_pg && k * kPage + i4 < n) c[u] = __ldg(reinterpret_cast<const float4 *>(P.page(k) + 3 * kPage + i4));
        }
#pragma unroll
        for (int u = 0; u < 2; u++) {
            const int k = k0 + 4 * u + sub, p = k * kPage + i4;
            if (k >= n_pg || p >= n) continue;
            f(__float_as_uint(c[u].x));
            if (p + 1 < n) f(__float_as_uint(c[u].y));
            if (p + 2 < n) f(__float_as_uint(c[u].z));
            if (p + 3 < n) f(__float_as_uint(c[u].w));
        }
    }
}

__device__ void select_pair(const FrustumPages &pts, SelSmem &S, bool cached, int n, int k, unsigned kmin,
                            unsigned kmax, float &v_lo, float &v_hi)
{
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5;
    if (kmin == kmax) { v_lo = v_hi = __uint_as_float(kmin); return; }
    int shift = max(0, (32 - __clz(kmax - kmin)) - kSelBits);   // digit = (rel >> shift) & 2047; level 1: rel >> shift < 2048
    int pshift = 32;          // current set: (rel >> pshift) == (lo_rel >> pshift); 32 = every key
    unsigned lo_rel = 0;
    int rank = k;             // rank of the wanted key inside the current set
    // keys above the current set: the nearest non-empty bin seen so far (nb_*), whose minimum is only
    // needed if the (k+1)-th key is not in the final bin; it is evaluated lazily in a later pass
    bool nb_valid = false;
    unsigned nb_lo = 0;
    int nb_shift = 0;
    unsigned above = 0xffffffffu;
    for (;;) {
        for (int i = tid; i < kSelBins; i += nt) S.hist[i] = 0;
        if (tid == 0) { S.misc[3] = kSelBins; S.misc[4] = 0; S.misc[5] = 0xffffffffu; }
        __syncthreads();
        unsigned my_above = 0xffffffffu;
        for_each_key(pts, S, cached, n, [&](unsigned key) {
            const unsigned rel = key - kmin;
            if (nb_valid && (rel >> nb_shift) == (nb_lo >> nb_shift)) my_above = min(my_above, key);
            if (pshift < 32 && (rel >> pshift) != (lo_rel >> pshift)) return;
            atomicAdd(&S.hist[(rel >> shift) & (kSelBins - 1)], 1u);
        });
        if (nb_valid) {
            my_above = __reduce_min_sync(0xffffffffu, my_above);
            if (lane == 0 && my_above != 0xffffffffu) atomicMin(&S.misc[5], my_above);
        }
        __syncthreads();
        if (nb_valid) { above = min(above, S.misc[5]); nb_valid = false; }
        // ---- locate the bin holding `rank`: 8 bins per thread, block scan of the 256 partial sums
        unsigned c[kSelBins / kStatsThreads], local = 0;
#pragma unroll
        for (int j = 0; j < kSelBins / kStatsThreads; j++) { c[j] = S.hist[tid * (kSelBins / kStatsThreads) + j]; local += c[j]; }
        unsigned inc = local;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned v = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += v;
        }
        if (lane == 31) S.warp_sum[warp] = inc;
        __syncthreads();
        unsigned excl = inc - local;
        for (int w = 0; w < warp; w++) excl += S.warp_sum[w];
        if ((unsigned)rank >= excl && (unsigned)rank < excl + local) {
            unsigned acc = excl;
#pragma unroll
            for (int j = 0; j < kSelBins / kStatsThreads; j++) {
                if ((unsigned)rank >= acc && (unsigned)rank < acc + c[j]) {
                    S.misc[0] = tid * (kSelBins / kStatsThreads) + j;
                    S.misc[1] = acc;
                    S.misc[2] = c[j];
                }
                acc += c[j];
            }
        }
        __syncthreads();
        const unsigned B = S.misc[0], below = S.misc[1], cB = S.misc[2];
        {   // nearest non-empty bin above B: the first one per thread, then per warp, one atomic per warp
            unsigned mine = kSelBins;
#pragma unroll
            for (int j = kSelBins / kStatsThreads - 1; j >= 0; j--) {
                const unsigned bin = tid * (kSelBins / kStatsThreads) + j;
                if (bin > B && c[j]) mine = bin;
            }
            mine = __reduce_min_sync(0xffffffffu, mine);
            if (lane == 0 && mine < (unsigned)kSelBins) atomicMin(&S.misc[3], mine);
        }
        __syncthreads();
        const unsigned Bn = S.misc[3];
        rank -= (int)below;
        const unsigned hi_part = (pshift < 32) ? ((lo_rel >> pshift) << pshift) : 0u;
        const unsigned bin_lo = hi_part | (B << shift);
        const bool has_next = Bn < (unsigned)kSelBins;
        const unsigned next_lo = hi_part | (Bn << shift);
        const bool second_in_bin = (unsigned)(rank + 1) < cB;

        if (shift == 0) {                         // a bin is one exact key
            v_lo = __uint_as_float(kmin + bin_lo);
            if (second_in_bin) v_hi = v_lo;
            else if (has_next) v_hi = __uint_as_float(kmin + next_lo);
            else v_hi = (above != 0xffffffffu) ? __uint_as_float(above) : v_lo;
            __syncthreads();
            return;
        }
        if (cB <= (unsigned)kSelList) {           // finish: collect the bin, rank by counting
            unsigned nmin = 0xffffffffu;
            for_each_key(pts, S, cached, n, [&](unsigned key) {
                const unsigned rel = key - kmin;
                if (pshift < 32 && (rel >> pshift) != (lo_rel >> pshift)) return;
                const unsigned digit = (rel >> shift) & (kSelBins - 1);
                if (digit == B) S.list[atomicAdd(&S.misc[4], 1u)] = key;
                else if (!second_in_bin && has_next && digit == Bn) nmin = min(nmin, key);
            });
            if (!second_in_bin && has_next) {
                nmin = __reduce_min_sync(0xffffffffu, nmin);
                if (lane == 0 && nmin != 0xffffffffu) atomicMin(&S.misc[5], nmin);
            }
            __syncthreads();
            const int m = (int)cB;
            for (int e = tid; e < m; e += nt) {
                const unsigned key = S.list[e];
                int lt = 0, le = 0;
                for (int j = 0; j < m; j++) { const unsigned o = S.list[j]; lt += o < key; le += o <= key; }
                if (lt <= rank && rank < le) S.misc[6] = key;               // same value from every writer
                if (second_in_bin && lt <= rank + 1 && rank + 1 < le) S.misc[7] = key;
            }
            __syncthreads();
            v_lo = __uint_as_float(S.misc[6]);
            if (second_in_bin) v_hi = __uint_as_float(S.misc[7]);
            else if (has_next) v_hi = __uint_as_float(S.misc[5]);
            else v_hi = (above != 0xffffffffu) ? __uint_as_float(above) : v_lo;
            __syncthreads();
            return;
        }
        // ---- refine the crowded bin with the next digit
        if (has_next) { nb_valid = true; nb_lo = next_lo; nb_shift = shift; }
        lo_rel = bin_lo;
        pshift = shift;
        shift = max(0, shift - kSelBits);
        __syncthreads();
    }
}

// Two ranks k1 <= k2 at once, first level only: ONE histogram pass and ONE collect pass serve both (the near and the
// far depth quantile of a frustum).  Returns false -- nothing decided, the caller runs select_pair per rank -- when the
// bins are too crowded to finish by rank counting.  v[0], v[1] = keys of rank k1, k1 + 1; v[2], v[3] = k2, k2 + 1.
__device__ bool select_two(const FrustumPages &pts, SelSmem &S, bool cached, int n, int k1, int k2, unsigned kmin,
                           unsigned kmax, float (&v)[4])
{
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5;
    if (kmin == kmax) { v[0] = v[1] = v[2] = v[3] = __uint_as_float(kmin); return true; }
    const int shift = max(0, (32 - __clz(kmax - kmin)) - kSelBits);
    for (int i = tid; i < kSelBins; i += nt) S.hist[i] = 0;
    unsigned *m2 = S.list + kSelList - 8;      // the second rank's misc[] (the lists stay below this tail)
    if (tid == 0) { S.misc[3] = kSelBins; S.misc[4] = 0; S.misc[5] = 0xffffffffu; m2[3] = kSelBins; m2[4] = 0; m2[5] = 0xffffffffu; }
    __syncthreads();
    for_each_key(pts, S, cached, n, [&](unsigned key) { atomicAdd(&S.hist[((key - kmin) >> shift) & (kSelBins - 1)], 1u); });
    __syncthreads();
    unsigned c[kSelBins / kStatsThreads], local = 0;
#pragma unroll
    for (int j = 0; j < kSelBins / kStatsThreads; j++) { c[j] = S.hist[tid * (kSelBins / kStatsThreads) + j]; local += c[j]; }
    unsigned inc = local;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) S.warp_sum[warp] = inc;
    __syncthreads();
    unsigned excl = inc - local;
    for (int w = 0; w < warp; w++) excl += S.warp_sum[w];
#pragma unroll
    for (int r = 0; r < 2; r++) {
        const unsigned rank = (unsigned)(r ? k2 : k1);
        unsigned *mm = r ? m2 : S.misc;
        if (rank >= excl && rank < excl + local) {
            unsigned acc = excl;
#pragma unroll
            for (int j = 0; j < kSelBins / kStatsThreads; j++) {
                if (rank >= acc && rank < acc + c[j]) { mm[0] = tid * (kSelBins / kStatsThreads) + j; mm[1] = acc; mm[2] = c[j]; }
                acc += c[j];
            }
        }
    }
    __syncthreads();
    const unsigned B1 = S.misc[0], below1 = S.misc[1], c1 = S.misc[2], B2 = m2[0], below2 = m2[1], c2 = m2[2];
#pragma unroll
    for (int r = 0; r < 2; r++) {      // nearest non-empty bin above each
        const unsigned B = r ? B2 : B1;
        unsigned mine = kSelBins;
#pragma unroll
        for (int j = kSelBins / kStatsThreads - 1; j >= 0; j--) {
            const unsigned bin = tid * (kSelBins / kStatsThreads) + j;
            if (bin > B && c[j]) mine = bin;
        }
        mine = __reduce_min_sync(0xffffffffu, mine);
        if (lane == 0 && mine < (unsigned)kSelBins) atomicMin(r ? &m2[3] : &S.misc[3], mine);
    }
    __syncthreads();
    const unsigned Bn1 = S.misc[3], Bn2 = m2[3];
    const int r1 = k1 - (int)below1, r2 = k2 - (int)below2;
    const bool sec1 = (unsigned)(r1 + 1) < c1, sec2 = (unsigned)(r2 + 1) < c2;       // rank + 1 in the same bin
    const bool nx1 = Bn1 < (unsigned)kSelBins, nx2 = Bn2 < (unsigned)kSelBins;
    if (shift == 0) {                          // a bin is one exact key
        v[0] = __uint_as_float(kmin + B1);
        v[1] = sec1 ? v[0] : nx1 ? __uint_as_float(kmin + Bn1) : v[0];
        v[2] = __uint_as_float(kmin + B2);
        v[3] = sec2 ? v[2] : nx2 ? __uint_as_float(kmin + Bn2) : v[2];
        __syncthreads();
        return true;
    }
    const bool same = B1 == B2;
    if ((same ? c1 : c1 + c2) > (unsigned)(kSelList - 16)) { __syncthreads(); return false; }
    // ---- collect: list 1 grows from S.list[0], list 2 (if it is another bin) from S.list[c1]
    unsigned n1 = 0xffffffffu, n2 = 0xffffffffu;
    for_each_key(pts, S, cached, n, [&](unsigned key) {
        const unsigned digit = ((key - kmin) >> shift) & (kSelBins - 1);
        if (digit == B1) S.list[atomicAdd(&S.misc[4], 1u)] = key;
        else if (digit == B2) S.list[c1 + atomicAdd(&m2[4], 1u)] = key;
        if (!sec1 && nx1 && digit == Bn1) n1 = min(n1, key);
        if (!sec2 && nx2 && digit == Bn2) n2 = min(n2, key);
    });
    n1 = __reduce_min_sync(0xffffffffu, n1);
    n2 = __reduce_min_sync(0xffffffffu, n2);
    if (lane == 0 && n1 != 0xffffffffu) atomicMin(&S.misc[5], n1);
    if (lane == 0 && n2 != 0xffffffffu) atomicMin(&m2[5], n2);
    __syncthreads();
#pragma unroll
    for (int r = 0; r < 2; r++) {
        const unsigned *lst = (r && !same) ? S.list + c1 : S.list;
        const int m = (int)((r && !same) ? c2 : c1), rank = r ? r2 : r1;
        const bool sec = r ? sec2 : sec1;
        unsigned *mm = r ? m2 : S.misc;
        for (int e = tid; e < m; e += nt) {
            const unsigned key = lst[e];
            int lt = 0, le = 0;
            for (int j = 0; j < m; j++) { const unsigned o = lst[j]; lt += o < key; le += o <= key; }
            if (lt <= rank && rank < le) mm[6] = key;               // same value from every writer
            if (sec && lt <= rank + 1 && rank + 1 < le) mm[7] = key;
        }
    }
    __syncthreads();
    v[0] = __uint_as_float(S.misc[6]);
    v[1] = sec1 ? __uint_as_float(S.misc[7]) : nx1 ? __uint_as_float(S.misc[5]) : v[0];
    v[2] = __uint_as_float(m2[6]);
    v[3] = sec2 ? __uint_as_float(m2[7]) : nx2 ? __uint_as_float(m2[5]) : v[2];
    __syncthreads();
    return true;
}

// The interpolation of torch.quantile given the two order statistics around the position
__device__ __forceinline__ float quantile_lerp(float a, float bv, float w)
{
    const float diff = __fsub_rn(bv, a);
    return (w < 0.5f) ? __fmaf_rn(w, diff, a) : __fmaf_rn(-diff, __fsub_rn(1.0f, w), bv);
}

// torch.quantile(depth, q), linear interpolation (ATen Sorting.cpp quantile_compute + lerp)
__device__ float block_quantile(const FrustumPages &pts, SelSmem &S, bool cached, int n, float q, float dmin,
                                float dmax)
{
    const float pos = __fmul_rn(q, (float)(n - 1));
    const float lo = floorf(pos), hi = ceilf(pos);
    const float w = __fsub_rn(pos, lo);
    const int klo = (int)lo, khi = (int)hi;
    float a, bv;
    if (khi == 0) { a = dmin; bv = dmin; }
    else if (klo == n - 1) { a = dmax; bv = dmax; }
    else {
        select_pair(pts, S, cached, n, klo, __float_as_uint(dmin), __float_as_uint(dmax), a, bv);
        if (khi == klo) bv = a;
    }
    const float diff = __fsub_rn(bv, a);
    return (w < 0.5f) ? __fmaf_rn(w, diff, a) : __fmaf_rn(-diff, __fsub_rn(1.0f, w), bv);
}

__global__ void __launch_bounds__(kStatsThreads, FNP_STATS_MIN_CTAS) stats_kernel(const fnp_seeker_batch b, const fnp_seeker_cfg cfg)
{
    __shared__ SelSmem S;
    __shared__ float s_red[8][8];
    __shared__ float s_geo[16];  // close[3], vec[3]
    const int f = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n = b.cand_npts[f];
    float *st = b.cand_stats + (size_t)f * kStatsFloats;
    if (n <= 0 || b.status[0] != 0) {
        if (tid == 0) { st[9] = 0.f; }
        return;
    }
    FrustumPages pts;
    pts.tab = b.page_tab + (size_t)f * b.page_tab_stride;
    pts.pool = b.frustum_pts;
    pts.page_floats = b.page_planes * kPage;

    // ---- min / max of depth and of x, y, z.  A page is 4 planes of 64 16-byte vectors: thread t takes vector
    // t & 63 of plane t >> 6 (warps 0-1: x, 2-3: y, 4-5: z, 6-7: depth), four pages in flight per thread.
    const float INF = __int_as_float(0x7f800000);
    float mn[4] = {INF, INF, INF, INF}, mx[4] = {-INF, -INF, -INF, -INF};
    const bool cached = n <= kStatsCache;                         // depth keys stay in shared memory
    const int n_pg = (n + kPage - 1) / kPage;
    {
        const int plane = tid >> 6, i4 = (tid & 63) * 4;
        float lo = INF, hi = -INF;
        for (int k0 = 0; k0 < n_pg; k0 += 4) {
            float4 v[4];
#pragma unroll
            for (int u = 0; u < 4; u++)
                if (k0 + u < n_pg && (k0 + u) * kPage + i4 < n)
                    v[u] = __ldg(reinterpret_cast<const float4 *>(pts.page(k0 + u) + plane * kPage + i4));
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const int p = (k0 + u) * kPage + i4;            // first of the vector's four points
                if (k0 + u >= n_pg || p >= n) continue;
                const float e[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
                if (p + 3 < n) {                                // a whole vector (all but the frustum's last one)
                    lo = fminf(fminf(lo, e[0]), fminf(fminf(e[1], e[2]), e[3]));
                    hi = fmaxf(fmaxf(hi, e[0]), fmaxf(fmaxf(e[1], e[2]), e[3]));
                    if (cached && plane == 3)
                        *reinterpret_cast<uint4 *>(&S.key[p]) = make_uint4(__float_as_uint(e[0]), __float_as_uint(e[1]),
                                                                           __float_as_uint(e[2]), __float_as_uint(e[3]));
                } else {
#pragma unroll
                    for (int c = 0; c < 4; c++)
                        if (p + c < n) {                        // the tail of the last page is not initialised
                            lo = fminf(lo, e[c]); hi = fmaxf(hi, e[c]);
                            if (cached && plane == 3) S.key[p + c] = __float_as_uint(e[c]);
                        }
                }
            }
        }
        lo = warp_min(lo);
        hi = warp_max(hi);
        if (lane == 0) { s_red[warp][0] = lo; s_red[warp][1] = hi; }
    }
    __syncthreads();
#pragma unroll
    for (int a = 0; a < 4; a++) {
        mn[a] = fminf(s_red[2 * a][0], s_red[2 * a + 1][0]);
        mx[a] = fmaxf(s_red[2 * a][1], s_red[2 * a + 1][1]);
    }
    __syncthreads();

    // ---- depth quantiles (frustum_proposals_v1.py:616-648)
    float qmin = 0.f, qmax = 0.f;
    bool both = false;
    if (!(cfg.search_depth > 0.f)) {
        // near and far quantile from one histogram pass and one collect pass when neither is an end of the range
        const float p1 = __fmul_rn(cfg.lq, (float)(n - 1)), p2 = __fmul_rn(cfg.uq, (float)(n - 1));
        const int klo1 = (int)floorf(p1), khi1 = (int)ceilf(p1), klo2 = (int)floorf(p2), khi2 = (int)ceilf(p2);
        if (khi1 != 0 && klo1 != n - 1 && khi2 != 0 && klo2 != n - 1 && klo1 <= klo2) {
            float v[4];
            both = select_two(pts, S, cached, n, klo1, klo2, __float_as_uint(mn[3]), __float_as_uint(mx[3]), v);
            if (both) {
                qmin = quantile_lerp(v[0], khi1 == klo1 ? v[0] : v[1], __fsub_rn(p1, floorf(p1)));
                qmax = quantile_lerp(v[2], khi2 == klo2 ? v[2] : v[3], __fsub_rn(p2, floorf(p2)));
            }
        }
    }
    if (!both) {
        qmin = block_quantile(pts, S, cached, n, cfg.lq, mn[3], mx[3]);
        // search_depth (:619-623): the far end of the frustum is the near quantile + depth
        qmax = (cfg.search_depth > 0.f) ? __fadd_rn(qmin, cfg.search_depth)
                                        : block_quantile(pts, S, cached, n, cfg.uq, mn[3], mx[3]);
    }
    // the centre quantile only feeds weighted_centre_xyz (:631-636), which only the distance term reads
    const bool want_wc = b.hyp_dist != nullptr;
    const float qc = want_wc ? block_quantile(pts, S, cached, n, cfg.cq, mn[3], mx[3]) : 0.f;
    const float dmax = fminf(qmax, cfg.max_dist);
    const float dmin = fmaxf(qmin, cfg.frustum_min);

    if (tid == 0) {
        const int frame = b.cand_frame[f];
        const bool kitti = cfg.variant == FNP_VARIANT_KITTI;
        const float *cm = b.cam_mats + ((size_t)frame * 6 + b.cand_cam[f]) * 24;
        const float *bx = b.cand_box2d + (size_t)f * 4;
        const float lo[3] = {bx[0], bx[1], dmin}, hi[3] = {bx[2], bx[3], dmax};
        const float tpl[8][3] = {{1, 1, -1}, {1, -1, -1}, {-1, -1, -1}, {-1, 1, -1},
                                 {1, 1, 1}, {1, -1, 1}, {-1, -1, 1}, {-1, 1, 1}};
        float c[8][3];
        for (int k = 0; k < 8; k++) {
            float uvd[3];
            for (int a = 0; a < 3; a++) {
                const float whl = __fsub_rn(hi[a], lo[a]);
                const float cen = __fmul_rn(__fadd_rn(hi[a], lo[a]), 0.5f);
                uvd[a] = __fadd_rn(__fmul_rn(whl, tpl[k][a] * 0.5f), cen);
            }
            // KITTI variant: the (8,4)@(4,4) matmul of rect_to_lidar rounds every product on its own (fewer than 33 rows)
            if (kitti) unproject_kitti(b.cam_mats + (size_t)frame * 144, uvd[0], uvd[1], uvd[2], c[k][0], c[k][1], c[k][2], false);
            else unproject(cm + 12, cm + 21, uvd[0], uvd[1], uvd[2], c[k][0], c[k][1], c[k][2]);
        }
        if (cfg.clamp_bottom > 0) {
            for (int a = 0; a < 3; a++) {
                float cmin = c[0][a], cmax = c[0][a];
                for (int k = 1; k < 8; k++) { cmin = fminf(cmin, c[k][a]); cmax = fmaxf(cmax, c[k][a]); }
                const float f1 = fmaxf(mn[a], cmin), f2 = fminf(mx[a], cmax);
                for (int k = 0; k < 8; k++) c[k][a] = fminf(fmaxf(c[k][a], f1), f2);
            }
        }
        for (int a = 0; a < 3; a++) {
            float bev[4];
            for (int i = 0; i < 4; i++) bev[i] = __fmul_rn(__fadd_rn(c[2 * i][a], c[2 * i + 1][a]), 0.5f);
            const float close = __fmul_rn(__fadd_rn(bev[0], bev[1]), 0.5f);
            const float far = __fmul_rn(__fadd_rn(bev[2], bev[3]), 0.5f);
            s_geo[a] = close;
            s_geo[3 + a] = __fsub_rn(far, close);
        }
        if (cfg.search_depth > 0.f) {   // :841-842  center_vec / center_vec.norm() * search_depth
            const float nv = norm3(s_geo[3], s_geo[4], s_geo[5]);
            for (int a = 0; a < 3; a++) s_geo[3 + a] = __fmul_rn(__fdiv_rn(s_geo[3 + a], nv), cfg.search_depth);
        }
        // weighted_centre_xyz (:631-636): the 2D box centre at the cq depth quantile, unprojected
        if (want_wc) {
            const float uc = __fmul_rn(__fadd_rn(bx[0], bx[2]), 0.5f), vc = __fmul_rn(__fadd_rn(bx[1], bx[3]), 0.5f);
            if (kitti) unproject_kitti(b.cam_mats + (size_t)frame * 144, uc, vc, qc, st[10], st[11], st[12], false);
            else unproject(cm + 12, cm + 21, uc, vc, qc, st[10], st[11], st[12]);
        }
        st[0] = dmin; st[1] = dmax; st[2] = qc;
        for (int a = 0; a < 3; a++) { st[3 + a] = mn[a]; st[6 + a] = mx[a]; }
        st[9] = (float)n;
        for (int k = 0; k < 8; k++)
            for (int a = 0; a < 3; a++) st[16 + k * 3 + a] = c[k][a];
    }
    __syncthreads();
    const int M = cfg.num_mags;
    for (int i = tid; i < M * 3; i += blockDim.x) {
        const int m = i / 3, a = i % 3;
        b.centres[((size_t)f * M + m) * 3 + a] = __fadd_rn(s_geo[a], __fmul_rn(s_geo[3 + a], b.mags[m]));
    }
}

// ======================================================================================
// Stage 2a: hypotheses
// ======================================================================================
// 2D IoU of the image-plane bounding box of the 8 shifted corners with a 2D box (calc_iou, :1392-1411)
template <bool KITTI = false>
__device__ __forceinline__ float view_iou(const float *__restrict__ L, const float4 box2d, const float (&cor)[8][3],
                                          const float (&shift)[3], const float img_w, const float img_h)
{
    const float area2 = __fmul_rn(__fsub_rn(box2d.z, box2d.x), __fsub_rn(box2d.w, box2d.y));
    const float INF = __int_as_float(0x7f800000);
    float x1 = INF, y1 = INF, x2 = -INF, y2 = -INF;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        float u, v, d;
        if (KITTI)
            project_kitti(L, __fadd_rn(cor[k][0], shift[0]), __fadd_rn(cor[k][1], shift[1]), __fadd_rn(cor[k][2], shift[2]), u, v, d);
        else
            project(L, __fadd_rn(cor[k][0], shift[0]), __fadd_rn(cor[k][1], shift[1]),
                    __fadd_rn(cor[k][2], shift[2]), img_w, img_h, u, v, d);
        u = fminf(fmaxf(u, 0.f), img_w);
        v = fminf(fmaxf(v, 0.f), img_h);
        x1 = fminf(x1, u); x2 = fmaxf(x2, u); y1 = fminf(y1, v); y2 = fmaxf(y2, v);
    }
    const float area1 = __fmul_rn(__fsub_rn(x2, x1), __fsub_rn(y2, y1));
    const float lx = fmaxf(x1, box2d.x), ly = fmaxf(y1, box2d.y);
    const float rx = fminf(x2, box2d.z), ry = fminf(y2, box2d.w);
    const float iw = fmaxf(__fsub_rn(rx, lx), 0.f), ih = fmaxf(__fsub_rn(ry, ly), 0.f);
    const float inter = __fmul_rn(iw, ih);
    const float uni = __fsub_rn(__fadd_rn(area1, area2), inter);
    return __fdiv_rn(inter, uni);
}

// EXTRAS = false is the shipped configuration (single-view IoU, no hyp_dist): the optional terms are
// compiled out so that they cost the hot path no registers.
// the shipped instance at 64 registers (8 CTAs per SM, 32 B of spills): 0.448 -> 0.429 ms per 256 cfg2 frames; 7 CTAs 0.435,
// 5 CTAs 0.489 (profiles/r02u_ab_hypotheses_occupancy.txt)
#ifndef FNP_HYP_MIN_CTAS
#define FNP_HYP_MIN_CTAS 8
#endif
template <bool EXTRAS, bool KITTI = false>
__global__ void __launch_bounds__(128, EXTRAS ? 4 : FNP_HYP_MIN_CTAS) hypotheses_kernel(const fnp_seeker_batch b, const fnp_seeker_cfg cfg)
{
    __shared__ int s_wcnt[4];
    __shared__ int s_base;
    __shared__ float s_dmm[4][2];
    const int f = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int J = cfg.num_yaw_size, M = cfg.num_mags, H = J * M;
    const bool empty = (b.cand_npts[f] <= 0) || (b.status[0] != 0);
    if (empty) {
        if (tid == 0) b.hyp_nvalid[f] = 0;
        if (b.hyp_valid_dbg)
            for (int h = tid; h < H; h += blockDim.x) b.hyp_valid_dbg[(size_t)f * H + h] = 0;
        return;
    }
    const int frame = b.cand_frame[f];
    const int label = b.cand_label[f];
    const float *L = b.cam_mats + ((size_t)frame * 6 + b.cand_cam[f]) * 24;
    const float4 box2d = reinterpret_cast<const float4 *>(b.cand_box2d)[f];
    const bool multicam = EXTRAS && (cfg.flags & FNP_SEEKER_MULTICAM_IOU) != 0;
    const int fc0 = b.frame_cand_start[frame], fc1 = b.frame_cand_start[frame + 1];
    const bool want_dist = EXTRAS && b.hyp_dist != nullptr;
    float wc[3] = {0.f, 0.f, 0.f};
    if (want_dist) {
        const float *st = b.cand_stats + (size_t)f * kStatsFloats;
        wc[0] = st[10]; wc[1] = st[11]; wc[2] = st[12];
    }
    float dist_mn = __int_as_float(0x7f800000), dist_mx = -__int_as_float(0x7f800000);
    const float *bb_tab = b.base_boxes + (size_t)(label - 1) * J * 7;
    const float *bc_tab = b.base_corners + (size_t)(label - 1) * J * 24;
    if (tid == 0) s_base = 0;
    __syncthreads();

    for (int h0 = 0; h0 < H; h0 += blockDim.x) {
        const int h = h0 + tid;
        bool valid = false;
        float box[7] = {0, 0, 0, 0, 0, 0, 0};
        float iou = 0.f, dist = 0.f;
        if (h < H) {
            const int m = h / J, j = h - m * J;
            const float *ct = b.centres + ((size_t)f * M + m) * 3;
            const float *bc = bc_tab + (size_t)j * 24;
            const float *bb = bb_tab + (size_t)j * 7;
            const float ctr[3] = {ct[0], ct[1], ct[2]};
            float cor[8][3], e[8];
            float mxn = -__int_as_float(0x7f800000);
#pragma unroll
            for (int k = 0; k < 8; k++) {
#pragma unroll
                for (int a = 0; a < 3; a++) cor[k][a] = __fadd_rn(__ldg(bc + k * 3 + a), ctr[a]);
                e[k] = -norm3(cor[k][0], cor[k][1], cor[k][2]);
                mxn = fmaxf(mxn, e[k]);
            }
            float sum = 0.f;
#pragma unroll
            for (int k = 0; k < 8; k++) { e[k] = fnp_exp(__fsub_rn(e[k], mxn)); sum = __fadd_rn(sum, e[k]); }
            float front[3] = {0.f, 0.f, 0.f};
#pragma unroll
            for (int k = 0; k < 8; k++) {
                const float w = __fdiv_rn(e[k], sum);
#pragma unroll
                for (int a = 0; a < 3; a++) front[a] = __fadd_rn(front[a], __fmul_rn(w, cor[k][a]));
            }
            float shift[3];
#pragma unroll
            for (int a = 0; a < 3; a++) {
                const float cc = __fadd_rn(__ldg(bb + a), ctr[a]);
                shift[a] = __fsub_rn(cc, front[a]);
                box[a] = __fadd_rn(cc, shift[a]);
            }
#pragma unroll
            for (int a = 3; a < 7; a++) box[a] = __ldg(bb + a);
            const bool near_enough = norm3(front[0], front[1], front[2]) < cfg.max_dist;
            if (!multicam) iou = view_iou<KITTI>(L, box2d, cor, shift, cfg.img_w, cfg.img_h);
            else {
                // multicam_ious (:1413-1429): every candidate of the frame with points and the same label
                // (this one included), summed in candidate order, over (number of non-zero IoUs + 1e-6)
                float sum_iou = 0.f;
                int nz = 0;
                for (int i = fc0; i < fc1; i++) {
                    if (b.cand_label[i] != label || b.cand_npts[i] <= 0) continue;
                    const float vi = view_iou(b.cam_mats + ((size_t)frame * 6 + b.cand_cam[i]) * 24,
                                              reinterpret_cast<const float4 *>(b.cand_box2d)[i], cor, shift,
                                              cfg.img_w, cfg.img_h);
                    sum_iou = __fadd_rn(sum_iou, vi);
                    nz += vi > 0.f;
                }
                iou = __fdiv_rn(sum_iou, __fadd_rn((float)nz, 1e-6f));
            }
            if (want_dist) {   // torch.cdist(front, weighted_centre_xyz) (:889), evaluated directly
                dist = norm3(__fsub_rn(front[0], wc[0]), __fsub_rn(front[1], wc[1]), __fsub_rn(front[2], wc[2]));
                if (near_enough) { dist_mn = fminf(dist_mn, dist); dist_mx = fmaxf(dist_mx, dist); }
            }
            valid = near_enough && (iou > cfg.min_cam_iou);
            if (b.hyp_boxes_dbg) {
                float *o = b.hyp_boxes_dbg + ((size_t)f * H + h) * 7;
#pragma unroll
                for (int a = 0; a < 7; a++) o[a] = box[a];
            }
            if (b.hyp_iou_dbg) b.hyp_iou_dbg[(size_t)f * H + h] = iou;
            if (b.hyp_valid_dbg) b.hyp_valid_dbg[(size_t)f * H + h] = valid ? 1 : 0;
        }
        // ordered compaction of the valid hypotheses
        const unsigned mk = __ballot_sync(0xffffffffu, valid);
        if (lane == 0) s_wcnt[warp] = __popc(mk);
        __syncthreads();
        int base = s_base;
        for (int w = 0; w < warp; w++) base += s_wcnt[w];
        if (valid) {
            const int r = base + __popc(mk & ((1u << lane) - 1u));
            const BoxPrep p = prep_box(box);
            float4 *dst = reinterpret_cast<float4 *>(b.hyp_prep + ((size_t)f * H + r) * 8);
            dst[0] = make_float4(p.cx, p.cy, p.cz, p.hz);
            dst[1] = make_float4(p.cosa, p.sina, p.tx, p.ty);
            b.hyp_index[(size_t)f * H + r] = h;
            b.hyp_iou[(size_t)f * H + r] = iou;
            if (want_dist) b.hyp_dist[(size_t)f * H + r] = dist;
        }
        __syncthreads();
        if (tid == 0) s_base = base + s_wcnt[0] + s_wcnt[1] + s_wcnt[2] + s_wcnt[3];
        __syncthreads();
    }
    if (tid == 0) b.hyp_nvalid[f] = s_base;
    if (want_dist) {   // dists_ranked is normalised over the hypotheses within max_dist (:891)
        dist_mn = warp_min(dist_mn);
        dist_mx = warp_max(dist_mx);
        if (lane == 0) { s_dmm[warp][0] = dist_mn; s_dmm[warp][1] = dist_mx; }
        __syncthreads();
        if (tid == 0) {
            float *st = b.cand_stats + (size_t)f * kStatsFloats;
            st[13] = fminf(fminf(s_dmm[0][0], s_dmm[1][0]), fminf(s_dmm[2][0], s_dmm[3][0]));
            st[14] = fmaxf(fmaxf(s_dmm[0][1], s_dmm[1][1]), fmaxf(s_dmm[2][1], s_dmm[3][1]));
        }
    }
}

// ======================================================================================
// Stage 2b: scoring -- per-hypothesis point counts
// ======================================================================================
constexpr int kScoreThreads = 128;
constexpr int kScoreTile = 512;  // points per TMA stage (8 KB)

constexpr int kScoreKMax = 4;                                   // hypotheses per thread in a full chunk
constexpr int kScoreChunk = kScoreThreads * kScoreKMax;         // hypotheses of a full chunk

// The nv valid hypotheses of a frustum are cut into nv / 512 full chunks (4 per thread) and one
// remainder chunk of ceil(rem / 128) per thread, so that the padding stays below 128 hypotheses
// per frustum (with 512-wide chunks only, the padded work was 1.42x the useful work on cfg2).
__host__ __device__ inline int score_chunks(int nv) { return (nv + kScoreChunk - 1) / kScoreChunk; }

// Work items of the scoring stage.  Frustum f with P_f points and nv_f valid hypotheses is cut
// into S_f = ceil(P_f / split_points) point splits x score_chunks(nv_f) hypothesis
// chunks; every (split, chunk) pair is one CTA-sized item, so the largest frustums no longer
// set the kernel's duration.  A thread keeps its counts in registers for the whole item and adds
// them to row f of `counts` with one integer RED per hypothesis at the end (integer addition is
// associative: the totals do not depend on the order in which the splits finish).
__global__ void __launch_bounds__(1024) plan_items_kernel(const fnp_seeker_batch b, const int H, const int sweep)
{
    __shared__ int s_warp_i[32];
    __shared__ int s_carry_i;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_carry_i = 0;
    __syncthreads();
    for (int base = 0; base < b.n_cands; base += 1024) {
        const int f = base + tid;
        int items = 0;
        if (f < b.n_cands) {
            const int np = b.cand_npts[f], nv = b.hyp_nvalid[f];
            if (np > 0 && nv > 0) items = ((np + b.split_points - 1) / b.split_points) * (sweep ? 1 : score_chunks(nv));
        }
        int inc_i = items;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int a = __shfl_up_sync(0xffffffffu, inc_i, o);
            if (lane >= o) inc_i += a;
        }
        if (lane == 31) s_warp_i[warp] = inc_i;
        __syncthreads();
        if (warp == 0) {
            int wi = s_warp_i[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int a = __shfl_up_sync(0xffffffffu, wi, o);
                if (lane >= o) wi += a;
            }
            s_warp_i[lane] = wi;
        }
        __syncthreads();
        const int ci = s_carry_i;
        if (f < b.n_cands) b.cand_item_start[f] = ci + (warp ? s_warp_i[warp - 1] : 0) + inc_i - items;
        __syncthreads();
        if (tid == 1023) s_carry_i = ci + s_warp_i[31];
        __syncthreads();
    }
    if (tid == 0) {
        b.cand_item_start[b.n_cands] = s_carry_i;
        b.status[2] = s_carry_i;
        b.status[3] = 0;
        b.status[4] = 0;            // work-item counter of the persistent scoring CTAs
        if (s_carry_i > b.max_items) b.status[0] |= 2;
    }
}

__global__ void __launch_bounds__(128) write_items_kernel(const fnp_seeker_batch b, const int H, const int sweep)
{
    const int f = blockIdx.x;
    const int i0 = b.cand_item_start[f], n = b.cand_item_start[f + 1] - i0;
    if (n <= 0 || (b.status[0] & 2)) return;
    const int nv = b.hyp_nvalid[f];
    const int nchunks = sweep ? 1 : score_chunks(nv);   // the sweep kernel takes all hypotheses of a split at once
    for (int i = threadIdx.x; i < n; i += blockDim.x) {   // split-major: neighbours share a point tile
        const int c = i % nchunks;
        const int left = nv - c * kScoreChunk;             // hypotheses from this chunk's base on
        const int K = left >= kScoreChunk ? kScoreKMax : (left + kScoreThreads - 1) / kScoreThreads;
        reinterpret_cast<int4 *>(b.items)[i0 + i] = make_int4(f, c * kScoreChunk, i / nchunks, K);
    }
}

// Packed-fp32x2 form of the in-box predicate for TWO points against one hypothesis.  Same
// arithmetic per lane as in_box() (sub.rn, mul.rn, fma.rn are IEEE per lane):
//   sx = x - cx, sy = y - cy, sz = z - cz, lx = fma(sx, cosa, rn(sy * -sina)),
//   ly = fma(sy, cosa, rn(sx * sina)), inside = !(|sz| > hz) & |lx| <= tx & |ly| <= ty.
// 7 packed FP instructions (FADD2 x3, FMUL2 x2, FFMA2 x2) + 6 FSETP + 2 predicated IADD per
// two tests, instead of 14 + 6 + 2.
struct HypPacked {
    unsigned long long cx2, cy2, cz2, cosa2, nsina2, sina2;   // each value duplicated in both halves
    float hz, tx, ty;
};

__device__ __forceinline__ unsigned long long dup2(float v)
{
    unsigned long long r;
    asm("mov.b64 %0, {%1, %1};" : "=l"(r) : "f"(v));
    return r;
}

__device__ __forceinline__ float lo_half(unsigned long long v) { return __uint_as_float((unsigned)v); }

__device__ __forceinline__ void count_pair(int &cnt, unsigned long long xx, unsigned long long yy,
                                           unsigned long long zz, const HypPacked &h)
{
    asm("{\n"
        " .reg .b64 sx, sy, sz, m1, m2, lx, ly;\n"
        " .reg .f32 a0, a1, b0, b1, c0, c1;\n"
        " .reg .pred p, q;\n"
        " sub.rn.f32x2 sx, %1, %4;\n"
        " sub.rn.f32x2 sy, %2, %5;\n"
        " sub.rn.f32x2 sz, %3, %6;\n"
        " mul.rn.f32x2 m1, sy, %8;\n"
        " mul.rn.f32x2 m2, sx, %9;\n"
        " fma.rn.f32x2 lx, sx, %7, m1;\n"
        " fma.rn.f32x2 ly, sy, %7, m2;\n"
        " mov.b64 {a0, a1}, lx;\n"
        " mov.b64 {b0, b1}, ly;\n"
        " mov.b64 {c0, c1}, sz;\n"
        " abs.f32 a0, a0;\n abs.f32 a1, a1;\n abs.f32 b0, b0;\n abs.f32 b1, b1;\n abs.f32 c0, c0;\n abs.f32 c1, c1;\n"
        " setp.leu.f32 p, c0, %10;\n"
        " setp.le.and.f32 p, a0, %11, p;\n"
        " setp.le.and.f32 p, b0, %12, p;\n"
        " setp.leu.f32 q, c1, %10;\n"
        " setp.le.and.f32 q, a1, %11, q;\n"
        " setp.le.and.f32 q, b1, %12, q;\n"
        " @p add.s32 %0, %0, 1;\n"
        " @q add.s32 %0, %0, 1;\n"
        "}\n"
        : "+r"(cnt)
        : "l"(xx), "l"(yy), "l"(zz), "l"(h.cx2), "l"(h.cy2), "l"(h.cz2), "l"(h.cosa2), "l"(h.nsina2), "l"(h.sina2),
          "f"(h.hz), "f"(h.tx), "f"(h.ty));
}

// Persistent CTAs pull (frustum, hypothesis chunk, point split) work items off a device
// counter.  A CTA keeps K hypotheses per thread in registers for the whole item and streams
// the item's points through a two-stage shared-memory ring filled by TMA bulk copies
// (cp.async.bulk + mbarrier complete_tx): the x, y, z planes of a page are 3 KB contiguous, one
// copy per page; every thread reads every staged point pair with broadcast LDS.64.
constexpr int kScorePages = kScoreTile / kPage;      // pages per TMA stage
struct ScoreSmem {
    float tile[2][kScorePages][3][kPage];   // [stage][page][x | y | z][slot]
    uint64_t bar[2];
    int item;
};

template <int K>
__device__ __forceinline__ void score_item(const fnp_seeker_batch &b, const int H, ScoreSmem &S, unsigned &it,
                                           const int f, const int h_base, const int split)
{
    const int tid = threadIdx.x;
    const int nv = b.hyp_nvalid[f];
    const int npts = b.cand_npts[f];
    const int p0 = split * b.split_points;                    // a multiple of the page size
    const int n = min(npts, p0 + b.split_points) - p0;
    const int n_tiles = (n + kScoreTile - 1) / kScoreTile;
    const int *tab = b.page_tab + (size_t)f * b.page_tab_stride + p0 / kPage;
    const size_t page_floats = (size_t)b.page_planes * kPage;

    auto issue = [&](int t) {      // one thread: the pages of tile t into stage (it + t) & 1
        const int pages = min(kScorePages, (n - t * kScoreTile + kPage - 1) / kPage);
        const unsigned st = (it + t) & 1u;
        mbar_expect_tx(&S.bar[st], (uint32_t)pages * 3u * kPage * 4u);
        for (int q = 0; q < pages; q++)
            tma_load_1d(S.tile[st][q], b.frustum_pts + (size_t)(tab[t * kScorePages + q] - 1) * page_floats, 3u * kPage * 4u,
                        &S.bar[st]);
    };
    if (tid == 0)
        for (int t = 0; t < 2 && t < n_tiles; t++) issue(t);

    HypPacked hp[K];
    int cnt[K];
#pragma unroll
    for (int k = 0; k < K; k++) {
        const int r = h_base + k * kScoreThreads + tid;
        cnt[k] = 0;
        float4 a = make_float4(0.f, 0.f, 0.f, -1.f), c = make_float4(1.f, 0.f, -1.f, -1.f);   // never inside
        if (r < nv) {
            const float4 *src = reinterpret_cast<const float4 *>(b.hyp_prep + ((size_t)f * H + r) * 8);
            a = __ldg(src); c = __ldg(src + 1);
        }
        hp[k].cx2 = dup2(a.x); hp[k].cy2 = dup2(a.y); hp[k].cz2 = dup2(a.z); hp[k].hz = a.w;
        hp[k].cosa2 = dup2(c.x); hp[k].nsina2 = dup2(-c.y); hp[k].sina2 = dup2(c.y);
        hp[k].tx = c.z; hp[k].ty = c.w;
    }

    for (int t = 0; t < n_tiles; t++) {
        const unsigned st = (it + t) & 1u;
        mbar_wait(&S.bar[st], ((it + t) >> 1) & 1u);
        const int m_tile = min(kScoreTile, n - t * kScoreTile);   // points in this tile
        for (int q = 0; q * kPage < m_tile; q++) {
            const int m_pts = min(kPage, m_tile - q * kPage);
            const int m_full = m_pts >> 1;                         // complete pairs
            const unsigned long long *xs = reinterpret_cast<const unsigned long long *>(S.tile[st][q][0]);
            const unsigned long long *ys = reinterpret_cast<const unsigned long long *>(S.tile[st][q][1]);
            const unsigned long long *zs = reinterpret_cast<const unsigned long long *>(S.tile[st][q][2]);
            int i = 0;
            for (; i + 2 <= m_full; i += 2) {
                const unsigned long long x0 = xs[i], y0 = ys[i], z0 = zs[i];
                const unsigned long long x1 = xs[i + 1], y1 = ys[i + 1], z1 = zs[i + 1];
#pragma unroll
                for (int k = 0; k < K; k++) {
                    count_pair(cnt[k], x0, y0, z0, hp[k]);
                    count_pair(cnt[k], x1, y1, z1, hp[k]);
                }
            }
            for (; i < m_full; i++) {
                const unsigned long long x0 = xs[i], y0 = ys[i], z0 = zs[i];
#pragma unroll
                for (int k = 0; k < K; k++) count_pair(cnt[k], x0, y0, z0, hp[k]);
            }
            if (m_pts & 1) {   // last point of the frustum
                const float px = S.tile[st][q][0][m_pts - 1], py = S.tile[st][q][1][m_pts - 1], pz = S.tile[st][q][2][m_pts - 1];
#pragma unroll
                for (int k = 0; k < K; k++) {
                    BoxPrep bp;
                    bp.cx = lo_half(hp[k].cx2); bp.cy = lo_half(hp[k].cy2); bp.cz = lo_half(hp[k].cz2);
                    bp.cosa = lo_half(hp[k].cosa2); bp.sina = lo_half(hp[k].sina2);
                    bp.hz = hp[k].hz; bp.tx = hp[k].tx; bp.ty = hp[k].ty;
                    count_if(cnt[k], in_box(px, py, pz, bp));
                }
            }
        }
        __syncthreads();  // everyone is done with stage st
        if (tid == 0 && t + 2 < n_tiles) issue(t + 2);
    }
    it += (unsigned)n_tiles;

    int *out = b.counts + (size_t)f * H;
#pragma unroll
    for (int k = 0; k < K; k++) {
        const int r = h_base + k * kScoreThreads + tid;
        if (r < nv && cnt[k]) atomicAdd(out + r, cnt[k]);      // RED.ADD, result unused
    }
}

__global__ void __launch_bounds__(kScoreThreads) score_kernel(const fnp_seeker_batch b, const int H)
{
    __shared__ __align__(128) ScoreSmem S;

    const int tid = threadIdx.x;
    if (b.status[0] & 2) return;
    const int n_items = b.status[2];
    if (tid == 0) {
        mbar_init(&S.bar[0], 1);
        mbar_init(&S.bar[1], 1);
        mbar_fence_init();
    }
    unsigned it = 0;   // tiles consumed so far by this CTA: stage = it & 1, parity = (it >> 1) & 1

    for (;;) {
        __syncthreads();                       // everyone is done with the previous item (and S.item)
        if (tid == 0) S.item = atomicAdd(&b.status[4], 1);
        __syncthreads();
        const int item_id = S.item;
        if (item_id >= n_items) break;
        const int4 item = reinterpret_cast<const int4 *>(b.items)[item_id];   // frustum, first hypothesis, split, K
        switch (item.w) {
            case 1: score_item<1>(b, H, S, it, item.x, item.y, item.z); break;
            case 2: score_item<2>(b, H, S, it, item.x, item.y, item.z); break;
            case 3: score_item<3>(b, H, S, it, item.x, item.y, item.z); break;
            default: score_item<4>(b, H, S, it, item.x, item.y, item.z); break;
        }
    }
}

// ======================================================================================
// Stage 2b, sweep mode: per-hypothesis point counts without testing every pair
// ======================================================================================
// Arithmetic and derivation: fnp_sweep.cuh (shared with the host model tools/sweep_model.cu).
// One CTA per frustum: line fit + deviation of every column.  Dynamic shared memory: 15 J words.
__global__ void __launch_bounds__(128) sweep_prep_kernel(const fnp_seeker_batch b, const int J, const int M)
{
    extern __shared__ int s_raw[];
    int *s_first = s_raw;                                  // [J]
    int *s_last = s_raw + J;                               // [J]
    int *s_r0 = s_raw + 2 * J;                             // [J] compacted slot of the column's first valid step
    float *s_c0 = reinterpret_cast<float *>(s_raw + 3 * J);   // [J][3]
    float *s_c1 = s_c0 + 3 * J;                            // [J][3], later the slopes
    unsigned *s_dev = reinterpret_cast<unsigned *>(s_c1 + 3 * J);   // [J][3] max of C - line (float bits, >= 0)
    unsigned *s_den = s_dev + 3 * J;                                // [J][3] max of line - C
    __shared__ unsigned s_maxabs, s_maxabs_z;
    const int f = blockIdx.x, tid = threadIdx.x;
    const int H = J * M;
    const int nv = b.hyp_nvalid[f];
    SweepCol *out = reinterpret_cast<SweepCol *>(b.sweep_cols) + (size_t)f * J;
    for (int j = tid; j < J; j += blockDim.x) {
        s_first[j] = 0x7fffffff;
        s_last[j] = -1;
        s_dev[3 * j] = s_dev[3 * j + 1] = s_dev[3 * j + 2] = 0u;
        s_den[3 * j] = s_den[3 * j + 1] = s_den[3 * j + 2] = 0u;
    }
    if (tid == 0) { s_maxabs = 0u; s_maxabs_z = 0u; }
    __syncthreads();
    const int *hidx = b.hyp_index + (size_t)f * H;
    float mabs = 0.f, mabs_z = 0.f;
    for (int r = tid; r < nv; r += blockDim.x) {
        const int h = hidx[r], m = h / J, j = h - m * J;
        atomicMin(&s_first[j], m);
        atomicMax(&s_last[j], m);
        const float *pp = b.hyp_prep + ((size_t)f * H + r) * 8;
        mabs = fmaxf(mabs, fmaxf(fabsf(pp[0]), fmaxf(fabsf(pp[1]), fabsf(pp[2]))));
        mabs_z = fmaxf(mabs_z, fabsf(pp[2]));
    }
    if (tid < 6 && nv > 0) {   // point AABB: pmin xyz, pmax xyz
        const float v = fabsf(b.cand_stats[(size_t)f * kStatsFloats + 3 + tid]);
        mabs = fmaxf(mabs, v);
        if (tid == 2 || tid == 5) mabs_z = v;
    }
    atomicMax(&s_maxabs, __float_as_uint(mabs));
    atomicMax(&s_maxabs_z, __float_as_uint(mabs_z));
    __syncthreads();
    for (int r = tid; r < nv; r += blockDim.x) {
        const int h = hidx[r], m = h / J, j = h - m * J;
        const bool first = (m == s_first[j]), last = (m == s_last[j]);
        if (first || last) {
            float Cv[3];
            sweep_axes(load_prep(b.hyp_prep, (size_t)f * H + r), Cv);
            for (int k = 0; k < 3; k++) {
                if (first) s_c0[3 * j + k] = Cv[k];
                if (last) s_c1[3 * j + k] = Cv[k];
            }
            if (first) s_r0[j] = r;
        }
    }
    __syncthreads();
    for (int i = tid; i < 3 * J; i += blockDim.x) {
        const int j = i / 3;
        const int span = s_last[j] - s_first[j];
        s_c1[i] = span > 0 ? __fdiv_rn(__fsub_rn(s_c1[i], s_c0[i]), (float)span) : 0.f;   // slope per depth step
    }
    __syncthreads();
    for (int r = tid; r < nv; r += blockDim.x) {
        const int h = hidx[r], m = h / J, j = h - m * J;
        float Cv[3];
        sweep_axes(load_prep(b.hyp_prep, (size_t)f * H + r), Cv);
        const float dm = (float)(m - s_first[j]);
        for (int k = 0; k < 3; k++) {
            const float line = __fmaf_rn(s_c1[3 * j + k], dm, s_c0[3 * j + k]);
            const float d = __fsub_rn(Cv[k], line);
            if (d > 0.f) atomicMax(&s_dev[3 * j + k], __float_as_uint(d));
            if (d < 0.f) atomicMax(&s_den[3 * j + k], __float_as_uint(-d));
        }
    }
    __syncthreads();
    const float eps = sweep_eps(__uint_as_float(s_maxabs)), eps_z = sweep_eps_z(__uint_as_float(s_maxabs_z));
    for (int j = tid; j < J; j += blockDim.x) {
        const int m0 = s_first[j], m1 = s_last[j];
        SweepCol c;
        if (m1 >= m0) {
            // every hypothesis of the column carries the same cosa, sina, tx, ty, hz: read the first one
            const float dev[3] = {__uint_as_float(s_dev[3 * j]), __uint_as_float(s_dev[3 * j + 1]),
                                  __uint_as_float(s_dev[3 * j + 2])};
            const float den[3] = {__uint_as_float(s_den[3 * j]), __uint_as_float(s_den[3 * j + 1]),
                                  __uint_as_float(s_den[3 * j + 2])};
            c = sweep_col_build(m0, m1, s_c0 + 3 * j, s_c1 + 3 * j, dev, den,
                                load_prep(b.hyp_prep, (size_t)f * H + s_r0[j]), eps, eps_z);
        } else {
            c = SweepCol{};
            c.m0 = 0; c.m1 = -1;
        }
        out[j] = c;
    }
}

#ifndef FNP_SWEEP_THREADS
#define FNP_SWEEP_THREADS 256
#endif
constexpr int kSweepThreads = FNP_SWEEP_THREADS;
constexpr int kSweepWarps = kSweepThreads / 32;
constexpr int kSweepChunk = kPage;   // points per (column, chunk) warp item = one page

// Entries (point | column << 16, packed steps) of a WARP's uncertain-step queue.  A piece (256 points of one column)
// pushes at most 256; a warp drains its queue before a piece that might not fit.
#ifndef FNP_SWEEP_QUEUE
#define FNP_SWEEP_QUEUE 384
#endif
constexpr int kSweepQueue = FNP_SWEEP_QUEUE;
static_assert(kSweepQueue >= kSweepChunk, "a piece must fit an empty queue");
__host__ __device__ inline size_t sweep_smem_bytes(int SP, int H, int J)
{
    return (size_t)J * sizeof(SweepCol) + (size_t)kSweepWarps * kSweepQueue * 8 + (size_t)SP * 12 + (size_t)H * 4 +
           (size_t)((H + 3) & ~3) * 2 + 16 + 128;      // + one scratch word per lane
}

#ifndef FNP_SWEEP_MIN_CTAS
#define FNP_SWEEP_MIN_CTAS 4
#endif

// A point that lies in no hypothesis of any column: the tail of a split's last page is filled with it, so that the
// sweep needs no "is this lane's point live" predicate (its possible range is empty in every column: one of
// U, V is >= 0.7e18, far beyond any centre, and 1e18 / slope stays finite).
#define FNP_SWEEP_FAR 1e18f

// *addr += v in shared memory, unconditionally (the caller points lanes that have nothing to add at their own scratch
// word: ptxas turns a predicated RED back into a branch around it, five instructions instead of two)
__device__ __forceinline__ void red_shared(const unsigned addr, const int v)
{
    asm volatile("red.shared.add.s32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}

// Exact predicates of `qn` queued entries of one warp (its own queue region `q`): expanded to single depth steps and
// spread evenly over the lanes -- every lane takes one step at a time, whichever point and column it belongs to.
__device__ __noinline__ void sweep_drain(const uint2 *q, const int qn, const SweepCol *s_col, const float *s_pts, int *s_diff,
                                         const short *s_slot, const float *prep_f, const int J, const int M)
{
    const int lane = threadIdx.x & 31;
    auto red = [](int *p, int v) { atomicAdd(p, v); };
    __syncwarp();      // the entries were written by other lanes of this warp: order their stores before the loads below
    for (int qb = 0; qb < qn; qb += 32) {
        uint2 ent = make_uint2(0u, 0u);
        if (qb + lane < qn) ent = q[qb + lane];
        const int cnt = sweep_packed_count(ent.y);
        int incl = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        const int total = __shfl_sync(0xffffffffu, incl, 31);
        for (int t0 = 0; t0 < total; t0 += 32) {
            const int t = t0 + lane;
            // owner = first lane whose inclusive prefix exceeds t
            int own = 0;
#pragma unroll
            for (int step = 16; step; step >>= 1) {
                const int v = __shfl_sync(0xffffffffu, incl, own + step - 1);
                if (v <= t) own += step;
            }
            own = min(own, 31);
            const unsigned e0 = __shfl_sync(0xffffffffu, ent.x, own);
            const unsigned e1 = __shfl_sync(0xffffffffu, ent.y, own);
            const int first = __shfl_sync(0xffffffffu, incl - cnt, own);
            if (t < total) {
                const int i = (int)(e0 & 0xffffu), j = (int)(e0 >> 16);
                const float4 rot = *reinterpret_cast<const float4 *>(&s_col[j].cosa);     // cosa, sina, tx, ty
                const int m0 = s_col[j].m0, D = s_col[j].m1 - m0;
                const float *pp = s_pts + (i >> 8) * (3 * kPage) + (i & (kPage - 1));
                sweep_exact_step_col(pp[0], pp[kPage], pp[2 * kPage], sweep_packed_step(e1, t - first), D, s_diff + j * M + m0,
                                     s_slot + m0 * J + j, J, prep_f, rot.x, rot.y, rot.z, rot.w, red);
            }
        }
    }
}

// Persistent CTAs pull (frustum, point split) items.  Per item:
//   stage   column parameters, the split's pages (x, y, z planes as they lie in the pool), cleared difference arrays,
//           slot table;
//   sweep   warps pull (column, 256-point chunk) pieces off a shared counter; per point one range solve
//           (sweep_solve) and the branch-free bookkeeping of sweep_emit: the definite range as two unconditional
//           shared-memory REDs (lanes with nothing to add aim at their own scratch word), the uncertain steps --
//           ~9 % of the pairs have any -- as one entry into the WARP's own queue region (ballot + popc, no atomic);
//           a warp drains its queue (sweep_drain) when the next piece might not fit and when the pieces run out;
//   scan    prefix sum over the depth steps of every column, one integer RED per valid hypothesis
//           into row f of `counts`.
__global__ void __launch_bounds__(kSweepThreads, FNP_SWEEP_MIN_CTAS) sweep_score_kernel(const fnp_seeker_batch b, const int J, const int M)
{
    extern __shared__ __align__(16) unsigned char s_dyn[];
    const int H = J * M, SP = b.split_points;
    SweepCol *s_col = reinterpret_cast<SweepCol *>(s_dyn);                      // [J]   (80 B each: 16 B aligned)
    uint2 *s_q = reinterpret_cast<uint2 *>(s_col + J);                          // [warps][kSweepQueue] uncertain-step queues
    float *s_pts = reinterpret_cast<float *>(s_q + kSweepWarps * kSweepQueue);  // [SP / 256][x | y | z][256]: the split's pages
    int *s_diff = reinterpret_cast<int *>(s_pts + 3 * SP);                      // [J][M] difference array, then counts
    short *s_slot = reinterpret_cast<short *>(s_diff + H);                      // [H] compacted slot of hypothesis h, -1
    int *s_ctl = reinterpret_cast<int *>(s_slot + ((H + 3) & ~3));              // [0] item [1] next piece [4..35] scratch

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned lt_mask = (1u << lane) - 1u;
    if (b.status[0] & 2) return;
    const int n_items = b.status[2];
    uint2 *q_w = s_q + warp * kSweepQueue;                                      // this warp's queue region
    const unsigned scratch_addr = smem_u32(s_ctl + 4 + lane);                   // this lane's scratch word (its own bank)

    for (;;) {
        __syncthreads();
        if (tid == 0) {
            s_ctl[0] = atomicAdd(&b.status[4], 1);
            s_ctl[1] = 0;
        }
        __syncthreads();
        const int item_id = s_ctl[0];
        if (item_id >= n_items) break;
        const int4 item = reinterpret_cast<const int4 *>(b.items)[item_id];   // frustum, -, split, -
        const int f = item.x, split = item.z;
        const int nv = b.hyp_nvalid[f], npts = b.cand_npts[f];
        const int p0 = split * SP;
        const int n = min(npts, p0 + SP) - p0;
        const float *prep_f = b.hyp_prep + (size_t)f * H * 8;

        // ---- stage
        {
            const float4 *src = reinterpret_cast<const float4 *>(b.sweep_cols + (size_t)f * J * FNP_SWEEP_COL_FLOATS);
            float4 *dst = reinterpret_cast<float4 *>(s_col);
            for (int i = tid; i < J * (FNP_SWEEP_COL_FLOATS / 4); i += kSweepThreads) dst[i] = __ldg(src + i);
            // the x, y, z planes of the split's pages, as they lie in the pool (coalesced, no transposition); slots past
            // the split's last point (the unwritten tail of the last page) become far points
            const int *tab = b.page_tab + (size_t)f * b.page_tab_stride + p0 / kPage;
            const int n_pg = (n + kPage - 1) / kPage;
            constexpr int kVec = 3 * kPage / 4;        // 16-byte vectors of a page's x, y, z planes
            for (int i = tid; i < n_pg * kVec; i += kSweepThreads) {
                const int q = i / kVec, v = i - q * kVec;
                const float4 *page = reinterpret_cast<const float4 *>(b.frustum_pts + (size_t)(tab[q] - 1) * (size_t)(b.page_planes * kPage));
                float4 val = __ldg(page + v);
                const int first = q * kPage + 4 * (v & (kPage / 4 - 1));      // point index of val.x
                if (first + 3 >= n) {
                    const float pad = v < kPage / 4 ? FNP_SWEEP_FAR : 0.f;    // x plane: far; y, z planes: 0
                    if (first >= n) val.x = pad;
                    if (first + 1 >= n) val.y = pad;
                    if (first + 2 >= n) val.z = pad;
                    val.w = pad;
                }
                reinterpret_cast<float4 *>(s_pts)[i] = val;
            }
            for (int h = tid; h < H; h += kSweepThreads) { s_diff[h] = 0; s_slot[h] = -1; }
        }
        __syncthreads();
        {
            const int *hidx = b.hyp_index + (size_t)f * H;
            for (int r = tid; r < nv; r += kSweepThreads) s_slot[hidx[r]] = (short)r;
        }
        __syncthreads();

        // ---- sweep
        const int n_chunks = (n + kSweepChunk - 1) / kSweepChunk;
        const int n_pieces = J * n_chunks;
        int qn = 0;                                  // entries in this warp's queue (warp-uniform)
        for (;;) {
            int piece = 0;
            if (lane == 0) piece = atomicAdd(&s_ctl[1], 1);
            piece = __shfl_sync(0xffffffffu, piece, 0);
            const bool done = piece >= n_pieces;
            if (done || qn + kSweepChunk > kSweepQueue) {      // out of pieces, or the next piece might not fit
                sweep_drain(q_w, qn, s_col, s_pts, s_diff, s_slot, prep_f, J, M);
                __syncwarp();      // ... and the loads above before the next piece's stores into the same region
                qn = 0;
            }
            if (done) break;
            const int j = piece % J, ch = piece / J;
            const SweepCol c = s_col[j];            // warp-uniform: lives in registers for the whole piece
            if (c.m1 < c.m0) continue;
            const int D = c.m1 - c.m0;
            int *diff = s_diff + j * M + c.m0;       // indexed by dm = m - m0
            const unsigned diff_addr = smem_u32(diff);
            int base_cnt = 0;
            const int n_pass = (min(n - ch * kSweepChunk, kSweepChunk) + 63) >> 6;   // 64 points per pass
            const float *px = s_pts + ch * (3 * kPage) + lane;
            unsigned key = (unsigned)(ch * kSweepChunk + lane) | ((unsigned)j << 16);
            // two points per lane and pass: the two range solves are independent instruction chains
            for (int pass = 0; pass < n_pass; pass++, px += 64, key += 64) {
                const float xa = px[0], ya = px[kPage], za = px[2 * kPage];
                const float xb = px[32], yb = px[kPage + 32], zb = px[2 * kPage + 32];
                const SweepRanges ra = sweep_solve(c, xa, ya, za);
                const SweepRanges rb = sweep_solve(c, xb, yb, zb);
                const SweepEmit ea = sweep_emit(ra, D), eb = sweep_emit(rb, D);
                red_shared(ea.add_lo ? diff_addr + 4u * (unsigned)ra.a : scratch_addr, 1);
                red_shared(ea.add_hi ? diff_addr + 4u * (unsigned)ra.e + 4u : scratch_addr, -1);
                red_shared(eb.add_lo ? diff_addr + 4u * (unsigned)rb.a : scratch_addr, 1);
                red_shared(eb.add_hi ? diff_addr + 4u * (unsigned)rb.e + 4u : scratch_addr, -1);
                base_cnt += (int)ea.from_zero + (int)eb.from_zero;
                const unsigned mka = __ballot_sync(0xffffffffu, ea.uncertain), mkb = __ballot_sync(0xffffffffu, eb.uncertain);
                if (ea.uncertain) q_w[qn + __popc(mka & lt_mask)] = make_uint2(key, ea.packed);
                qn += __popc(mka);
                if (eb.uncertain) q_w[qn + __popc(mkb & lt_mask)] = make_uint2(key + 32u, eb.packed);
                qn += __popc(mkb);
            }
            base_cnt = __reduce_add_sync(0xffffffffu, base_cnt);
            if (lane == 0 && base_cnt) atomicAdd(diff, base_cnt);   // ranges that start at the column's first step
        }
        __syncthreads();

        // ---- prefix sum over the depth steps of every column (warp per column, in place)
        for (int j = warp; j < J; j += kSweepWarps) {
            int carry = 0;
            for (int mb = 0; mb < M; mb += 32) {
                const int m = mb + lane;
                int v = m < M ? s_diff[j * M + m] : 0;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int t = __shfl_up_sync(0xffffffffu, v, o);
                    if (lane >= o) v += t;
                }
                v += carry;
                if (m < M) s_diff[j * M + m] = v;
                carry = __shfl_sync(0xffffffffu, v, 31);
            }
        }
        __syncthreads();
        int *out = b.counts + (size_t)f * H;
        for (int h = tid; h < H; h += kSweepThreads) {
            const int r = s_slot[h];
            if (r >= 0) {
                const int m = h / J, j = h - m * J;
                const int cnt = s_diff[j * M + m];
                if (cnt) atomicAdd(out + r, cnt);      // RED.ADD: the splits of a frustum add up in any order
            }
        }
    }
}

// ======================================================================================
// Stage 2b, KITTI variant: ONE batched first-match points_in_boxes_gpu over the valid hypotheses of a frustum
// (frustum_proposals_v1_kitti.py:644-648; roiaware_pool3d_kernel.cu:313-359): a point counts for the FIRST hypothesis,
// in compacted order, that contains it.  CTA per (frustum, 4096-point split); every thread walks the hypotheses of
// its point until the first hit (the hypotheses are read by all lanes at once: L1 broadcast).
// ======================================================================================
constexpr int kFmThreads = 256, kFmSplit = 4096;
__global__ void __launch_bounds__(kFmThreads) firstmatch_kernel(const fnp_seeker_batch b, const int H)
{
    const int f = blockIdx.x;
    const int nv = b.hyp_nvalid[f], npts = b.cand_npts[f];
    if (nv <= 0 || npts <= 0 || (b.status[0] & 2)) return;
    const int p0 = blockIdx.y * kFmSplit;
    if (p0 >= npts) return;
    const int p1 = min(npts, p0 + kFmSplit);
    int *cnt = b.counts + (size_t)f * H;
    for (int i = p0 + (int)threadIdx.x; i < p1; i += kFmThreads) {
        const float *pg = page_of(b, f, i >> 8) + (i & (kPage - 1));
        const float x = pg[0], y = pg[kPage], z = pg[2 * kPage];
        for (int r = 0; r < nv; r++) {
            if (in_box(x, y, z, load_prep(b.hyp_prep, (size_t)f * H + r))) {
                atomicAdd(cnt + r, 1);
                break;
            }
        }
    }
}

// ======================================================================================
// Stage 3: score + greedy argmax
// ======================================================================================
// Optional stage 2c: n_far of every compacted hypothesis = frustum points whose norm exceeds the norm of
// the hypothesis' nearest corner (calc_occl_scores, frustum_proposals_v1.py:408-477; the corners are rebuilt
// from the box the way boxes_to_corners_3d does, box_utils.py:28-52).  One thread per hypothesis, the
// norms of a tile of points in shared memory, read as broadcast LDS.128.
constexpr int kOcclThreads = 256;
constexpr int kOcclTile = 2048;

__global__ void __launch_bounds__(kOcclThreads) occl_kernel(const fnp_seeker_batch b, const int J, const int H)
{
    __shared__ __align__(16) float s_mag[kOcclTile];
    const int f = blockIdx.x, tid = threadIdx.x;
    const int nv = b.hyp_nvalid[f];
    const int r = blockIdx.y * kOcclThreads + tid;
    if ((int)(blockIdx.y * kOcclThreads) >= nv || b.status[0] != 0) return;
    const float INF = __int_as_float(0x7f800000);
    float m1 = INF;
    if (r < nv) {
        const float *pp = b.hyp_prep + ((size_t)f * H + r) * 8;
        const int j = b.hyp_index[(size_t)f * H + r] % J;
        const float *bb = b.base_boxes + ((size_t)(b.cand_label[f] - 1) * J + j) * 7;
        const float ca = cosf(bb[6]), sa = sinf(bb[6]);
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const float sx = (k == 0 || k == 1 || k == 4 || k == 5) ? 0.5f : -0.5f;   // box_utils.py:42-45
            const float sy = (k == 0 || k == 3 || k == 4 || k == 7) ? 0.5f : -0.5f;
            const float sz = (k >= 4) ? 0.5f : -0.5f;
            const float x = __fmul_rn(bb[3], sx), y = __fmul_rn(bb[4], sy), z = __fmul_rn(bb[5], sz);
            const float cx = __fadd_rn(__fmaf_rn(y, -sa, __fmul_rn(x, ca)), pp[0]);
            const float cy = __fadd_rn(__fmaf_rn(y, ca, __fmul_rn(x, sa)), pp[1]);
            const float cz = __fadd_rn(z, pp[2]);
            m1 = fminf(m1, norm3(cx, cy, cz));
        }
    }
    const int n = b.cand_npts[f];
    int cnt = 0;
    for (int t0 = 0; t0 < n; t0 += kOcclTile) {
        const int tn = min(kOcclTile, n - t0);
        for (int i = tid; i < kOcclTile; i += kOcclThreads) {
            float m = -INF;   // padding never counts
            if (i < tn) {
                const int p = t0 + i;
                const float *rec = page_of(b, f, p >> 8) + (p & (kPage - 1));
                m = norm3(rec[0], rec[kPage], rec[2 * kPage]);
            }
            s_mag[i] = m;
        }
        __syncthreads();
        const float4 *sm4 = reinterpret_cast<const float4 *>(s_mag);
        const int n4 = (tn + 3) >> 2;
#pragma unroll 4
        for (int i = 0; i < n4; i++) {
            const float4 m = sm4[i];
            cnt += (m.x > m1) + (m.y > m1) + (m.z > m1) + (m.w > m1);
        }
        __syncthreads();
    }
    if (r < nv) b.hyp_nfar[(size_t)f * H + r] = cnt;
}

// ======================================================================================
// Stage 3: second-stage score + greedy argmax
// ======================================================================================
__device__ __forceinline__ float block_max128(float v, float *s4, const int lane, const int warp)
{
    v = warp_max(v);
    if (lane == 0) s4[warp] = v;
    __syncthreads();
    v = fmaxf(fmaxf(s4[0], s4[1]), fmaxf(s4[2], s4[3]));
    __syncthreads();
    return v;
}

// Warp-wide arg-max of (score, index), lowest index on ties; every lane gets the result.
// besti == 0x7fffffff means "no entry".
__device__ __forceinline__ void warp_argmax(float &best, int &besti)
{
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        const float ob = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, besti, o);
        if (oi != 0x7fffffff && (besti == 0x7fffffff || ob > best || (ob == best && oi < besti))) { best = ob; besti = oi; }
    }
}

// Block-wide arg-max of (score, index) over 128 threads, lowest index on ties; every thread gets the result.
__device__ __forceinline__ void block_argmax128(float &best, int &besti, float *s_f, int *s_i, const int lane,
                                                const int warp)
{
    warp_argmax(best, besti);
    if (lane == 0) { s_f[warp] = best; s_i[warp] = besti; }
    __syncthreads();
    best = s_f[0]; besti = s_i[0];
#pragma unroll
    for (int w = 1; w < 4; w++) {
        const float ob = s_f[w];
        const int oi = s_i[w];
        if (oi != 0x7fffffff && (besti == 0x7fffffff || ob > best || (ob == best && oi < besti))) { best = ob; besti = oi; }
    }
    __syncthreads();
}

constexpr int kSelectMaxTopkH = 32768;   // hypotheses per frustum the suppression bitmask of topk > 1 covers

// The weights and switches of the second-stage score.  Every stage-3 kernel forms the score with hyp_score, so
// that a setting scored by select_multi_kernel gets the bits select_kernel gives it.
struct ScoreTerms {
    float dns_w, iou_w, dst_w, ego_w, occl_w;
    bool kitti, mult, occl_mult, use_dist, use_occl_w, use_ego;
};

// Second-stage score of one hypothesis (frustum_proposals_v1.py:996-1026; FrustumProposerOGKITTI :650-654).
// count / den: its point count over the frustum's normaliser; dist, dmin, dden: the distance term (read only with
// use_dist); fail / fden: its occlusion score and the normaliser max + 1e-6 (use_occl_w, occl_mult); ego / emx: the
// norm of its centre and the largest such norm (use_ego).
__device__ __forceinline__ float hyp_score(const ScoreTerms &t, const int count, const float den, const float iou,
                                           const float dist, const float dmin, const float dden, const float fail,
                                           const float fden, const float ego, const float emx)
{
    const float dens = __fdiv_rn((float)count, den);
    const float dr = t.use_dist ? __fsub_rn(1.0f, __fdiv_rn(__fsub_rn(dist, dmin), dden)) : 1.0f;
    float sc;
    if (t.kitti)
        sc = __fadd_rn(__fadd_rn(__fadd_rn(t.dns_w, dens), __fmul_rn(t.iou_w, iou)), __fmul_rn(dr, t.dst_w));
    else if (t.mult)
        sc = __fmul_rn(__fmul_rn(__fmul_rn(__fmul_rn(__fmul_rn(dens, t.dns_w), iou), t.iou_w), dr), t.dst_w);
    else {
        sc = __fadd_rn(__fmul_rn(dens, t.dns_w), __fmul_rn(iou, t.iou_w));
        if (t.use_dist) sc = __fadd_rn(sc, __fmul_rn(dr, t.dst_w));
    }
    if (t.use_occl_w) sc = __fadd_rn(sc, __fmul_rn(t.occl_w, __fsub_rn(1.0f, __fdiv_rn(fail, fden))));
    if (t.use_ego) sc = __fadd_rn(sc, __fmul_rn(t.ego_w, __fdiv_rn(ego, emx)));
    if (t.occl_mult) sc = __fmul_rn(__fmul_rn(dens, iou), fail);
    return sc;
}

// EXTRAS = false is the shipped configuration (density + IoU, top-1): the optional terms, the score table and
// the suppression bitmask of topk > 1 are compiled out.
template <bool EXTRAS>
__global__ void __launch_bounds__(128) select_kernel(const fnp_seeker_batch b, const fnp_seeker_cfg cfg)
{
    __shared__ float s_f[4];
    __shared__ int s_i[4];
    __shared__ unsigned s_dead[EXTRAS ? kSelectMaxTopkH / 32 : 1];
    const int f = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int J = cfg.num_yaw_size, H = J * cfg.num_mags;
    const int T = EXTRAS ? max(cfg.topk, 1) : 1;
    const int nv = b.hyp_nvalid[f];
    if (nv <= 0 || (b.status[0] & 2)) {
        for (int k = tid; k < T; k += blockDim.x) {
            b.out_best[(size_t)f * T + k] = -1; b.out_score[(size_t)f * T + k] = 0.f; b.out_count[(size_t)f * T + k] = 0;
        }
        return;
    }
    const int *cbase = b.counts + (size_t)f * H;
    const float *pbase = b.hyp_prep + (size_t)f * H * 8;
    const bool mult = EXTRAS && (cfg.flags & FNP_SEEKER_MULT) != 0, occl_mult = EXTRAS && (cfg.flags & FNP_SEEKER_OCCL_MULT) != 0;
    const bool use_dist = EXTRAS && ((cfg.dst_w != 0.f) || mult || cfg.variant == FNP_VARIANT_KITTI);
    const bool use_fail = EXTRAS && ((cfg.occl_w > 0.f) || occl_mult);
    const bool use_ego = EXTRAS && cfg.ego_w > 0.f;
    const bool use_occl_w = EXTRAS && cfg.occl_w > 0.f;
    const long long npts = b.cand_npts[f];
    const int *nfar = use_fail ? b.hyp_nfar + (size_t)f * H : nullptr;
    // the reference's occlusion score: n_far * n_out (a (P,1) & (P,) broadcast, :453), stored as float
#define FNP_FAIL(r) __ll2float_rn((long long)nfar[r] * (npts - (long long)cbase[r]))
    // FrustumProposerOGKITTI (frustum_proposals_v1_kitti.py:650-654): first-match counts over their SUM, and
    // score = dns_w + density + iou_w iou + dst_w dists_ranked
    const bool kitti = EXTRAS && cfg.variant == FNP_VARIANT_KITTI;
    int mxi = 0, sumi = 0;
    float fmx = 0.f, emx = 0.f;
    for (int r = tid; r < nv; r += blockDim.x) {
        mxi = max(mxi, cbase[r]);
        sumi += cbase[r];
        if (use_fail) fmx = fmaxf(fmx, FNP_FAIL(r));
        if (use_ego) emx = fmaxf(emx, norm3(pbase[r * 8], pbase[r * 8 + 1], pbase[r * 8 + 2]));
    }
    float den = __fadd_rn(block_max128((float)mxi, s_f, lane, warp), 1e-8f);
    if (kitti) {      // integer-valued floats: the sum is exact in any order (below 2^24 points)
        sumi = __reduce_add_sync(0xffffffffu, sumi);
        if (lane == 0) s_i[warp] = sumi;
        __syncthreads();
        den = __fadd_rn((float)(s_i[0] + s_i[1] + s_i[2] + s_i[3]), 1e-8f);
        __syncthreads();
    }
    float fden = 1.f, dmin = 0.f, dden = 1.f;
    if (use_fail) fden = __fadd_rn(block_max128(fmx, s_f, lane, warp), 1e-6f);
    if (use_ego) emx = block_max128(emx, s_f, lane, warp);
    if (use_dist) {
        const float *st = b.cand_stats + (size_t)f * kStatsFloats;
        dmin = st[13];
        dden = __fadd_rn(__fsub_rn(st[14], dmin), 1e-8f);
    }
    // argmax of score, lowest index wins ties (stable descending sort + top-1)
    const ScoreTerms terms = {cfg.dns_w, cfg.iou_w, cfg.dst_w, cfg.ego_w, cfg.occl_w, kitti, mult, occl_mult, use_dist,
                              use_occl_w, use_ego};
    float best = -__int_as_float(0x7f800000);
    int besti = 0x7fffffff;
    for (int r = tid; r < nv; r += blockDim.x) {
        const float sc = hyp_score(terms, cbase[r], den, b.hyp_iou[(size_t)f * H + r],
                                   use_dist ? b.hyp_dist[(size_t)f * H + r] : 0.f, dmin, dden,
                                   (use_occl_w || occl_mult) ? FNP_FAIL(r) : 0.f, fden,
                                   use_ego ? norm3(pbase[r * 8], pbase[r * 8 + 1], pbase[r * 8 + 2]) : 0.f, emx);
        if (T > 1) b.hyp_score[(size_t)f * H + r] = sc;
        if (sc > best || besti == 0x7fffffff) { best = sc; besti = r; }
    }
#undef FNP_FAIL
    if (T > 1) {
        for (int i = tid; i < (nv + 31) >> 5; i += blockDim.x) s_dead[i] = 0u;
    }
    block_argmax128(best, besti, s_f, s_i, lane, warp);     // also orders the hyp_score / s_dead writes
    const float *bb_tab = b.base_boxes + (size_t)(b.cand_label[f] - 1) * J * 7;
    for (int k = 0;;) {
        const float *pp = pbase + (size_t)besti * 8;
        const float *bb = bb_tab + (size_t)(b.hyp_index[(size_t)f * H + besti] % J) * 7;
        if (tid == 0) {
            float *o = b.out_boxes + ((size_t)f * T + k) * 7;
            o[0] = pp[0]; o[1] = pp[1]; o[2] = pp[2];
            o[3] = bb[3]; o[4] = bb[4]; o[5] = bb[5]; o[6] = bb[6];
            b.out_best[(size_t)f * T + k] = besti;
            b.out_score[(size_t)f * T + k] = best;
            b.out_count[(size_t)f * T + k] = cbase[besti];
        }
        if (++k >= T) break;
        // nms_normal_gpu (:1030, iou3d_nms.cpp:162-209): the kept box suppresses every later one with an
        // axis-aligned BEV IoU above the threshold; the next kept box is the best survivor
        const float abox[5] = {pp[0], pp[1], 0.f, bb[3], bb[4]};
        if (tid == 0) atomicOr(&s_dead[besti >> 5], 1u << (besti & 31));
        for (int r = tid; r < nv; r += blockDim.x) {
            if ((s_dead[r >> 5] >> (r & 31)) & 1u) continue;
            const float *bq = bb_tab + (size_t)(b.hyp_index[(size_t)f * H + r] % J) * 7;
            const float qbox[5] = {pbase[r * 8], pbase[r * 8 + 1], 0.f, bq[3], bq[4]};
            if (r != besti && iou_normal(abox, qbox) > cfg.nms_normal) atomicOr(&s_dead[r >> 5], 1u << (r & 31));
        }
        __syncthreads();
        best = -__int_as_float(0x7f800000);
        besti = 0x7fffffff;
        for (int r = tid; r < nv; r += blockDim.x) {
            if ((s_dead[r >> 5] >> (r & 31)) & 1u) continue;
            const float sc = b.hyp_score[(size_t)f * H + r];
            if (sc > best || besti == 0x7fffffff) { best = sc; besti = r; }
        }
        block_argmax128(best, besti, s_f, s_i, lane, warp);
        if (besti == 0x7fffffff) {       // fewer survivors than topk: the remaining slots stay empty
            for (int kk = k + tid; kk < T; kk += blockDim.x) {
                b.out_best[(size_t)f * T + kk] = -1; b.out_score[(size_t)f * T + kk] = 0.f; b.out_count[(size_t)f * T + kk] = 0;
            }
            break;
        }
    }
}

// Stage 3 for many select-level settings over one execution of stages 1-2c (fnp_seeker_select_multi).  One CTA
// per frustum stages the frustum's per-hypothesis inputs in shared memory once -- count and IoU, and the planes some
// setting reads: distance, occlusion score, centre norm -- then warp w scores settings w, w + 8, ...: the setting's
// valid set is the compacted hypotheses with iou > its min_cam_iou, the count / occlusion / ego normalisers are
// maxima over that set, and the arg-max of hyp_score over it breaks ties on the lowest index (compaction keeps the
// original order, so that is also the lowest original index: select_kernel's choice for a cfg with those values).
// KITTI = true is FrustumProposerOGKITTI's score (fnp_seeker_select_multi admits it only when every setting keeps the
// cfg's min_cam_iou, so the valid set, and with it every first-match count, is the one stages 1-2c produced): the
// count normaliser is the SUM of the compacted counts, exact in any order below 2^24 points as in select_kernel, the
// distance plane is always staged and the score is hyp_score with kitti = true.
constexpr int kMultiThreads = 256;
constexpr int kMultiPlaneDist = 1, kMultiPlaneFail = 2, kMultiPlaneEgo = 4;

struct SelectSettings {
    fnp_select_setting s[FNP_SELECT_MAX_SETTINGS];
};

template <bool KITTI>
__global__ void __launch_bounds__(kMultiThreads) select_multi_kernel(const fnp_seeker_batch b, const int J, const int H,
                                                                    const SelectSettings set, const int n_set,
                                                                    const int planes, float *out_boxes, float *out_score,
                                                                    int32_t *out_best, int32_t *out_count)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int f = blockIdx.x, F = b.n_cands;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nv = (b.status[0] & 2) ? 0 : b.hyp_nvalid[f];
    int *s_cnt = reinterpret_cast<int *>(smem);
    float *s_iou = reinterpret_cast<float *>(s_cnt + H);
    float *p_next = s_iou + H;
    float *s_dist = (KITTI || (planes & kMultiPlaneDist)) ? p_next : nullptr;
    p_next += s_dist ? H : 0;
    float *s_fail = (planes & kMultiPlaneFail) ? p_next : nullptr;
    p_next += s_fail ? H : 0;
    float *s_ego = (planes & kMultiPlaneEgo) ? p_next : nullptr;
    const size_t fH = (size_t)f * H;
    const float *pbase = b.hyp_prep + fH * 8;
    const long long npts = b.cand_npts[f];
    for (int r = threadIdx.x; r < nv; r += kMultiThreads) {
        const int c = b.counts[fH + r];
        s_cnt[r] = c;
        s_iou[r] = b.hyp_iou[fH + r];
        if (s_dist) s_dist[r] = b.hyp_dist[fH + r];
        // the reference's occlusion score n_far * n_out, as select_kernel's FNP_FAIL forms it
        if (s_fail) s_fail[r] = __ll2float_rn((long long)b.hyp_nfar[fH + r] * (npts - (long long)c));
        if (s_ego) s_ego[r] = norm3(pbase[r * 8], pbase[r * 8 + 1], pbase[r * 8 + 2]);
    }
    float dmin = 0.f, dden = 1.f;
    if (s_dist) {
        const float *st = b.cand_stats + (size_t)f * kStatsFloats;
        dmin = st[13];
        dden = __fadd_rn(__fsub_rn(st[14], dmin), 1e-8f);
    }
    __syncthreads();
    const float *bb_tab = b.base_boxes + (size_t)(b.cand_label[f] - 1) * J * 7;
    for (int si = warp; si < n_set; si += kMultiThreads / 32) {
        const fnp_select_setting p = set.s[si];
        const bool mult = (p.flags & FNP_SEEKER_MULT) != 0, occl_mult = (p.flags & FNP_SEEKER_OCCL_MULT) != 0;
        const ScoreTerms t = KITTI ? ScoreTerms{p.dns_w, p.iou_w, p.dst_w, 0.f, 0.f, true, false, false, true, false, false}
                                   : ScoreTerms{p.dns_w, p.iou_w, p.dst_w, p.ego_w, p.occl_w, false, mult, occl_mult,
                                                (p.dst_w != 0.f) || mult, p.occl_w > 0.f, p.ego_w > 0.f};
        const bool use_fail = t.use_occl_w || t.occl_mult;
        const float thr = p.min_cam_iou;
        int mxi = 0;
        float fmx = 0.f, emx = 0.f;
        for (int r = lane; r < nv; r += 32) {
            if (!(s_iou[r] > thr)) continue;
            mxi = KITTI ? mxi + s_cnt[r] : max(mxi, s_cnt[r]);
            if (use_fail) fmx = fmaxf(fmx, s_fail[r]);
            if (t.use_ego) emx = fmaxf(emx, s_ego[r]);
        }
        const float den = KITTI ? __fadd_rn((float)__reduce_add_sync(0xffffffffu, mxi), 1e-8f)
                                : __fadd_rn(warp_max((float)mxi), 1e-8f);
        const float fden = use_fail ? __fadd_rn(warp_max(fmx), 1e-6f) : 1.f;
        if (t.use_ego) emx = warp_max(emx);
        float best = -__int_as_float(0x7f800000);
        int besti = 0x7fffffff;
        for (int r = lane; r < nv; r += 32) {
            if (!(s_iou[r] > thr)) continue;
            const float sc = hyp_score(t, s_cnt[r], den, s_iou[r], t.use_dist ? s_dist[r] : 0.f, dmin, dden,
                                       use_fail ? s_fail[r] : 0.f, fden, t.use_ego ? s_ego[r] : 0.f, emx);
            if (sc > best || besti == 0x7fffffff) { best = sc; besti = r; }
        }
        warp_argmax(best, besti);
        // every lane writes lane 0's choice: the lanes agree after warp_argmax unless scores are unordered (NaN)
        best = __shfl_sync(0xffffffffu, best, 0);
        besti = __shfl_sync(0xffffffffu, besti, 0);
        const size_t o = (size_t)si * F + f;
        if (lane < 7) {
            float v = 0.f;      // a frustum without a hypothesis valid for the setting: zeros, best -1
            if (besti != 0x7fffffff)
                v = lane < 3 ? pbase[(size_t)besti * 8 + lane] : bb_tab[(size_t)(b.hyp_index[fH + besti] % J) * 7 + lane];
            out_boxes[o * 7 + lane] = v;
        }
        if (lane == 0) {
            const bool none = besti == 0x7fffffff;
            out_best[o] = none ? -1 : besti;
            out_score[o] = none ? 0.f : best;
            out_count[o] = none ? 0 : s_cnt[besti];
        }
    }
}

}  // namespace fnp

// ======================================================================================
// C ABI
// ======================================================================================
using namespace fnp;

static int check_batch(const fnp_seeker_cfg *cfg, const fnp_seeker_batch *b)
{
    if (!cfg || !b) return FNP_EINVAL;
    if (b->n_frames < 0 || b->n_cands < 0 || b->n_tiles < 0) return FNP_EINVAL;
    if (cfg->num_mags < 1 || cfg->num_yaw_size < 1) return FNP_EINVAL;
    if (b->max_items < 0 || b->split_points < FNP_PAGE_POINTS || (b->split_points % FNP_PAGE_POINTS) != 0) return FNP_EINVAL;
    return FNP_OK;
}

// Tuning / test switches (fnp_set_option): not part of the stable ABI.
static int g_opt_cull_sectors = 1;      // stage 1 consults the per-frame sector table (0: every camera for every point)

extern "C" int fnp_set_option(const char *name, int value)
{
    if (!name) return FNP_EINVAL;
    const std::string n(name);
    if (n == "cull_sectors") { g_opt_cull_sectors = value; return FNP_OK; }
    return FNP_EINVAL;
}

static size_t cull_smem(const fnp_seeker_batch *b)
{
    return sizeof(CullSmem) + (size_t)b->max_cands_per_frame * (16 + 4 + 4) + (size_t)kCullList * (16 + 4 + 4) + 16;
}

template <int W, bool KITTI>
static int launch_cull(const fnp_seeker_cfg *cfg, const fnp_seeker_batch *b, cudaStream_t st)
{
    const int n_cu = cell_cols(cfg->img_w), n_cv = cell_rows(cfg->img_h);
    const size_t sa = cull_smem(b), sc = (size_t)n_cu * n_cv * W * 4;
    if (sa > 200 * 1024 || sc > 200 * 1024) return FNP_EINVAL;
    cudaFuncSetAttribute(cull_kernel<W, KITTI>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sa);
    cudaFuncSetAttribute(cell_table_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sc);
    cudaMemsetAsync(b->cell_masks + (size_t)b->n_frames * 6 * n_cu * n_cv * W, 0, (size_t)b->n_frames * kSectors * 4, st);
    cell_table_kernel<<<b->n_frames * 6, 128, sc, st>>>(*b, n_cu, n_cv, cfg->img_w, cfg->img_h, KITTI ? 1 : 0);
    // the azimuth-sector table is built from lidar2image: not in the KITTI variant (one camera anyway)
    cull_kernel<W, KITTI><<<b->n_tiles, kCullThreads, sa, st>>>(*b, cfg->img_w, cfg->img_h, n_cu, n_cv,
                                                               KITTI ? 0 : g_opt_cull_sectors);
    cull_finish_kernel<<<1, 32, 0, st>>>(*b);
    return FNP_OK;
}

extern "C" size_t fnp_seeker_cell_mask_bytes(const fnp_seeker_cfg *cfg, int n_frames, int max_cands_per_frame)
{
    const int W = fnp_seeker_mask_words(max_cands_per_frame);
    if (!cfg || n_frames < 0 || W < 0) return 0;
    // per (frame, camera rank, cell) W words, then the 64-entry sector table of every frame
    return (size_t)n_frames * 6 * cell_cols(cfg->img_w) * cell_rows(cfg->img_h) * W * 4 + (size_t)n_frames * kSectors * 4;
}

extern "C" int fnp_seeker_cull_tile(void) { return FNP_CULL_TILE; }

extern "C" int fnp_seeker_mask_words(int max_cands_per_frame)
{
    const int w = divup(max_cands_per_frame > 0 ? max_cands_per_frame : 1, 32);
    return w <= 1 ? 1 : w <= 2 ? 2 : w <= 4 ? 4 : w <= 8 ? 8 : w <= 16 ? 16 : w <= 32 ? 32 : -1;
}

extern "C" int fnp_seeker_cull(const fnp_seeker_cfg *cfg, const fnp_seeker_batch *b, void *stream)
{
    int rc = check_batch(cfg, b);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if (b->n_cands == 0 || b->n_tiles == 0) {
        cudaMemsetAsync(b->status, 0, 8 * sizeof(int32_t), st);
        if (b->n_cands) cudaMemsetAsync(b->cand_npts, 0, sizeof(int32_t) * (size_t)b->n_cands, st);
        FNP_LAUNCH_CHECK();
        return FNP_OK;
    }
    if (!b->points || !b->page_tab || !b->frustum_pts || !b->cell_masks || !b->cam_cand_start || b->point_stride < 3 ||
        b->xyz_offset < 0 || b->xyz_offset + 3 > b->point_stride || (b->page_planes != 4 && b->page_planes != 5) ||
        b->page_tab_stride < 1 || b->pts_capacity < FNP_PAGE_POINTS || (b->pts_capacity % FNP_PAGE_POINTS) != 0)
        return FNP_EINVAL;
    cudaMemsetAsync(b->status, 0, 8 * sizeof(int32_t), st);      // [5] = page cursor
    cudaMemsetAsync(b->cand_npts, 0, sizeof(int32_t) * (size_t)b->n_cands, st);
    cudaMemsetAsync(b->page_tab, 0, sizeof(int32_t) * (size_t)b->n_cands * (size_t)b->page_tab_stride, st);
    const int W = fnp_seeker_mask_words(b->max_cands_per_frame);
    if (W < 0 || W != b->mask_words) return FNP_EINVAL;   // more than 1024 candidates in one frame
    if (cfg->variant == FNP_VARIANT_KITTI) {      // up to 128 candidates per frame in this variant
        switch (W) {
            case 1: rc = launch_cull<1, true>(cfg, b, st); break;
            case 2: rc = launch_cull<2, true>(cfg, b, st); break;
            case 4: rc = launch_cull<4, true>(cfg, b, st); break;
            default: rc = FNP_EINVAL; break;
        }
    } else
    switch (W) {      // the words of a cell's candidate mask are a compile-time constant of the membership loop
        case 1: rc = launch_cull<1, false>(cfg, b, st); break;
        case 2: rc = launch_cull<2, false>(cfg, b, st); break;
        case 4: rc = launch_cull<4, false>(cfg, b, st); break;
        case 8: rc = launch_cull<8, false>(cfg, b, st); break;
        case 16: rc = launch_cull<16, false>(cfg, b, st); break;
        default: rc = launch_cull<32, false>(cfg, b, st); break;
    }
    if (rc) return rc;
    FNP_LAUNCH_CHECK();
    return FNP_OK;
}

extern "C" int fnp_seeker_frustum_stats(const fnp_seeker_cfg *cfg, const fnp_seeker_batch *b, void *stream)
{
    int rc = check_batch(cfg, b);
    if (rc) return rc;
    if (b->n_cands == 0) return FNP_OK;
    stats_kernel<<<b->n_cands, 256, 0, (cudaStream_t)stream>>>(*b, *cfg);
    FNP_LAUNCH_CHECK();
    return FNP_OK;
}

extern "C" int fnp_seeker_hypotheses(const fnp_seeker_cfg *cfg, const fnp_seeker_batch *b, void *stream)
{
    int rc = check_batch(cfg, b);
    if (rc) return rc;
    if (b->n_cands == 0) return FNP_OK;
    if (cfg->variant == FNP_VARIANT_KITTI) {
        if (!b->hyp_dist || (cfg->flags & FNP_SEEKER_MULTICAM_IOU)) return FNP_EINVAL;   // this head always ranks distances
        hypotheses_kernel<true, true><<<b->n_cands, 128, 0, (cudaStream_t)stream>>>(*b, *cfg);
    } else if ((cfg->flags & FNP_SEEKER_MULTICAM_IOU) || b->hyp_dist)
        hypotheses_kernel<true><<<b->n_cands, 128, 0, (cudaStream_t)stream>>>(*b, *cfg);
    else
        hypotheses_kernel<false><<<b->n_cands, 128, 0, (cudaStream_t)stream>>>(*b, *cfg);
    FNP_LAUNCH_CHECK();
    return FNP_OK;
}

// Scoring mode of a batch (see FNP_SCORE_* in fnp.h); < 0: invalid request.
static int resolve_score_mode(const fnp_seeker_cfg *cfg, const fnp_seeker_batch *b)
{
    const int J = cfg->num_yaw_size, M = cfg->num_mags;
    const long long H = (long long)J * M;
    const bool fits = b->sweep_cols && H <= 32767 && M <= 255 && J <= 65535 && b->split_points <= 65536 && sweep_smem_bytes(b->split_points, (int)H, J) <= 200 * 1024 &&
                      (size_t)15 * J * 4 <= 48 * 1024;
    switch (b->score_mode) {
        case FNP_SCORE_DIRECT: return FNP_SCORE_DIRECT;
        case FNP_SCORE_SWEEP: return fits ? FNP_SCORE_SWEEP : -1;
        case FNP_SCORE_AUTO: return (fits && M >= FNP_SWEEP_MIN_MAGS) ? FNP_SCORE_SWEEP : FNP_SCORE_DIRECT;
        default: return -1;
    }
}

extern "C" int fnp_seeker_score(const fnp_seeker_cfg *cfg, const fnp_seeker_batch *b, void *stream)
{
    int rc = check_batch(cfg, b);
    if (rc) return rc;
    if (b->n_cands == 0) return FNP_OK;
    const int J = cfg->num_yaw_size, M = cfg->num_mags, H = M * J;
    cudaStream_t st = (cudaStream_t)stream;
    if (!b->items || !b->cand_item_start || !b->counts) return FNP_EINVAL;
    if (cfg->variant == FNP_VARIANT_KITTI) {      // first-match counts: its own kernel, no work items
        cudaMemsetAsync(b->counts, 0, sizeof(int32_t) * (size_t)b->n_cands * H, st);
        // a frustum holds at most the rows of the largest frame: page_tab_stride pages
        int rows = (int)(((long long)b->page_tab_stride * kPage + kFmSplit - 1) / kFmSplit);
        rows = rows < 1 ? 1 : rows > 65535 ? 65535 : rows;
        firstmatch_kernel<<<dim3(b->n_cands, rows), kFmThreads, 0, st>>>(*b, H);
        FNP_LAUNCH_CHECK();
        return FNP_OK;
    }
    const int mode = resolve_score_mode(cfg, b);
    if (mode < 0) return FNP_EINVAL;
    const int sweep = mode == FNP_SCORE_SWEEP;
    // per device: a process may run engines on several GPUs (function attributes and the SM count are per device)
    static int sms_of[64] = {0};
    int dev = 0;
    cudaGetDevice(&dev);
    int n_sms = 0;
    if (dev >= 0 && dev < 64 && sms_of[dev]) n_sms = sms_of[dev];
    else {
        cudaDeviceGetAttribute(&n_sms, cudaDevAttrMultiProcessorCount, dev);
        if (dev >= 0 && dev < 64) sms_of[dev] = n_sms;
    }
    cudaMemsetAsync(b->counts, 0, sizeof(int32_t) * (size_t)b->n_cands * H, st);
    if (sweep) sweep_prep_kernel<<<b->n_cands, 128, (size_t)15 * J * 4, st>>>(*b, J, M);
    plan_items_kernel<<<1, 1024, 0, st>>>(*b, H, sweep);
    write_items_kernel<<<b->n_cands, 128, 0, st>>>(*b, H, sweep);
    if (b->max_items > 0) {
        // persistent CTAs: a whole number of CTAs per SM (148 SMs on B200), capped by the item capacity
        if (sweep) {
            const size_t smem = sweep_smem_bytes(b->split_points, H, J);
            static size_t smem_set[64] = {0};
            if (dev < 0 || dev >= 64 || smem > smem_set[dev]) {
                cudaFuncSetAttribute(sweep_score_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
                if (dev >= 0 && dev < 64) smem_set[dev] = smem;
            }
            int per_sm = 0;
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sweep_score_kernel, kSweepThreads, smem);
            if (per_sm < 1) return FNP_EINVAL;
            const int grid = b->max_items < n_sms * per_sm ? b->max_items : n_sms * per_sm;
            sweep_score_kernel<<<grid, kSweepThreads, smem, st>>>(*b, J, M);
        } else {
            const int per_sm = 6;
            const int grid = b->max_items < n_sms * per_sm ? b->max_items : n_sms * per_sm;
            score_kernel<<<grid, kScoreThreads, 0, st>>>(*b, H);
        }
    }
    FNP_LAUNCH_CHECK();
    return FNP_OK;
}

/* Which scoring kernel fnp_seeker_score would run for this batch: FNP_SCORE_DIRECT or FNP_SCORE_SWEEP
 * (FNP_EINVAL: the requested mode cannot run, e.g. SWEEP without sweep_cols). */
extern "C" int fnp_seeker_score_mode(const fnp_seeker_cfg *cfg, const fnp_seeker_batch *b)
{
    if (!cfg || !b) return FNP_EINVAL;
    const int m = resolve_score_mode(cfg, b);
    return m < 0 ? FNP_EINVAL : m;
}

extern "C" int fnp_seeker_select(const fnp_seeker_cfg *cfg, const fnp_seeker_batch *b, void *stream)
{
    int rc = check_batch(cfg, b);
    if (rc) return rc;
    const bool kitti = cfg->variant == FNP_VARIANT_KITTI;
    if (kitti && (cfg->flags != 0 || cfg->ego_w > 0.f || cfg->occl_w > 0.f)) return FNP_EINVAL;   // not terms of that head's score
    if (((cfg->dst_w != 0.f) || (cfg->flags & FNP_SEEKER_MULT) || kitti) && !b->hyp_dist) return FNP_EINVAL;
    if (((cfg->occl_w > 0.f) || (cfg->flags & FNP_SEEKER_OCCL_MULT)) && !b->hyp_nfar) return FNP_EINVAL;
    if (cfg->topk > 1 && (!b->hyp_score || cfg->num_yaw_size * cfg->num_mags > kSelectMaxTopkH)) return FNP_EINVAL;
    if (b->n_cands == 0) return FNP_OK;
    const bool extras = cfg->dst_w != 0.f || cfg->ego_w > 0.f || cfg->occl_w > 0.f || cfg->flags != 0 || cfg->topk > 1 || kitti;
    if (extras)
        select_kernel<true><<<b->n_cands, 128, 0, (cudaStream_t)stream>>>(*b, *cfg);
    else
        select_kernel<false><<<b->n_cands, 128, 0, (cudaStream_t)stream>>>(*b, *cfg);
    FNP_LAUNCH_CHECK();
    return FNP_OK;
}

extern "C" int fnp_seeker_select_multi(const fnp_seeker_cfg *cfg, const fnp_seeker_batch *b,
                                       const fnp_select_setting *settings_host, int n_settings, float *out_boxes,
                                       float *out_score, int32_t *out_best, int32_t *out_count, void *stream)
{
    int rc = check_batch(cfg, b);
    if (rc) return rc;
    if (!settings_host || n_settings < 1 || n_settings > FNP_SELECT_MAX_SETTINGS) return FNP_EINVAL;
    // topk > 1: the suppression pass is not repeated per setting
    if (cfg->topk > 1) return FNP_EINVAL;
    const bool kitti = cfg->variant == FNP_VARIANT_KITTI;
    SelectSettings set = {};
    int planes = kitti ? kMultiPlaneDist : 0;
    for (int i = 0; i < n_settings; i++) {
        const fnp_select_setting &s = settings_host[i];
        if (s.flags & ~(FNP_SEEKER_MULT | FNP_SEEKER_OCCL_MULT)) return FNP_EINVAL;
        if (!(s.min_cam_iou >= cfg->min_cam_iou)) return FNP_EINVAL;    // compacted at cfg's threshold
        if (kitti) {
            // first-match counts depend on the valid set: only the one stages 1-2c compacted, and only that head's terms
            uint32_t a, c;
            memcpy(&a, &s.min_cam_iou, 4);
            memcpy(&c, &cfg->min_cam_iou, 4);
            if (a != c || s.flags != 0 || s.ego_w > 0.f || s.occl_w > 0.f) return FNP_EINVAL;
        }
        if ((s.dst_w != 0.f) || (s.flags & FNP_SEEKER_MULT)) planes |= kMultiPlaneDist;
        if ((s.occl_w > 0.f) || (s.flags & FNP_SEEKER_OCCL_MULT)) planes |= kMultiPlaneFail;
        if (s.ego_w > 0.f) planes |= kMultiPlaneEgo;
        set.s[i] = s;
    }
    if (((planes & kMultiPlaneDist) && !b->hyp_dist) || ((planes & kMultiPlaneFail) && !b->hyp_nfar)) return FNP_EINVAL;
    if (b->n_cands == 0) return FNP_OK;
    if (!out_boxes || !out_score || !out_best || !out_count || !b->counts) return FNP_EINVAL;
    const int J = cfg->num_yaw_size, H = J * cfg->num_mags;
    const size_t smem = (size_t)H * 4 * (2 + __builtin_popcount(planes));
    if (smem > 200 * 1024) return FNP_EINVAL;
    auto kernel = kitti ? select_multi_kernel<true> : select_multi_kernel<false>;
    cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    kernel<<<b->n_cands, kMultiThreads, smem, (cudaStream_t)stream>>>(*b, J, H, set, n_settings, planes, out_boxes,
                                                                      out_score, out_best, out_count);
    FNP_LAUNCH_CHECK();
    return FNP_OK;
}

extern "C" int fnp_seeker_occlusion(const fnp_seeker_cfg *cfg, const fnp_seeker_batch *b, void *stream)
{
    int rc = check_batch(cfg, b);
    if (rc) return rc;
    if (!(cfg->occl_w > 0.f) && !(cfg->flags & FNP_SEEKER_OCCL_MULT)) return FNP_OK;
    if (!b->hyp_nfar) return FNP_EINVAL;
    if (b->n_cands == 0) return FNP_OK;
    const int J = cfg->num_yaw_size, H = J * cfg->num_mags;
    occl_kernel<<<dim3(b->n_cands, divup(H, kOcclThreads)), kOcclThreads, 0, (cudaStream_t)stream>>>(*b, J, H);
    FNP_LAUNCH_CHECK();
    return FNP_OK;
}

extern "C" int fnp_seeker_run(const fnp_seeker_cfg *cfg, const fnp_seeker_batch *b, void *stream)
{
    int rc;
    if ((rc = fnp_seeker_cull(cfg, b, stream))) return rc;
    if ((rc = fnp_seeker_frustum_stats(cfg, b, stream))) return rc;
    if ((rc = fnp_seeker_hypotheses(cfg, b, stream))) return rc;
    if ((rc = fnp_seeker_score(cfg, b, stream))) return rc;
    if ((rc = fnp_seeker_occlusion(cfg, b, stream))) return rc;
    return fnp_seeker_select(cfg, b, stream);
}
