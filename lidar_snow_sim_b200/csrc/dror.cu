// dror.cu -- dynamic radius outlier removal (DROR) of device-resident clouds, batched.
//
// Replaces dynamic_radius_outlier_filter (lib/cadc_devkit/other/dror.py:288-334): a Python loop with one FLANN k-NN query
// per point, whose results the DENSE data path reads back from per-frame pickles (dense_dataset.py:588-616).  The rule
// it computes, restated without k-NN (DESIGN.md 7.4): with
//     sr_i  = max(alpha * beta * pi / 180 * sqrt(x_i^2 + y_i^2), sr_min)           float64, in the reference's order
//     d2_ij = ((0 + dx^2) + dy^2) + dz^2,  dx = x_i - x_j, ...                      float32, FLANN's L2_Simple order
//     c_i   = #{ j in the cloud, i included : sqrt((double)d2_ij) < sr_i }
// point i is kept iff c_i >= k_min + 1.  The count is an integer: the result is exact and deterministic.
//
//   k_dror_keys     per row: 64-bit key = cloud | invalid | 3-D Morton code of a uniform grid (finest cell C0, clamped at
//                   the grid edge); rows outside the crop / behind the cloud's count get the invalid bit
//   cub::DeviceRadixSort::SortPairs   (key, row) of the whole batch, stable: cloud b stays in its slot, valid rows first
//   k_dror_gather   xyz of the sorted rows as float4
//   k_dror_query    per sorted row: ~9 sorted neighbours first (enough for most kept points), else every point of the
//                   <= 8 cells of level L (cell >= 2 * padded sr) that meet the query box; stops at k_min + 1 hits
//   cub::DeviceScan::ExclusiveSum     of (kept + snow << 32) per row: the stable, slot-compacted destination of every
//                   kept row and, per cloud, the kept and snow counts
//   k_dror_counts / k_dror_scatter
//
// CUB (from the CUDA toolkit's headers) does the sort and the scan: a stable 45-bit radix sort of 4 M pairs and a 64-bit
// scan are library-grade primitives, and neither needs anything the rule would specialise.
//
// Invariants (tested in tests/test_dror.py with a NumPy model of the search, and on the device against the oracle):
//   completeness   the cell function floor((v - ORIGIN) / C0), clamped to [0, 2^13), is monotone in v (evaluated in
//                  float64, where it is exact for float32 inputs).  A point j the rule admits satisfies
//                  |x_j - x_i| < sr_i * (1 + 2^-18) + 1e-6 per axis (float32 rounding of d2 is at most 5 ulps), so it
//                  lies in the padded box and its cell in one of the visited cells.  Scanning more points than the
//                  cells hold is harmless: every candidate is tested with the exact rule.
//   arithmetic     d2 with __fmul_rn / __fadd_rn (no FMA); sr in float64, (((alpha * beta) * pi) / 180) * r.
//   determinism    no atomics; the sort is stable and a cloud's rows never leave its slot.
#include "common.cuh"
#include <cmath>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

namespace {

constexpr int DROR_TPB = 256;
constexpr double GRID_ORIGIN = -512.0;          // m, every axis
constexpr double GRID_INV_C0 = 8.0;             // finest cell C0 = 1/8 m
constexpr double GRID_C0 = 0.125;
constexpr int GRID_BITS = 13;                   // 8192 cells of C0 per axis: +-512 m
constexpr int GRID_MAX = (1 << GRID_BITS) - 1;
constexpr int KEY_CLOUD_SHIFT = 40;             // bits 0..38 Morton code, bit 39 invalid, bits 40.. cloud index
constexpr unsigned long long KEY_INVALID = 1ull << 39;
constexpr double PAD_REL = 1.0 / 262144.0;      // 2^-18
constexpr double PAD_ABS = 1e-6;                // m
constexpr int WINDOW = 4;                       // sorted neighbours on each side tried first

struct DrorArgs {
    const float *pts;
    int F;
    const int64_t *cloud_off;        // [B+1] device
    const int32_t *cloud_cnt;        // [B] or NULL
    int n_clouds;
    int64_t n_total;
    double sr_scale;                 // alpha * beta * pi / 180, evaluated left to right on the host
    double sr_min;
    int need;                        // k_min + 1
    int crop;
    float cx0, cx1, cy0, cy1;
    unsigned long long *key;         // [N] input keys of the sort
    int *row;                        // [N] input values of the sort
    const unsigned long long *skey;  // [N] sorted keys
    const int *srow;                 // [N] sorted rows
    float4 *sxyz;                    // [N] sorted xyz
    unsigned long long *flag;        // [N+1] kept + (snow << 32) per row
    const unsigned long long *scan;  // [N+1] exclusive scan of flag
    uint8_t *codes;                  // [N] 0 snow, 1 kept, 2 outside the crop
    float *out;                      // [N*F] or NULL
    int32_t *out_counts, *out_n_snow;
};

__device__ __forceinline__ int cloud_rows(const DrorArgs &a, int b)
{
    return a.cloud_cnt ? a.cloud_cnt[b] : (int)(a.cloud_off[b + 1] - a.cloud_off[b]);
}

// grid cell of a coordinate: monotone (non-decreasing) in v, clamping included; exact for float32 inputs
__device__ __forceinline__ int grid_cell(double v)
{
    const double c = floor((v - GRID_ORIGIN) * GRID_INV_C0);
    if (!(c > 0.0)) return 0;                   // NaN lands in cell 0
    return c > (double)GRID_MAX ? GRID_MAX : (int)c;
}

__device__ __forceinline__ unsigned long long spread3(unsigned v)
{
    unsigned long long x = v & 0x1fffffu;
    x = (x | (x << 32)) & 0x1f00000000ffffull;
    x = (x | (x << 16)) & 0x1f0000ff0000ffull;
    x = (x | (x << 8)) & 0x100f00f00f00f00full;
    x = (x | (x << 4)) & 0x10c30c30c30c30c3ull;
    x = (x | (x << 2)) & 0x1249249249249249ull;
    return x;
}

__device__ __forceinline__ unsigned long long morton3(unsigned cx, unsigned cy, unsigned cz)
{
    return spread3(cx) | (spread3(cy) << 1) | (spread3(cz) << 2);
}

// the reference's per-point search radius (dror.py:316-321): r = np.linalg.norm([x, y]) in float64
__device__ __forceinline__ double search_radius(const DrorArgs &a, float x, float y)
{
    const double xd = x, yd = y;
    const double r = sqrt(__dadd_rn(__dmul_rn(xd, xd), __dmul_rn(yd, yd)));
    const double sr = __dmul_rn(a.sr_scale, r);
    return sr < a.sr_min ? a.sr_min : sr;
}

// FLANN L2_Simple (flann/algorithms/dist.h): ((0 + dx*dx) + dy*dy) + dz*dz in float32, each step rounded
__device__ __forceinline__ float l2_simple(float4 q, float4 p)
{
    const float dx = __fsub_rn(q.x, p.x), dy = __fsub_rn(q.y, p.y), dz = __fsub_rn(q.z, p.z);
    return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
}

// The test sqrt((double)d2) < sr of dror.py:329-331 for a float32 d2 is d2 <= hit_limit(sr): sqrt is correctly rounded
// and non-decreasing, so the float32 values that pass are all values up to the largest one that does.  Found from
// (float)(sr * sr) in a step or two, once per query point, so that the candidate loop compares float32 only.
__device__ __forceinline__ float hit_limit(double sr)
{
    float f = (float)(sr * sr);
    while (f > 0.0f && !(sqrt((double)f) < sr)) f = nextafterf(f, 0.0f);
    for (;;) {
        const float up = nextafterf(f, INFINITY);
        if (up == INFINITY || !(sqrt((double)up) < sr)) return f;
        f = up;
    }
}

__global__ void __launch_bounds__(DROR_TPB) k_dror_keys(DrorArgs a)
{
    const int b = blockIdx.y;
    const int64_t beg = a.cloud_off[b];
    const int slot = (int)(a.cloud_off[b + 1] - beg);
    const int n = cloud_rows(a, b);
    for (int i = blockIdx.x * DROR_TPB + threadIdx.x; i < slot; i += gridDim.x * DROR_TPB) {
        const int64_t r = beg + i;
        unsigned long long key = (unsigned long long)b << KEY_CLOUD_SHIFT;
        if (i < n) {
            const float *p = a.pts + r * a.F;
            const float x = p[0], y = p[1], z = p[2];
            // get_cube_mask (dror.py:73-84): np.logical_and(x_mask, y_mask, z_mask) passes z_mask as `out`, z is ignored
            if (a.crop && !(a.cx0 <= x && x <= a.cx1 && a.cy0 <= y && y <= a.cy1)) {
                key |= KEY_INVALID;
                a.codes[r] = 2;
            } else {
                key |= morton3(grid_cell(x), grid_cell(y), grid_cell(z));
            }
        } else {
            key |= KEY_INVALID;
        }
        a.key[r] = key;
        a.row[r] = (int)r;
        a.flag[r] = 0ull;
    }
    if (b == a.n_clouds - 1 && blockIdx.x == 0 && threadIdx.x == 0) a.flag[a.n_total] = 0ull;
}

__global__ void __launch_bounds__(DROR_TPB) k_dror_gather(DrorArgs a)
{
    const int64_t p = (int64_t)blockIdx.x * DROR_TPB + threadIdx.x;
    if (p >= a.n_total) return;
    const float *s = a.pts + (int64_t)a.srow[p] * a.F;
    a.sxyz[p] = make_float4(s[0], s[1], s[2], 0.0f);
}

// first position in [lo, hi) whose sorted key is >= k
__device__ __forceinline__ int64_t lower_bound(const unsigned long long *key, int64_t lo, int64_t hi, unsigned long long k)
{
    while (lo < hi) {
        const int64_t mid = lo + ((hi - lo) >> 1);
        if (key[mid] < k) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

__global__ void __launch_bounds__(DROR_TPB) k_dror_query(DrorArgs a)
{
    const int64_t p = (int64_t)blockIdx.x * DROR_TPB + threadIdx.x;
    if (p >= a.n_total) return;
    const unsigned long long kp = a.skey[p];
    if (kp & KEY_INVALID) return;
    const int b = (int)(kp >> KEY_CLOUD_SHIFT);
    const int64_t seg_lo = a.cloud_off[b], seg_hi = a.cloud_off[b + 1];
    const float4 q = a.sxyz[p];
    const double sr = search_radius(a, q.x, q.y);
    const unsigned long long tag = kp >> 39;                   // cloud and the (clear) invalid bit
    // sr <= 0 (sr_min <= 0 at the origin) or NaN: no distance is below it, not even the point's own
    const bool open = sr > 0.0;
    const float lim = open ? hit_limit(sr) : 0.0f;
    // sorted neighbours: the Morton order puts most of a surface point's neighbours next to it.  A lower bound of c_i
    int hits = 0;
    const int64_t w0 = p - WINDOW > seg_lo ? p - WINDOW : seg_lo, w1 = p + WINDOW + 1 < seg_hi ? p + WINDOW + 1 : seg_hi;
    for (int64_t j = w0; open && j < w1 && hits < a.need; j++)
        if ((a.skey[j] >> 39) == tag && l2_simple(q, a.sxyz[j]) <= lim) hits++;
    bool keep = hits >= a.need;
    if (open && !keep) {
        // every point of the <= 8 level-L cells that meet the padded box [q - rp, q + rp]
        const double rp = sr * (1.0 + PAD_REL) + PAD_ABS;
        int L = 0;
        while (L < GRID_BITS && GRID_C0 * (double)(1 << L) < 2.0 * rp) L++;
        const int x0 = grid_cell((double)q.x - rp) >> L, x1 = grid_cell((double)q.x + rp) >> L;
        const int y0 = grid_cell((double)q.y - rp) >> L, y1 = grid_cell((double)q.y + rp) >> L;
        const int z0 = grid_cell((double)q.z - rp) >> L, z1 = grid_cell((double)q.z + rp) >> L;
        const unsigned long long base = (unsigned long long)b << KEY_CLOUD_SHIFT;
        const int sh = 3 * L;
        // the key range spanned by all the cells; scanned directly when it is short
        const unsigned long long kmin = base | (morton3(x0, y0, z0) << sh);
        const unsigned long long kmax = base | ((morton3(x1, y1, z1) + 1ull) << sh);
        const int64_t lo0 = lower_bound(a.skey, seg_lo, seg_hi, kmin);
        const int64_t hi0 = lower_bound(a.skey, lo0, seg_hi, kmax);
        hits = 0;
        if (hi0 - lo0 <= 64) {
            for (int64_t j = lo0; j < hi0 && hits < a.need; j++)
                if (l2_simple(q, a.sxyz[j]) <= lim) hits++;
        } else {
            for (int cz = z0; cz <= z1 && hits < a.need; cz++)
                for (int cy = y0; cy <= y1 && hits < a.need; cy++)
                    for (int cx = x0; cx <= x1 && hits < a.need; cx++) {
                        const unsigned long long m = morton3(cx, cy, cz);
                        const int64_t j0 = lower_bound(a.skey, lo0, hi0, base | (m << sh));
                        const int64_t j1 = lower_bound(a.skey, j0, hi0, base | ((m + 1ull) << sh));
                        for (int64_t j = j0; j < j1 && hits < a.need; j++)
                            if (l2_simple(q, a.sxyz[j]) <= lim) hits++;
                    }
        }
        keep = hits >= a.need;
    }
    const int r = a.srow[p];
    a.codes[r] = keep ? 1 : 0;
    a.flag[r] = keep ? 1ull : (1ull << 32);
}

__global__ void k_dror_counts(DrorArgs a)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= a.n_clouds) return;
    const unsigned long long d = a.scan[a.cloud_off[b + 1]] - a.scan[a.cloud_off[b]];
    a.out_counts[b] = (int32_t)(d & 0xffffffffull);
    a.out_n_snow[b] = (int32_t)(d >> 32);
}

// stable slot compaction: kept row r of cloud b goes to off[b] + (kept rows of b before r)
__global__ void __launch_bounds__(DROR_TPB) k_dror_scatter(DrorArgs a)
{
    const int b = blockIdx.y;
    const int64_t beg = a.cloud_off[b];
    const int n = cloud_rows(a, b);
    const unsigned long long s0 = a.scan[beg];
    for (int i = blockIdx.x * DROR_TPB + threadIdx.x; i < n; i += gridDim.x * DROR_TPB) {
        const int64_t r = beg + i;
        if (!(a.flag[r] & 1ull)) continue;
        const int64_t dst = beg + (int64_t)((a.scan[r] - s0) & 0xffffffffull);
        const float *s = a.pts + r * a.F;
        float *o = a.out + dst * a.F;
        for (int f = 0; f < a.F; f++) o[f] = s[f];
    }
}

inline int64_t align_up(int64_t v, int64_t al) { return (v + al - 1) / al * al; }

int sort_end_bit(int n_clouds)
{
    int bits = 0;
    while (bits < 24 && (1ll << bits) < (int64_t)n_clouds) bits++;
    return KEY_CLOUD_SHIFT + bits;
}

struct DrorLayout { int64_t off, key0, key1, row0, row1, sxyz, flag, scan, temp, temp_bytes, total; };

// -1 if CUB cannot size its scratch (no usable CUDA device)
DrorLayout dror_layout(int64_t n_total, int n_clouds)
{
    DrorLayout L;
    L.total = -1;
    const int n = (int)n_total;
    size_t sort_bytes = 0, scan_bytes = 0;
    cub::DoubleBuffer<unsigned long long> dk(nullptr, nullptr);
    cub::DoubleBuffer<int> dv(nullptr, nullptr);
    if (cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, dk, dv, n, 0, sort_end_bit(n_clouds)) != cudaSuccess)
        return L;
    if (cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, (const unsigned long long *)nullptr,
                                      (unsigned long long *)nullptr, n + 1) != cudaSuccess)
        return L;
    L.temp_bytes = (int64_t)std::max(sort_bytes, scan_bytes);
    int64_t o = 0;
    L.off = o;   o = align_up(o + (int64_t)(n_clouds + 1) * 8, 256);
    L.key0 = o;  o = align_up(o + n_total * 8, 256);
    L.key1 = o;  o = align_up(o + n_total * 8, 256);
    L.row0 = o;  o = align_up(o + n_total * 4, 256);
    L.row1 = o;  o = align_up(o + n_total * 4, 256);
    L.sxyz = o;  o = align_up(o + n_total * 16, 256);
    L.flag = o;  o = align_up(o + (n_total + 1) * 8, 256);
    L.scan = o;  o = align_up(o + (n_total + 1) * 8, 256);
    L.temp = o;  o = align_up(o + L.temp_bytes, 256);
    L.total = o;
    return L;
}

}  // namespace

extern "C" {

int64_t lss_dror_workspace_bytes(int64_t n_total, int n_clouds)
{
    if (n_total < 0 || n_total >= (1ll << 31) - 1 || n_clouds < 0) return -1;
    return dror_layout(n_total, n_clouds).total;
}

lss_status lss_dror_batch(lss_engine *e, const float *d_points, int n_features, const int64_t *h_cloud_offsets,
                          const int32_t *d_cloud_counts, int n_clouds, double alpha_deg, double beta, int k_min,
                          double sr_min, const float *h_crop_xy, uint8_t *d_codes, float *d_out_points,
                          int32_t *d_out_counts, int32_t *d_out_n_snow, void *d_workspace, int64_t workspace_bytes,
                          void *stream)
{
    if (!e) return LSS_ERR_INVALID_ARG;
    if (!h_cloud_offsets || n_clouds < 0 || !d_out_counts || !d_out_n_snow)
        return lss_fail(e, LSS_ERR_INVALID_ARG, "null argument");
    if (n_features < 3) return lss_fail(e, LSS_ERR_INVALID_ARG, "n_features >= 3 required");
    if (k_min < 0) return lss_fail(e, LSS_ERR_INVALID_ARG, "k_min >= 0 required");
    if (!std::isfinite(alpha_deg) || !std::isfinite(beta) || !std::isfinite(sr_min))
        return lss_fail(e, LSS_ERR_INVALID_ARG, "alpha, beta and sr_min must be finite");
    if (n_clouds > 65535) return lss_fail(e, LSS_ERR_INVALID_ARG, "at most 65535 clouds per call");
    if (h_cloud_offsets[0] != 0) return lss_fail(e, LSS_ERR_INVALID_ARG, "cloud_offsets[0] must be 0");
    const int B = n_clouds;
    const int64_t N = h_cloud_offsets[B];
    if (N >= (1ll << 31) - 1) return lss_fail(e, LSS_ERR_INVALID_ARG, "batch too large");
    int64_t max_n = 0;
    for (int b = 0; b < B; b++) {
        const int64_t nb = h_cloud_offsets[b + 1] - h_cloud_offsets[b];
        if (nb < 0) return lss_fail(e, LSS_ERR_INVALID_ARG, "cloud_offsets must be non-decreasing");
        max_n = std::max(max_n, nb);
    }
    DeviceGuard g(e->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (B == 0 || N == 0) {
        ZeroRegions z;
        z.add(d_out_counts, sizeof(int32_t) * B);
        z.add(d_out_n_snow, sizeof(int32_t) * B);
        LSS_CUDA_CHECK(e, lss_zero_async(e, z, st));
        return LSS_OK;
    }
    if (!d_points || !d_codes || !d_workspace) return lss_fail(e, LSS_ERR_INVALID_ARG, "null argument");
    const DrorLayout L = dror_layout(N, B);
    if (L.total < 0) return lss_fail(e, LSS_ERR_CUDA, "cannot size the sort / scan scratch");
    if (workspace_bytes < L.total) return lss_fail(e, LSS_ERR_WORKSPACE, "workspace too small");
    char *ws = (char *)d_workspace;
    DrorArgs a;
    a.pts = d_points;
    a.F = n_features;
    a.cloud_off = (const int64_t *)(ws + L.off);
    a.cloud_cnt = d_cloud_counts;
    a.n_clouds = B;
    a.n_total = N;
    a.sr_scale = alpha_deg * beta * LSS_PI / 180.0;              // dror.py:318, left to right
    a.sr_min = sr_min;
    a.need = k_min + 1;                                          // k = k_min + 1 neighbours, self included (:307, :323)
    a.crop = h_crop_xy != nullptr;
    a.cx0 = a.crop ? h_crop_xy[0] : 0.0f;
    a.cx1 = a.crop ? h_crop_xy[1] : 0.0f;
    a.cy0 = a.crop ? h_crop_xy[2] : 0.0f;
    a.cy1 = a.crop ? h_crop_xy[3] : 0.0f;
    a.flag = (unsigned long long *)(ws + L.flag);
    a.scan = (const unsigned long long *)(ws + L.scan);
    a.sxyz = (float4 *)(ws + L.sxyz);
    a.codes = d_codes;
    a.out = d_out_points;
    a.out_counts = d_out_counts;
    a.out_n_snow = d_out_n_snow;
    cub::DoubleBuffer<unsigned long long> dk((unsigned long long *)(ws + L.key0), (unsigned long long *)(ws + L.key1));
    cub::DoubleBuffer<int> dv((int *)(ws + L.row0), (int *)(ws + L.row1));
    a.key = dk.Current();
    a.row = dv.Current();
    LSS_CUDA_CHECK(e, lss_stage_upload(e, ws + L.off, h_cloud_offsets, sizeof(int64_t) * (B + 1), st));
    const unsigned row_blocks = (unsigned)std::max<int64_t>(1, std::min<int64_t>(256, (max_n + DROR_TPB - 1) / DROR_TPB));
    const unsigned all_blocks = (unsigned)((N + DROR_TPB - 1) / DROR_TPB);
    k_dror_keys<<<dim3(row_blocks, B), DROR_TPB, 0, st>>>(a);
    LSS_CUDA_CHECK(e, cudaGetLastError());
    size_t temp_bytes = (size_t)L.temp_bytes;
    LSS_CUDA_CHECK(e, cub::DeviceRadixSort::SortPairs(ws + L.temp, temp_bytes, dk, dv, (int)N, 0, sort_end_bit(B), st));
    a.skey = dk.Current();
    a.srow = dv.Current();
    k_dror_gather<<<all_blocks, DROR_TPB, 0, st>>>(a);
    k_dror_query<<<all_blocks, DROR_TPB, 0, st>>>(a);
    LSS_CUDA_CHECK(e, cudaGetLastError());
    temp_bytes = (size_t)L.temp_bytes;
    LSS_CUDA_CHECK(e, cub::DeviceScan::ExclusiveSum(ws + L.temp, temp_bytes, (const unsigned long long *)a.flag,
                                                     (unsigned long long *)(ws + L.scan), (int)N + 1, st));
    k_dror_counts<<<(B + 127) / 128, 128, 0, st>>>(a);
    if (d_out_points) k_dror_scatter<<<dim3(row_blocks, B), DROR_TPB, 0, st>>>(a);
    LSS_CUDA_CHECK(e, cudaGetLastError());
    e->launches += 4 + 2 + (d_out_points ? 1 : 0);               // + the radix sort's and the scan's own launches
    return LSS_OK;
}

}  // extern "C"
