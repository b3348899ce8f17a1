// project.cuh -- the GPD baseline's image projection (reference: PointNetGPD/model/dataset.py:78-198, collect_pc with
// projection=True) for one cloud and many grasps, on CUDA cores:
//   1. a hash grid over the cloud (cell = search radius 0.1), built once per call;
//   2. up to 30 nearest neighbours within radius 0.1 (the point itself included) of every point that lies in at least
//      one valid box -- searched once per point, in the cloud frame (distances do not depend on the grasp frame);
//   3. per (grasp, in-box point): covariance of the neighbours' grasp-frame coordinates in fp64 and the eigenvector of
//      its smallest eigenvalue (closed-form symmetric 3x3 solver, below).  Computed per grasp because the solver's sign
//      is not rotation-equivariant;
//   4. per (grasp, axis order): voxel keys, a block-wide bitonic sort of (key, input position), the first-50-points
//      rule, the largest-z-wins pixel scatter and the occupancy normalisation.
// Every sum runs in a fixed order and no atomics decide a value, so the images are bit-reproducible from run to run.
#pragma once
#include "common.cuh"

namespace pgpd {
namespace proj {

constexpr int IMG = 60;               // project_size (dataset.py:220-222)
constexpr int PIX = IMG * IMG;
constexpr int MAX_NN = 30;            // KDTreeSearchParamHybrid(radius=0.1, max_nn=30), dataset.py:78
constexpr double RADIUS = 0.1;
constexpr int VOXEL_CAP = 50;         // voxel_point_num, dataset.py:223
constexpr int MIN_POINTS = 50;        // min_point_limit, dataset.py:71
constexpr unsigned long long DROPPED = ~0ull;   // sort key of a point whose normal has a NaN (sorts last)

// ---- closed-form eigenvector of the smallest eigenvalue of a symmetric 3x3 matrix -------------------------------------
// D. Eberly, "A Robust Eigensolver for 3 x 3 Symmetric Matrices" (Geometric Tools, 2014): eigenvalues from the
// trigonometric solution of the characteristic cubic of the max-normalised matrix; the eigenvector of the eigenvalue
// that is simple by construction from the largest cross product of two rows of A - eI; the second from the 2x2 problem
// in the plane orthogonal to the first; the third as their cross product.  Point-cloud libraries use this form as
// their fast normal solver.  The sign it returns follows from the arithmetic alone (no orientation step).
struct V3 { double x, y, z; };
__device__ __forceinline__ V3 v3_cross(V3 a, V3 b) { return V3{a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }
__device__ __forceinline__ double v3_dot(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }

// a = (a00, a01, a02, a11, a12, a22)
__device__ inline V3 evec_of_simple(const double* a, double e) {
    const V3 r0{a[0] - e, a[1], a[2]}, r1{a[1], a[3] - e, a[4]}, r2{a[2], a[4], a[5] - e};
    const V3 c0 = v3_cross(r0, r1), c1 = v3_cross(r0, r2), c2 = v3_cross(r1, r2);
    const double d0 = v3_dot(c0, c0), d1 = v3_dot(c1, c1), d2 = v3_dot(c2, c2);
    double dmax = d0;
    int imax = 0;
    if (d1 > dmax) { dmax = d1; imax = 1; }
    if (d2 > dmax) imax = 2;
    const V3 c = imax == 0 ? c0 : (imax == 1 ? c1 : c2);
    const double s = sqrt(imax == 0 ? d0 : (imax == 1 ? d1 : d2));
    return V3{c.x / s, c.y / s, c.z / s};
}

// eigenvector of eigenvalue e orthogonal to the unit eigenvector w
__device__ inline V3 evec_orthogonal(const double* a, V3 w, double e) {
    V3 u;
    if (fabs(w.x) > fabs(w.y)) {
        const double inv = 1.0 / sqrt(w.x * w.x + w.z * w.z);
        u = V3{-w.z * inv, 0.0, w.x * inv};
    } else {
        const double inv = 1.0 / sqrt(w.y * w.y + w.z * w.z);
        u = V3{0.0, w.z * inv, -w.y * inv};
    }
    const V3 v = v3_cross(w, u);
    const V3 au{a[0] * u.x + a[1] * u.y + a[2] * u.z, a[1] * u.x + a[3] * u.y + a[4] * u.z, a[2] * u.x + a[4] * u.y + a[5] * u.z};
    const V3 av{a[0] * v.x + a[1] * v.y + a[2] * v.z, a[1] * v.x + a[3] * v.y + a[4] * v.z, a[2] * v.x + a[4] * v.y + a[5] * v.z};
    // (m00 m01; m01 m11) annihilates the eigenvector's (u, v) coordinates: take the normalised row of larger norm, rotated
    double m00 = v3_dot(u, au) - e, m01 = v3_dot(u, av), m11 = v3_dot(v, av) - e;
    const double f00 = fabs(m00), f01 = fabs(m01), f11 = fabs(m11);
    if (f00 >= f11) {
        if (fmax(f00, f01) <= 0.0) return u;
        if (f00 >= f01) { m01 /= m00; m00 = 1.0 / sqrt(1.0 + m01 * m01); m01 *= m00; }
        else            { m00 /= m01; m01 = 1.0 / sqrt(1.0 + m00 * m00); m00 *= m01; }
        return V3{m01 * u.x - m00 * v.x, m01 * u.y - m00 * v.y, m01 * u.z - m00 * v.z};
    }
    if (fmax(f11, f01) <= 0.0) return u;
    if (f11 >= f01) { m01 /= m11; m11 = 1.0 / sqrt(1.0 + m01 * m01); m01 *= m11; }
    else            { m11 /= m01; m01 = 1.0 / sqrt(1.0 + m11 * m11); m11 *= m01; }
    return V3{m11 * u.x - m01 * v.x, m11 * u.y - m01 * v.y, m11 * u.z - m01 * v.z};
}

// cov = (c00, c01, c02, c11, c12, c22).  Returns the zero vector when every entry is <= 0 with a zero maximum.
__device__ inline V3 smallest_eigenvector(const double* cov) {
    double mx = cov[0];
    for (int i = 1; i < 6; ++i) mx = fmax(mx, cov[i]);
    if (mx == 0.0) return V3{0.0, 0.0, 0.0};
    double a[6];
    for (int i = 0; i < 6; ++i) a[i] = cov[i] / mx;
    const double off = a[1] * a[1] + a[2] * a[2] + a[4] * a[4];
    if (off > 0.0) {
        const double q = (a[0] + a[3] + a[5]) / 3.0;
        const double b00 = a[0] - q, b11 = a[3] - q, b22 = a[5] - q;
        const double p = sqrt((b00 * b00 + b11 * b11 + b22 * b22 + off * 2.0) / 6.0);
        const double c00 = b11 * b22 - a[4] * a[4], c01 = a[1] * b22 - a[4] * a[2], c02 = a[1] * a[4] - b11 * a[2];
        const double det = (b00 * c00 - a[1] * c01 + a[2] * c02) / (p * p * p);
        const double hd = fmin(fmax(det * 0.5, -1.0), 1.0);
        const double ang = acos(hd) / 3.0;
        const double beta2 = cos(ang) * 2.0, beta0 = cos(ang + 2.09439510239319549) * 2.0, beta1 = -(beta0 + beta2);
        const double e0 = q + p * beta0, e1 = q + p * beta1, e2 = q + p * beta2;
        if (hd >= 0.0) {
            const V3 w2 = evec_of_simple(a, e2);
            if (e2 < e0 && e2 < e1) return w2;
            const V3 w1 = evec_orthogonal(a, w2, e1);
            if (e1 < e0 && e1 < e2) return w1;
            return v3_cross(w1, w2);
        }
        const V3 w0 = evec_of_simple(a, e0);
        if (e0 < e1 && e0 < e2) return w0;
        const V3 w1 = evec_orthogonal(a, w0, e1);
        if (e1 < e0 && e1 < e2) return w1;
        return v3_cross(w0, w1);
    }
    // diagonal: the axis of the smallest diagonal entry of the unscaled matrix, z on ties
    if (cov[0] < cov[3] && cov[0] < cov[5]) return V3{1.0, 0.0, 0.0};
    if (cov[3] < cov[0] && cov[3] < cov[5]) return V3{0.0, 1.0, 0.0};
    return V3{0.0, 0.0, 1.0};
}

// grasp-frame coordinates of cloud point j -- the arithmetic of k_crop_box
__device__ __forceinline__ V3 to_grasp(const float* __restrict__ pc, int j, const double* __restrict__ f) {
    const double px = (double)pc[(size_t)j * 3 + 0] - f[0], py = (double)pc[(size_t)j * 3 + 1] - f[1], pz = (double)pc[(size_t)j * 3 + 2] - f[2];
    return V3{f[3] * px + f[4] * py + f[5] * pz, f[6] * px + f[7] * py + f[8] * pz, f[9] * px + f[10] * py + f[11] * pz};
}

// ---- 1. hash grid ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int cell_coord(float v) {
    const double c = floor((double)v / RADIUS);
    return (int)fmin(fmax(c, -1.0e9), 1.0e9);
}
__device__ __forceinline__ unsigned cell_hash(int x, int y, int z, unsigned mask) {
    return ((unsigned)x * 73856093u ^ (unsigned)y * 19349663u ^ (unsigned)z * 83492791u) & mask;
}

__global__ void k_grid_count(const float* __restrict__ pc, int P, unsigned mask, int* __restrict__ bucket_cnt) {
    const int i = (int)(blockIdx.x * blockDim.x + threadIdx.x);
    if (i >= P) return;
    atomicAdd(&bucket_cnt[cell_hash(cell_coord(pc[(size_t)i * 3]), cell_coord(pc[(size_t)i * 3 + 1]), cell_coord(pc[(size_t)i * 3 + 2]), mask)], 1);
}

// exclusive prefix sum of H bucket counts -> start[0..H] and a copy in cursor[0..H); one block of 1024 threads
__global__ void k_grid_scan(const int* __restrict__ bucket_cnt, int H, int* __restrict__ start, int* __restrict__ cursor) {
    __shared__ int part[1024];
    const int tid = (int)threadIdx.x, chunk = (H + 1023) / 1024;
    const int b0 = min(tid * chunk, H), b1 = min(b0 + chunk, H);
    int s = 0;
    for (int b = b0; b < b1; ++b) s += bucket_cnt[b];
    part[tid] = s;
    __syncthreads();
    if (tid == 0) {
        int run = 0;
        for (int t = 0; t < 1024; ++t) { const int v = part[t]; part[t] = run; run += v; }
        start[H] = run;
    }
    __syncthreads();
    int run = part[tid];
    for (int b = b0; b < b1; ++b) { start[b] = run; cursor[b] = run; run += bucket_cnt[b]; }
}

// the order of points inside a bucket depends on atomic timing; nothing downstream depends on it (neighbours are
// selected and summed in (distance, index) order)
__global__ void k_grid_fill(const float* __restrict__ pc, int P, unsigned mask, int* __restrict__ cursor, int* __restrict__ cell_pts) {
    const int i = (int)(blockIdx.x * blockDim.x + threadIdx.x);
    if (i >= P) return;
    const unsigned h = cell_hash(cell_coord(pc[(size_t)i * 3]), cell_coord(pc[(size_t)i * 3 + 1]), cell_coord(pc[(size_t)i * 3 + 2]), mask);
    cell_pts[atomicAdd(&cursor[h], 1)] = i;
}

// ---- 2. which points need a normal: those in a box with >= MIN_POINTS points -----------------------------------------
__global__ void k_mark_needed(const int* __restrict__ offsets, int cap, const int* __restrict__ idx, unsigned char* __restrict__ need) {
    const int g = (int)blockIdx.x, o0 = offsets[g], n = offsets[g + 1] - o0;
    if (n < MIN_POINTS || o0 + n > cap) return;
    for (int k = (int)threadIdx.x; k < n; k += (int)blockDim.x) need[idx[o0 + k]] = 1;
}

// up to MAX_NN nearest cloud points with squared distance <= RADIUS^2, ascending (squared distance, index)
__global__ void k_knn(const float* __restrict__ pc, int P, const unsigned char* __restrict__ need, unsigned mask,
                      const int* __restrict__ start, const int* __restrict__ cell_pts, int* __restrict__ nb_cnt, int* __restrict__ nb) {
    const int i = (int)(blockIdx.x * blockDim.x + threadIdx.x);
    if (i >= P || !need[i]) return;
    const double r2 = RADIUS * RADIUS;
    const float qx = pc[(size_t)i * 3], qy = pc[(size_t)i * 3 + 1], qz = pc[(size_t)i * 3 + 2];
    const int cx = cell_coord(qx), cy = cell_coord(qy), cz = cell_coord(qz);
    double bd[MAX_NN];
    int bj[MAX_NN];
    int cnt = 0;
    unsigned seen[27];
    int nseen = 0;
    for (int dz = -1; dz <= 1; ++dz)
        for (int dy = -1; dy <= 1; ++dy)
            for (int dx = -1; dx <= 1; ++dx) {
                const unsigned h = cell_hash(cx + dx, cy + dy, cz + dz, mask);
                bool dup = false;
                for (int s = 0; s < nseen; ++s) dup = dup || seen[s] == h;
                if (dup) continue;                          // two cells hashed to one bucket: scan it once
                seen[nseen++] = h;
                for (int t = start[h]; t < start[h + 1]; ++t) {
                    const int j = cell_pts[t];
                    const double ex = (double)pc[(size_t)j * 3] - (double)qx, ey = (double)pc[(size_t)j * 3 + 1] - (double)qy,
                                 ez = (double)pc[(size_t)j * 3 + 2] - (double)qz;
                    const double d = ex * ex + ey * ey + ez * ez;
                    if (!(d <= r2)) continue;
                    if (cnt == MAX_NN && (d > bd[MAX_NN - 1] || (d == bd[MAX_NN - 1] && j > bj[MAX_NN - 1]))) continue;
                    int p = cnt < MAX_NN ? cnt++ : MAX_NN - 1;
                    while (p > 0 && (bd[p - 1] > d || (bd[p - 1] == d && bj[p - 1] > j))) { bd[p] = bd[p - 1]; bj[p] = bj[p - 1]; --p; }
                    bd[p] = d; bj[p] = j;
                }
            }
    nb_cnt[i] = cnt;
    for (int k = 0; k < cnt; ++k) nb[(size_t)i * MAX_NN + k] = bj[k];
}

// ---- 3. normals per (grasp, in-box point) -------------------------------------------------------------------------------
// Fewer than 3 neighbours, or a zero covariance, give (0, 0, 1).  Stored as fp32 (the reference keeps the normals of a
// voxel in a float32 buffer, dataset.py:173-183); a NaN component marks a point the projection drops (dataset.py:96-100).
__global__ void k_normals(const float* __restrict__ pc, const double* __restrict__ frames, const int* __restrict__ offsets, int cap,
                          const int* __restrict__ idx, const int* __restrict__ nb_cnt, const int* __restrict__ nb,
                          float* __restrict__ normals) {
    const int g = (int)blockIdx.x, o0 = offsets[g], o1 = offsets[g + 1];
    if (o1 - o0 < MIN_POINTS || o1 > cap) return;
    const double* f = frames + (size_t)g * FRAME_DOUBLES;
    for (int k = o0 + (int)threadIdx.x; k < o1; k += (int)blockDim.x) {
        const int i = idx[k], n = nb_cnt[i];
        V3 nrm{0.0, 0.0, 1.0};
        if (n >= 3) {
            double s[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};      // x, y, z, xx, xy, xz, yy, yz, zz
            for (int t = 0; t < n; ++t) {
                const V3 p = to_grasp(pc, nb[(size_t)i * MAX_NN + t], f);
                s[0] += p.x; s[1] += p.y; s[2] += p.z;
                s[3] += p.x * p.x; s[4] += p.x * p.y; s[5] += p.x * p.z; s[6] += p.y * p.y; s[7] += p.y * p.z; s[8] += p.z * p.z;
            }
            for (int t = 0; t < 9; ++t) s[t] /= (double)n;
            const double cov[6] = {s[3] - s[0] * s[0], s[4] - s[0] * s[1], s[5] - s[0] * s[2], s[6] - s[1] * s[1], s[7] - s[1] * s[2],
                                   s[8] - s[2] * s[2]};
            const V3 v = smallest_eigenvector(cov);
            if (!(v.x == 0.0 && v.y == 0.0 && v.z == 0.0)) nrm = v;
        }
        normals[(size_t)k * 3 + 0] = (float)nrm.x;
        normals[(size_t)k * 3 + 1] = (float)nrm.y;
        normals[(size_t)k * 3 + 2] = (float)nrm.z;
    }
}

// ---- 4. voxels and images per (grasp, axis order) ------------------------------------------------------------------------
// grid (G, orders), block 256.  keys: [orders][total] scratch.  Output channels of order o: chann 3 -> normals at 0..2;
// chann 12 -> occupancy at 4o, normals at 4o+1..4o+3.  Pixel (x, y) of the reference's [x][y][c] image is out[c][y][x].
constexpr int VOX_THREADS = 256;

__device__ __forceinline__ double block_reduce(double v, bool is_max, double* red) {
    const int tid = (int)threadIdx.x;
    red[tid] = v;
    __syncthreads();
    for (int s = VOX_THREADS / 2; s > 0; s >>= 1) {
        if (tid < s) red[tid] = is_max ? fmax(red[tid], red[tid + s]) : fmin(red[tid], red[tid + s]);
        __syncthreads();
    }
    const double r = red[0];
    __syncthreads();
    return r;
}

__global__ void __launch_bounds__(VOX_THREADS) k_voxelize(const float* __restrict__ pc, const double* __restrict__ frames,
                                                          const int* __restrict__ offsets, int cap, const int* __restrict__ idx,
                                                          const float* __restrict__ normals, int chann, unsigned long long* __restrict__ keys_all,
                                                          float* __restrict__ out, unsigned char* __restrict__ valid) {
    __shared__ int win[PIX];          // voxel key (x*60+y)*64+z of the voxel that wins pixel x*60+y, or -1
    __shared__ int cnt[PIX];          // its point count (<= VOXEL_CAP), 0 for an empty pixel
    __shared__ double red[VOX_THREADS];
    const int g = (int)blockIdx.x, o = (int)blockIdx.y, tid = (int)threadIdx.x;
    const int o0 = offsets[g], n = offsets[g + 1] - o0;
    const int chan0 = chann == 3 ? 0 : 4 * o, nch = chann == 3 ? 3 : 4, nrm0 = chann == 3 ? chan0 : chan0 + 1;
    float* img = out + (size_t)g * chann * PIX;
    if (o == 0 && tid == 0) valid[g] = n >= MIN_POINTS ? 1 : 0;
    for (int p = tid; p < nch * PIX; p += VOX_THREADS) img[(size_t)chan0 * PIX + p] = 0.f;
    if (n < MIN_POINTS) return;
    if (o0 + n > cap) {                                      // workspace sized for fewer in-box points: poison, not garbage
        if (o == 0 && tid == 0) valid[g] = 0;
        for (int p = tid; p < nch * PIX; p += VOX_THREADS) img[(size_t)chan0 * PIX + p] = NAN;
        return;
    }
    const double* f = frames + (size_t)g * FRAME_DOUBLES;
    // axis order of this image: [0,1,2], [1,2,0], [0,2,1] (dataset.py:104,110,113)
    const int ax = o == 1 ? 1 : 0, ay = o == 0 ? 1 : 2, az = o == 0 ? 2 : (o == 1 ? 0 : 1);
    const double res = (f[13] * 2.0) / (double)(IMG - 1);   // gripper width / (project_size - margin), dataset.py:159
    const int nord = chann == 12 ? 3 : 1;                    // keys of the orders interleaved: [point][order]
    unsigned long long* keys = keys_all + (size_t)o0 * nord + o;
    auto key = [&](int i) -> unsigned long long& { return keys[(size_t)i * nord]; };
    auto voxel = [&](int i) { return (int)(key(i) >> 32); };   // -1 for DROPPED, which matches no voxel and no pixel
    double xmin = INFINITY, xmax = -INFINITY, ymin = INFINITY, ymax = -INFINITY;
    for (int k = tid; k < n; k += VOX_THREADS) {
        const float* nv = normals + (size_t)(o0 + k) * 3;
        if (nv[0] != nv[0] || nv[1] != nv[1] || nv[2] != nv[2]) { key(k) = DROPPED; continue; }
        const V3 t = to_grasp(pc, idx[o0 + k], f);
        const double c[3] = {t.x, t.y, t.z};
        xmin = fmin(xmin, c[ax]); xmax = fmax(xmax, c[ax]); ymin = fmin(ymin, c[ay]); ymax = fmax(ymax, c[ay]);
        int v[3];
        for (int d = 0; d < 3; ++d) {                        // floor(coord / res + project_size / 2), dataset.py:162-167
            const double q = floor(c[d == 0 ? ax : (d == 1 ? ay : az)] / res + (double)(IMG / 2));
            v[d] = (int)fmin(fmax(q, 0.0), (double)(IMG - 1));   // in range for every in-box point; clamped for memory safety
        }
        key(k) = ((unsigned long long)((v[0] * IMG + v[1]) * 64 + v[2]) << 32) | (unsigned)k;
    }
    xmin = block_reduce(xmin, false, red); xmax = block_reduce(xmax, true, red);
    ymin = block_reduce(ymin, false, red); ymax = block_reduce(ymax, true, red);
    if (!(xmax - xmin > 0.0 || ymax - ymin > 0.0)) return;  // one image point (or none kept): all zeros, dataset.py:153-157
    // bitonic sort of key(0..n) ascending, virtually padded with +inf to a power of two
    int n2 = 1;
    while (n2 < n) n2 <<= 1;
    for (int size = 2; size <= n2; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int i = tid; i < n2 / 2; i += VOX_THREADS) {
                const int lo = (i / stride) * 2 * stride + i % stride;
                const int hi = stride == (size >> 1) ? (lo / size) * size + size - 1 - (lo % size) : lo + stride;
                if (hi < n) {
                    const unsigned long long a = key(lo), b = key(hi);
                    if (a > b) { key(lo) = b; key(hi) = a; }
                }
            }
            __syncthreads();
        }
    }
    for (int p = tid; p < PIX; p += VOX_THREADS) { win[p] = -1; cnt[p] = 0; }
    __syncthreads();
    // sorted by (x, y, z, input position): the last voxel of a pixel's run has the largest z and wins (numpy's last write)
    for (int i = tid; i < n; i += VOX_THREADS) {
        const int vk = voxel(i);
        if (vk >= 0 && (i + 1 == n || (voxel(i + 1) >> 6) != (vk >> 6))) win[vk >> 6] = vk;
    }
    __syncthreads();
    int cmax = 0;
    for (int i = tid; i < n; i += VOX_THREADS) {
        const int vk = voxel(i), pix = vk >> 6;
        if (vk < 0 || win[pix] != vk || (i > 0 && voxel(i - 1) == vk)) continue;   // first point of a winning voxel only
        // the first VOXEL_CAP points in input order, their fp32 normals summed in that order (dataset.py:178-186)
        float s0 = 0.f, s1 = 0.f, s2 = 0.f;
        int c = 0;
        for (int r = i; r < n && c < VOXEL_CAP && voxel(r) == vk; ++r, ++c) {
            const float* nv = normals + (size_t)(o0 + (int)(unsigned)key(r)) * 3;
            s0 += nv[0]; s1 += nv[1]; s2 += nv[2];
        }
        cnt[pix] = c;
        cmax = max(cmax, c);
        const int px = pix / IMG, py = pix % IMG, at = py * IMG + px;
        img[(size_t)(nrm0 + 0) * PIX + at] = (float)((double)s0 / (double)c);
        img[(size_t)(nrm0 + 1) * PIX + at] = (float)((double)s1 / (double)c);
        img[(size_t)(nrm0 + 2) * PIX + at] = (float)((double)s2 / (double)c);
    }
    if (chann == 3) return;
    const double occ_max = block_reduce((double)cmax, true, red);
    for (int p = tid; p < PIX; p += VOX_THREADS)
        if (cnt[p] > 0) img[(size_t)chan0 * PIX + (p % IMG) * IMG + p / IMG] = (float)((double)cnt[p] / occ_max);
}

// ---- workspace and host driver ----------------------------------------------------------------------------------------------
struct ProjWs {
    int H;
    int *bucket_cnt, *start, *cursor, *cell_pts, *nb_cnt, *nb;
    unsigned char* need;
    float* normals;
    unsigned long long* keys;
    size_t bytes;
};

inline void plan_project(void* base, int P, int total, int chann, ProjWs& w) {
    Carver c(base);
    int H = 1024;
    while (H < P) H <<= 1;
    w.H = H;
    const size_t Pn = (size_t)(P > 0 ? P : 1), Tn = (size_t)(total > 0 ? total : 1);
    w.bucket_cnt = c.take<int>(H);
    w.start = c.take<int>((size_t)H + 1);
    w.cursor = c.take<int>(H);
    w.cell_pts = c.take<int>(Pn);
    w.need = c.take<unsigned char>(Pn);
    w.nb_cnt = c.take<int>(Pn);
    w.nb = c.take<int>(Pn * MAX_NN);
    w.normals = c.take<float>(Tn * 3);
    w.keys = c.take<unsigned long long>(Tn * (chann == 12 ? 3 : 1));
    w.bytes = (c.off + 255) & ~(size_t)255;
}

// the largest in-box total a workspace of `bytes` holds for this P and chann (-1: not even an empty call fits)
inline int project_capacity(size_t bytes, int P, int chann) {
    ProjWs w;
    plan_project(nullptr, P, 0, chann, w);
    if (w.bytes > bytes) return -1;
    long long lo = 0, hi = 0x7fffffffLL / 32;
    while (lo < hi) {
        const long long mid = (lo + hi + 1) / 2;
        plan_project(nullptr, P, (int)mid, chann, w);
        if (w.bytes <= bytes) lo = mid; else hi = mid - 1;
    }
    return (int)lo;
}

// cap: the number of in-box points the workspace holds (project_capacity); grasps whose segment ends beyond it are
// written as NaN images with valid = 0
inline void project(const float* pc, int P, const double* frames, int G, const int* offsets, const int* idx, int cap, int chann,
                    float* out, unsigned char* valid, ProjWs& w, cudaStream_t s) {
    if (P > 0 && cap > 0) {
        const unsigned mask = (unsigned)w.H - 1u;
        cudaMemsetAsync(w.bucket_cnt, 0, (size_t)w.H * sizeof(int), s);
        cudaMemsetAsync(w.need, 0, (size_t)P, s);
        launch(k_grid_count, grid1d(P, 256), dim3(256), 0, s, pc, P, mask, w.bucket_cnt);
        launch(k_grid_scan, dim3(1), dim3(1024), 0, s, (const int*)w.bucket_cnt, w.H, w.start, w.cursor);
        launch(k_grid_fill, grid1d(P, 256), dim3(256), 0, s, pc, P, mask, w.cursor, w.cell_pts);
        launch(k_mark_needed, dim3(G), dim3(256), 0, s, offsets, cap, idx, w.need);
        launch(k_knn, grid1d(P, 128), dim3(128), 0, s, pc, P, (const unsigned char*)w.need, mask, (const int*)w.start,
               (const int*)w.cell_pts, w.nb_cnt, w.nb);
        launch(k_normals, dim3(G), dim3(128), 0, s, pc, frames, offsets, cap, idx, (const int*)w.nb_cnt, (const int*)w.nb, w.normals);
    }
    launch(k_voxelize, dim3(G, chann == 12 ? 3 : 1), dim3(VOX_THREADS), 0, s, pc, frames, offsets, cap, idx,
           (const float*)w.normals, chann, w.keys, out, valid);
}

}  // namespace proj
}  // namespace pgpd
