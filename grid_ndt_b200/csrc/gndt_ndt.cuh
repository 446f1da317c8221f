// gndt_ndt.cuh — NDT scan-to-map registration (gndt_register): the per-voxel Gaussians of the
// resident map and one derivative pass of a scan against them.
//
// prepare : one thread per voxel -> {mu, C = Sigma'^-1, usable count, cz}          (once per map)
// mean    : binary64 sum of the scan's finite points (the solver's centre)         (once per call)
// pass    : one thread per point -> score, gradient, Hessian and counts per block (once per pose)
// finish  : one warp sums the per-block partials in block order -> 32 doubles the host reads
// No atomics: every sum has a fixed order for a fixed grid, so results repeat bit for bit.
#pragma once
#include "gndt_device.cuh"
#include "gndt_reduce.cuh"
#include "gndt_label.cuh"

namespace gndt {

constexpr int kNdtThreads = 128;
constexpr int kNdtWidth = 32;  // pass: S, g[6], H upper triangle[21], n_points, n_matched, n_pairs, 0

struct NdtVoxel {  // 80 B
  double mu[3];
  double c[6];     // C = Sigma'^-1: xx xy xz yy yz zz
  u32 count;       // points of the voxel; 0 when it has no usable Gaussian
  int cz;          // contiguous z index
};

struct NdtPose {
  double r[9], t[3];  // x' = R p + t, row-major R
  double c[3];        // centre of the rotation increment
  double d1, d2;      // Magnusson's score constants
  float origin[3];
  float grid_len, z_len;
  u32 min_points;
};

// Sigma from the published record (so the oracle can rebuild it from gndt_copy_voxels), eigenvalues
// raised to >= 0.01 lambda_max, C = V diag(1/lambda') V^T.  eig3_sym's eigenvectors come from cross
// products of rows of (A - lambda I) and lose orthogonality between two close eigenvalues; the basis
// is therefore rebuilt from the eigenvector of the most isolated eigenvalue, which is accurate, and
// the subspace orthogonal to it (whose split does not matter when its two eigenvalues are close).
__global__ void __launch_bounds__(256) ndt_prepare_kernel(const Ctl *ctl, const gndt_voxel *table, NdtVoxel *out, int normalize_cov) {
  const u32 V = ctl->n_voxels;
  for (u32 v = blockIdx.x * blockDim.x + threadIdx.x; v < V; v += gridDim.x * blockDim.x) {
    const gndt_voxel r = table[v];
    NdtVoxel o = {};
    o.cz = contiguous_index(r.sz);
    if ((r.flags & GNDT_F_FITTED) && r.count >= 3) {
      const double n = (double)r.count, nm1 = n - 1.0;
      double s[6];
#pragma unroll
      for (int k = 0; k < 6; ++k)
        s[k] = normalize_cov ? __ddiv_rn(__dmul_rn((double)r.scatter[k], n), nm1) : __ddiv_rn((double)r.scatter[k], nm1);
      double w[3], E[3][3];
      eig3_sym(s, w, E);
      const double lmax = fmax(fmax(w[0], w[1]), w[2]);
      if (lmax > 0.0 && isfinite(lmax)) {
        // a = eigenvector of the isolated end of the spectrum, b = the other end made orthogonal, m = a x b
        const int ia = (w[1] - w[0] >= w[2] - w[1]) ? 0 : 2, ib = 2 - ia;
        double a[3] = {E[0][ia], E[1][ia], E[2][ia]}, b[3] = {E[0][ib], E[1][ib], E[2][ib]};
        const double an = rsqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]);
        a[0] *= an; a[1] *= an; a[2] *= an;
        const double ab = a[0] * b[0] + a[1] * b[1] + a[2] * b[2];
        b[0] -= ab * a[0]; b[1] -= ab * a[1]; b[2] -= ab * a[2];
        double bn = b[0] * b[0] + b[1] * b[1] + b[2] * b[2];
        if (!(bn > 1e-20)) {  // no usable second vector: any unit vector orthogonal to a
          const int k = (fabs(a[0]) <= fabs(a[1]) && fabs(a[0]) <= fabs(a[2])) ? 0 : (fabs(a[1]) <= fabs(a[2]) ? 1 : 2);
          double e[3] = {0.0, 0.0, 0.0};
          e[k] = 1.0;
          b[0] = e[0] - a[k] * a[0]; b[1] = e[1] - a[k] * a[1]; b[2] = e[2] - a[k] * a[2];
          bn = b[0] * b[0] + b[1] * b[1] + b[2] * b[2];
        }
        const double bi = rsqrt(bn);
        b[0] *= bi; b[1] *= bi; b[2] *= bi;
        const double m[3] = {a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]};
        const double floor_l = 0.01 * lmax;
        const double la = 1.0 / fmax(w[ia], floor_l), lb = 1.0 / fmax(w[ib], floor_l), lm = 1.0 / fmax(w[1], floor_l);
        const int ii[6] = {0, 0, 0, 1, 1, 2}, jj[6] = {0, 1, 2, 1, 2, 2};
#pragma unroll
        for (int k = 0; k < 6; ++k)
          o.c[k] = a[ii[k]] * a[jj[k]] * la + b[ii[k]] * b[jj[k]] * lb + m[ii[k]] * m[jj[k]] * lm;
        o.mu[0] = (double)r.mean[0]; o.mu[1] = (double)r.mean[1]; o.mu[2] = (double)r.mean[2];
        o.count = r.count;
      }
    }
    out[v] = o;
  }
}

// Sums of W values per thread -> one row of W doubles per block (warp_sum, then warps in order).
template <int W>
__device__ __forceinline__ void block_partials(double (&v)[W], double *partial) {
  __shared__ double s[kNdtThreads / 32][W];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < W; ++k) {
    const double t = warp_sum(v[k]);
    if (lane == 0) s[warp][k] = t;
  }
  __syncthreads();
  if (threadIdx.x < W) {
    double t = 0.0;
#pragma unroll
    for (int w = 0; w < kNdtThreads / 32; ++w) t += s[w][threadIdx.x];
    partial[(size_t)blockIdx.x * W + threadIdx.x] = t;
  }
}

__device__ __forceinline__ bool finite3(float a, float b, float c) { return isfinite(a) && isfinite(b) && isfinite(c); }

// sum of the finite points (binary64) and their number
__global__ void __launch_bounds__(kNdtThreads) ndt_mean_kernel(const float *in, size_t stride_f, size_t n, double *partial) {
  double v[4] = {0.0, 0.0, 0.0, 0.0};
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const float *q = in + i * stride_f;
    const float p0 = q[0], p1 = q[1], p2 = q[2];
    if (!finite3(p0, p1, p2)) continue;
    v[0] += (double)p0; v[1] += (double)p1; v[2] += (double)p2; v[3] += 1.0;
  }
  block_partials<4>(v, partial);
}

// first column of the (cx, cy)-sorted column table in [lo, hi) that is not below (cx, cy)
__device__ __forceinline__ u32 column_lower_bound(const gndt_column *cols, u32 lo, u32 hi, int cx, int cy) {
  while (lo < hi) {
    const u32 mid = (lo + hi) >> 1;
    const int2 k = *reinterpret_cast<const int2 *>(&cols[mid]);
    const int mx = contiguous_index(k.x), my = contiguous_index(k.y);
    if (mx < cx || (mx == cx && my < cy)) lo = mid + 1; else hi = mid;
  }
  return lo;
}

struct NdtAcc {
  double s[28];  // S, g[6], H upper triangle row by row
  u32 pairs;
};

// every candidate voxel of column `col` with |cz_v - cz| <= 1
__device__ __forceinline__ void ndt_column(const gndt_column &col, int cz, const NdtVoxel *vox, const double x[3],
                                           const double y[3], const NdtPose &P, NdtAcc &A) {
  u32 lo = col.voxel_begin, hi = col.voxel_begin + col.voxel_count;
  const u32 end = hi;
  while (lo < hi) {
    const u32 mid = (lo + hi) >> 1;
    if (vox[mid].cz < cz - 1) lo = mid + 1; else hi = mid;
  }
  for (u32 v = lo; v < end; ++v) {
    const NdtVoxel &g = vox[v];
    if (g.cz > cz + 1) break;
    if (g.count < P.min_points) continue;
    const double d[3] = {x[0] - g.mu[0], x[1] - g.mu[1], x[2] - g.mu[2]};
    const double *C = g.c;
    const double a[3] = {C[0] * d[0] + C[1] * d[1] + C[2] * d[2], C[1] * d[0] + C[3] * d[1] + C[4] * d[2],
                         C[2] * d[0] + C[4] * d[1] + C[5] * d[2]};  // C d
    const double q = d[0] * a[0] + d[1] * a[1] + d[2] * a[2];
    const double e = exp(-0.5 * P.d2 * q);
    const double w = P.d1 * P.d2 * e;
    // d^T C J_k: J = [I | -[y]x], so the rotation part is y x (C d)
    const double ga[6] = {a[0], a[1], a[2], y[1] * a[2] - y[2] * a[1], y[2] * a[0] - y[0] * a[2], y[0] * a[1] - y[1] * a[0]};
    // C M_l with M_l = e_l x y, the rotation columns of J
    const double M[3][3] = {{0.0, -y[2], y[1]}, {y[2], 0.0, -y[0]}, {-y[1], y[0], 0.0}};  // M[l] = e_l x y
    double CM[3][3];
#pragma unroll
    for (int l = 0; l < 3; ++l) {
      CM[l][0] = C[0] * M[l][0] + C[1] * M[l][1] + C[2] * M[l][2];
      CM[l][1] = C[1] * M[l][0] + C[3] * M[l][1] + C[4] * M[l][2];
      CM[l][2] = C[2] * M[l][0] + C[4] * M[l][1] + C[5] * M[l][2];
    }
    const double ay = a[0] * y[0] + a[1] * y[1] + a[2] * y[2];
    A.s[0] += -P.d1 * e;
#pragma unroll
    for (int k = 0; k < 6; ++k) A.s[1 + k] += w * ga[k];
    int idx = 7;
#pragma unroll
    for (int k = 0; k < 6; ++k) {
#pragma unroll
      for (int l = k; l < 6; ++l) {
        double jcj, dch = 0.0;  // J_k^T C J_l and d^T C h_kl
        if (l < 3) {
          const int ci = k * 3 + l - (k * (k + 1)) / 2;  // (k, l), k <= l < 3, in xx xy xz yy yz zz
          jcj = C[ci];
        } else if (k < 3) {
          jcj = CM[l - 3][k];
        } else {
          const int kk = k - 3, ll = l - 3;
          jcj = M[kk][0] * CM[ll][0] + M[kk][1] * CM[ll][1] + M[kk][2] * CM[ll][2];
          // h_kl = (e_k x (e_l x y) + e_l x (e_k x y)) / 2 = (e_l y_k + e_k y_l) / 2 - delta_kl y
          dch = 0.5 * (a[ll] * y[kk] + a[kk] * y[ll]) - (kk == ll ? ay : 0.0);
        }
        A.s[idx++] += w * (-P.d2 * ga[k] * ga[l] + jcj + dch);
      }
    }
    A.pairs += 1;
  }
}

// One derivative pass: every finite point at pose P against the 5 candidate columns.
__global__ void __launch_bounds__(kNdtThreads) ndt_pass_kernel(const float *in, size_t stride_f, size_t n, const NdtVoxel *vox,
                                                               const gndt_column *cols, u32 n_cols, NdtPose P, double *partial) {
  NdtAcc A;
#pragma unroll
  for (int k = 0; k < 28; ++k) A.s[k] = 0.0;
  A.pairs = 0;
  u32 n_points = 0, n_matched = 0;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const float *q = in + i * stride_f;
    const double p[3] = {(double)q[0], (double)q[1], (double)q[2]};
    if (!finite3(q[0], q[1], q[2])) continue;
    ++n_points;
    double x[3];
#pragma unroll
    for (int r = 0; r < 3; ++r)
      x[r] = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(P.r[3 * r], p[0]), __dmul_rn(P.r[3 * r + 1], p[1])), __dmul_rn(P.r[3 * r + 2], p[2])), P.t[r]);
    int cx, cy, cz;
    if (!point_indices(__double2float_rn(x[0]), __double2float_rn(x[1]), __double2float_rn(x[2]), P.origin, P.grid_len, P.z_len, cx, cy, cz))
      continue;
    const double y[3] = {x[0] - P.c[0], x[1] - P.c[1], x[2] - P.c[2]};
    const u32 before = A.pairs;
    // table order: row cx - 1, then (cx, cy - 1 .. cy + 1), then row cx + 1
    const u32 j0 = column_lower_bound(cols, 0, n_cols, cx, cy - 1);
    const u32 jm = column_lower_bound(cols, 0, j0, cx - 1, cy);
    if (jm < j0 && contiguous_index(cols[jm].sx) == cx - 1 && contiguous_index(cols[jm].sy) == cy) ndt_column(cols[jm], cz, vox, x, y, P, A);
    u32 j = j0;
    for (; j < n_cols; ++j) {
      const gndt_column c = cols[j];
      if (contiguous_index(c.sx) != cx || contiguous_index(c.sy) > cy + 1) break;
      ndt_column(c, cz, vox, x, y, P, A);
    }
    const u32 jp = column_lower_bound(cols, j, n_cols, cx + 1, cy);
    if (jp < n_cols && contiguous_index(cols[jp].sx) == cx + 1 && contiguous_index(cols[jp].sy) == cy) ndt_column(cols[jp], cz, vox, x, y, P, A);
    n_matched += A.pairs != before;
  }
  double v[kNdtWidth];
#pragma unroll
  for (int k = 0; k < 28; ++k) v[k] = A.s[k];
  v[28] = (double)n_points; v[29] = (double)n_matched; v[30] = (double)A.pairs; v[31] = 0.0;
  block_partials<kNdtWidth>(v, partial);
}

// one warp: out[k] = sum over blocks, in block order, of partial[b][k]
__global__ void ndt_finish_kernel(const double *partial, int n_blocks, int width, double *out) {
  const int k = threadIdx.x;
  if (k >= width) return;
  double t = 0.0;
  for (int b = 0; b < n_blocks; ++b) t += partial[(size_t)b * width + k];
  out[k] = t;
}

}  // namespace gndt
