// gndt_ndt.cuh — NDT scan-to-map registration (gndt_register): the per-voxel Gaussians of the
// resident map and one derivative pass of a scan against them.
//
// prepare : one thread per voxel -> {mu, C = Sigma'^-1 (or Sigma' for D2D), usable count, cz}  (once per map)
// level   : coarse columns (warp per x slab), then coarse voxels (thread per coarse column) of the
//           level of factor k: Chan merges of the fitted records, C as above    (once per map, k)
// mean    : binary64 sum of the scan's finite points (the solver's centre)         (once per call)
// pass    : one thread per point -> score, gradient, Hessian and counts per block (once per pose)
// d2d     : the same for one thread per scan Gaussian against the map's Gaussians  (once per pose)
// finish  : one warp sums the per-block partials in block order -> 32 doubles the host reads
// No atomics: every sum has a fixed order for a fixed grid, so results repeat bit for bit.
#pragma once
#include "gndt_device.cuh"
#include "gndt_reduce.cuh"
#include "gndt_label.cuh"

namespace gndt {

constexpr int kNdtThreads = 128;
constexpr int kNdtWidth = 32;  // pass: S, g[6], H upper triangle[21], n_points, n_matched, n_pairs, 0
constexpr int kNdtMaxFactor = 32;  // levels: factors 2..32, so a slab's rows fit the lanes of one warp

struct NdtVoxel {  // 80 B
  double mu[3];
  double c[6];     // C = Sigma'^-1 (Sigma' in the D2D form): xx xy xz yy yz zz
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
  int factor;         // level: cell indices are floor-divided by it (1 = the map level)
};

// floor(c / k) for k >= 1: contiguous index -1 and 0 never share a coarse cell
__host__ __device__ __forceinline__ int floor_div(int c, int k) { return c >= 0 ? c / k : -((k - 1 - c) / k); }

// C = Sigma'^-1 of a symmetric Sigma (xx xy xz yy yz zz) with its eigenvalues raised to >= 0.01
// lambda_max; false (c untouched) when lambda_max is not positive and finite.  eig3_sym's
// eigenvectors come from cross products of rows of (A - lambda I) and lose orthogonality between
// two close eigenvalues; the basis is therefore rebuilt from the eigenvector of the most isolated
// eigenvalue, which is accurate, and the subspace orthogonal to it (whose split does not matter
// when its two eigenvalues are close).  The map level and the coarse levels both use it.
// kCov: c = Sigma' itself (the floored covariance D2D adds to the scan's), from the same basis.
template <bool kCov = false>
__device__ __forceinline__ bool ndt_inverse_cov(double s[6], double c[6]) {
  double w[3], E[3][3];
  eig3_sym(s, w, E);
  const double lmax = fmax(fmax(w[0], w[1]), w[2]);
  if (!(lmax > 0.0 && isfinite(lmax))) return false;
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
  const double la = kCov ? fmax(w[ia], floor_l) : 1.0 / fmax(w[ia], floor_l);
  const double lb = kCov ? fmax(w[ib], floor_l) : 1.0 / fmax(w[ib], floor_l);
  const double lm = kCov ? fmax(w[1], floor_l) : 1.0 / fmax(w[1], floor_l);
  const int ii[6] = {0, 0, 0, 1, 1, 2}, jj[6] = {0, 1, 2, 1, 2, 2};
#pragma unroll
  for (int k = 0; k < 6; ++k)
    c[k] = a[ii[k]] * a[jj[k]] * la + b[ii[k]] * b[jj[k]] * lb + m[ii[k]] * m[jj[k]] * lm;
  return true;
}

// Sigma from the published record (so the oracle can rebuild it from gndt_copy_voxels); c = C, or
// Sigma' when kCov.
template <bool kCov>
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
      if (ndt_inverse_cov<kCov>(s, o.c)) {
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

// pair(g) for every candidate voxel g of column `col`: |cz_v - cz| <= 1, count >= min_points
template <class F>
__device__ __forceinline__ void ndt_column(const gndt_column &col, int cz, const NdtVoxel *vox, u32 min_points, F &&pair) {
  u32 lo = col.voxel_begin, hi = col.voxel_begin + col.voxel_count;
  const u32 end = hi;
  while (lo < hi) {
    const u32 mid = (lo + hi) >> 1;
    if (vox[mid].cz < cz - 1) lo = mid + 1; else hi = mid;
  }
  for (u32 v = lo; v < end; ++v) {
    const NdtVoxel &g = vox[v];
    if (g.cz > cz + 1) break;
    if (g.count < min_points) continue;
    pair(g);
  }
}

// column(c) for the candidate columns of cell (cx, cy) that exist, in table order: row cx - 1, then
// (cx, cy - 1 .. cy + 1), then row cx + 1.  P2D and D2D passes share it.
template <class F>
__device__ __forceinline__ void ndt_columns(const gndt_column *cols, u32 n_cols, int cx, int cy, F &&column) {
  const u32 j0 = column_lower_bound(cols, 0, n_cols, cx, cy - 1);
  const u32 jm = column_lower_bound(cols, 0, j0, cx - 1, cy);
  if (jm < j0 && contiguous_index(cols[jm].sx) == cx - 1 && contiguous_index(cols[jm].sy) == cy) column(cols[jm]);
  u32 j = j0;
  for (; j < n_cols; ++j) {
    const gndt_column c = cols[j];
    if (contiguous_index(c.sx) != cx || contiguous_index(c.sy) > cy + 1) break;
    column(c);
  }
  const u32 jp = column_lower_bound(cols, j, n_cols, cx + 1, cy);
  if (jp < n_cols && contiguous_index(cols[jp].sx) == cx + 1 && contiguous_index(cols[jp].sy) == cy) column(cols[jp]);
}

// one (point, voxel) pair of P2D: x the moved point, y = x - c
__device__ __forceinline__ void ndt_p2d_pair(const NdtVoxel &g, const double x[3], const double y[3], const NdtPose &P, NdtAcc &A) {
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

// One derivative pass: every finite point at pose P against the 5 candidate columns of its level.
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
    if (!point_indices<false>(__double2float_rn(x[0]), __double2float_rn(x[1]), __double2float_rn(x[2]), P.origin, P.grid_len, P.z_len,
                              0.f, 0.f, cx, cy, cz))
      continue;
    if (P.factor > 1) { cx = floor_div(cx, P.factor); cy = floor_div(cy, P.factor); cz = floor_div(cz, P.factor); }
    const double y[3] = {x[0] - P.c[0], x[1] - P.c[1], x[2] - P.c[2]};
    const u32 before = A.pairs;
    ndt_columns(cols, n_cols, cx, cy, [&](const gndt_column &c) {
      ndt_column(c, cz, vox, P.min_points, [&](const NdtVoxel &g) { ndt_p2d_pair(g, x, y, P, A); });
    });
    n_matched += A.pairs != before;
  }
  double v[kNdtWidth];
#pragma unroll
  for (int k = 0; k < 28; ++k) v[k] = A.s[k];
  v[28] = (double)n_points; v[29] = (double)n_matched; v[30] = (double)A.pairs; v[31] = 0.0;
  block_partials<kNdtWidth>(v, partial);
}

// One (scan Gaussian, map Gaussian) pair of D2D (Stoyanov et al. 2012): x = R mu_i + t, y = x - c,
// S = R Sigma'_i R^T, g.c = Sigma'_j.  With B = S + Sigma'_j, A = B^-1, m = x - mu_j, a = A m:
//   q_k  = 2 m_k.a - a.B_k a,   q_kl = 2 m_kl.a + 2 z_k.A z_l - a.B_kl a,   z_k = m_k - B_k a,
// where the rotation columns are m_l = e_l x y, B_l = K_l S - S K_l, B_kl = E_kl S + S E_kl +
// K_k S K_l^T + K_l S K_k^T (K_l = [e_l]x, E_kl = (K_k K_l + K_l K_k) / 2).  With s = S a and
// n_l = e_l x a these are a.B_l a = 2 (s x a)_l, B_l a = e_l x s - S n_l and a.B_kl a =
// s_l a_k + s_k a_l - 2 delta_kl a.s + 2 n_k.S n_l; every term is P2D's when S = 0.
__device__ __forceinline__ void ndt_d2d_pair(const NdtVoxel &g, const double x[3], const double y[3], const double S[6], const NdtPose &P,
                                             NdtAcc &A) {
  const double m[3] = {x[0] - g.mu[0], x[1] - g.mu[1], x[2] - g.mu[2]};
  const double b0 = S[0] + g.c[0], b1 = S[1] + g.c[1], b2 = S[2] + g.c[2], b3 = S[3] + g.c[3], b4 = S[4] + g.c[4], b5 = S[5] + g.c[5];
  // A = adj(B) / det(B); B is SPD since both covariances are floored
  const double c0 = b3 * b5 - b4 * b4, c1 = b2 * b4 - b1 * b5, c2 = b1 * b4 - b2 * b3;
  const double id = 1.0 / (b0 * c0 + b1 * c1 + b2 * c2);
  const double Ai[6] = {c0 * id, c1 * id, c2 * id, (b0 * b5 - b2 * b2) * id, (b1 * b2 - b0 * b4) * id, (b0 * b3 - b1 * b1) * id};
  const double a[3] = {Ai[0] * m[0] + Ai[1] * m[1] + Ai[2] * m[2], Ai[1] * m[0] + Ai[3] * m[1] + Ai[4] * m[2],
                       Ai[2] * m[0] + Ai[4] * m[1] + Ai[5] * m[2]};
  const double q = m[0] * a[0] + m[1] * a[1] + m[2] * a[2];
  const double e = exp(-0.5 * P.d2 * q);
  const double w = 0.5 * P.d1 * P.d2 * e;
  const double s[3] = {S[0] * a[0] + S[1] * a[1] + S[2] * a[2], S[1] * a[0] + S[3] * a[1] + S[4] * a[2], S[2] * a[0] + S[4] * a[1] + S[5] * a[2]};
  const double u[3] = {y[0] - s[0], y[1] - s[1], y[2] - s[2]};
  // q_k: 2 a for translations, 2 (y - s) x a for rotations
  const double qa[6] = {2.0 * a[0], 2.0 * a[1], 2.0 * a[2], 2.0 * (u[1] * a[2] - u[2] * a[1]), 2.0 * (u[2] * a[0] - u[0] * a[2]),
                        2.0 * (u[0] * a[1] - u[1] * a[0])};
  const double n[3][3] = {{0.0, -a[2], a[1]}, {a[2], 0.0, -a[0]}, {-a[1], a[0], 0.0}};  // n[l] = e_l x a
  double Sn[3][3], z[3][3], Az[3][3];
#pragma unroll
  for (int l = 0; l < 3; ++l) {
    Sn[l][0] = S[0] * n[l][0] + S[1] * n[l][1] + S[2] * n[l][2];
    Sn[l][1] = S[1] * n[l][0] + S[3] * n[l][1] + S[4] * n[l][2];
    Sn[l][2] = S[2] * n[l][0] + S[4] * n[l][1] + S[5] * n[l][2];
  }
  // z_l = e_l x (y - s) + S n_l
  z[0][0] = Sn[0][0]; z[0][1] = Sn[0][1] - u[2]; z[0][2] = Sn[0][2] + u[1];
  z[1][0] = Sn[1][0] + u[2]; z[1][1] = Sn[1][1]; z[1][2] = Sn[1][2] - u[0];
  z[2][0] = Sn[2][0] - u[1]; z[2][1] = Sn[2][1] + u[0]; z[2][2] = Sn[2][2];
#pragma unroll
  for (int l = 0; l < 3; ++l) {
    Az[l][0] = Ai[0] * z[l][0] + Ai[1] * z[l][1] + Ai[2] * z[l][2];
    Az[l][1] = Ai[1] * z[l][0] + Ai[3] * z[l][1] + Ai[4] * z[l][2];
    Az[l][2] = Ai[2] * z[l][0] + Ai[4] * z[l][1] + Ai[5] * z[l][2];
  }
  const double ay = a[0] * y[0] + a[1] * y[1] + a[2] * y[2], as = a[0] * s[0] + a[1] * s[1] + a[2] * s[2];
  A.s[0] += -P.d1 * e;
#pragma unroll
  for (int k = 0; k < 6; ++k) A.s[1 + k] += w * qa[k];
  int idx = 7;
#pragma unroll
  for (int k = 0; k < 6; ++k) {
#pragma unroll
    for (int l = k; l < 6; ++l) {
      double qkl;
      if (l < 3) {
        qkl = 2.0 * Ai[k * 3 + l - (k * (k + 1)) / 2];
      } else if (k < 3) {
        qkl = 2.0 * Az[l - 3][k];
      } else {
        const int kk = k - 3, ll = l - 3;
        const double zaz = z[kk][0] * Az[ll][0] + z[kk][1] * Az[ll][1] + z[kk][2] * Az[ll][2];
        const double mkl = 0.5 * (a[ll] * y[kk] + a[kk] * y[ll]) - (kk == ll ? ay : 0.0);
        const double bkl = s[ll] * a[kk] + s[kk] * a[ll] - (kk == ll ? 2.0 * as : 0.0) +
                           2.0 * (n[kk][0] * Sn[ll][0] + n[kk][1] * Sn[ll][1] + n[kk][2] * Sn[ll][2]);
        qkl = 2.0 * mkl + 2.0 * zaz - bkl;
      }
      A.s[idx++] += w * (qkl - 0.5 * P.d2 * qa[k] * qa[l]);
    }
  }
  A.pairs += 1;
}

// One D2D pass: every usable scan Gaussian (svox, c = Sigma'_i) at pose P against the 5 candidate
// columns of its level (vox, c = Sigma'_j).  Same grid, partials and counts as ndt_pass_kernel, with
// n_points = usable scan Gaussians.
__global__ void __launch_bounds__(kNdtThreads) ndt_d2d_pass_kernel(const NdtVoxel *svox, u32 n_svox, const NdtVoxel *vox,
                                                                   const gndt_column *cols, u32 n_cols, NdtPose P, double *partial) {
  NdtAcc A;
#pragma unroll
  for (int k = 0; k < 28; ++k) A.s[k] = 0.0;
  A.pairs = 0;
  u32 n_points = 0, n_matched = 0;
  for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n_svox; i += gridDim.x * blockDim.x) {
    const NdtVoxel sg = svox[i];
    if (sg.count < P.min_points) continue;  // count 0: no usable Gaussian
    ++n_points;
    double x[3];
#pragma unroll
    for (int r = 0; r < 3; ++r)
      x[r] = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(P.r[3 * r], sg.mu[0]), __dmul_rn(P.r[3 * r + 1], sg.mu[1])), __dmul_rn(P.r[3 * r + 2], sg.mu[2])),
                       P.t[r]);
    int cx, cy, cz;
    if (!point_indices<false>(__double2float_rn(x[0]), __double2float_rn(x[1]), __double2float_rn(x[2]), P.origin, P.grid_len, P.z_len,
                              0.f, 0.f, cx, cy, cz))
      continue;
    if (P.factor > 1) { cx = floor_div(cx, P.factor); cy = floor_div(cy, P.factor); cz = floor_div(cz, P.factor); }
    const double y[3] = {x[0] - P.c[0], x[1] - P.c[1], x[2] - P.c[2]};
    // S = R Sigma'_i R^T
    const double *Si = sg.c;
    double RS[3][3], S[6];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      RS[r][0] = P.r[3 * r] * Si[0] + P.r[3 * r + 1] * Si[1] + P.r[3 * r + 2] * Si[2];
      RS[r][1] = P.r[3 * r] * Si[1] + P.r[3 * r + 1] * Si[3] + P.r[3 * r + 2] * Si[4];
      RS[r][2] = P.r[3 * r] * Si[2] + P.r[3 * r + 1] * Si[4] + P.r[3 * r + 2] * Si[5];
    }
    const int ii[6] = {0, 0, 0, 1, 1, 2}, jj[6] = {0, 1, 2, 1, 2, 2};
#pragma unroll
    for (int k = 0; k < 6; ++k)
      S[k] = RS[ii[k]][0] * P.r[3 * jj[k]] + RS[ii[k]][1] * P.r[3 * jj[k] + 1] + RS[ii[k]][2] * P.r[3 * jj[k] + 2];
    const u32 before = A.pairs;
    ndt_columns(cols, n_cols, cx, cy, [&](const gndt_column &c) {
      ndt_column(c, cz, vox, P.min_points, [&](const NdtVoxel &g) { ndt_d2d_pair(g, x, y, S, P, A); });
    });
    n_matched += A.pairs != before;
  }
  double v[kNdtWidth];
#pragma unroll
  for (int k = 0; k < 28; ++k) v[k] = A.s[k];
  v[28] = (double)n_points; v[29] = (double)n_matched; v[30] = (double)A.pairs; v[31] = 0.0;
  block_partials<kNdtWidth>(v, partial);
}

// ---- levels: the Gaussians of cells of k x k x k map cells --------------------------------
// Coarse column tables are gndt_column records whose sx, sy, voxel_begin and voxel_count the pass
// reads; slope_begin / slope_count hold the range of their map columns in `members` instead.

// Level columns, one warp per x slab [kX, kX + k) of the map (X = X0 + warp), lane r < k on map row
// kX + r.  The slab and its rows are ranges of the (cx, cy)-sorted column table; each row is a sorted
// run of cy, so the warp emits its coarse columns in Y order by taking the smallest head Y of the
// rows at a time.  Count pass (EMIT = false): slab_count[warp].  Emit pass: the coarse column at
// slab_begin[warp] + j and its map columns, row by row, at the slab's own range of `members`.
template <bool EMIT>
__global__ void __launch_bounds__(256) ndt_level_columns_kernel(const gndt_column *cols, u32 n_cols, int k, int X0, u32 n_slabs,
                                                                u32 *slab_count, const u32 *slab_begin, gndt_column *ccols,
                                                                u32 *members) {
  const u32 warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= n_slabs) return;  // whole warps: blockDim is a multiple of 32
  const int x0 = (X0 + (int)warp) * k;
  const u32 lo = column_lower_bound(cols, 0, n_cols, x0, INT_MIN), hi = column_lower_bound(cols, lo, n_cols, x0 + k, INT_MIN);
  u32 r_lo = hi, r_hi = hi;
  if (lane < k) {
    r_lo = column_lower_bound(cols, lo, hi, x0 + lane, INT_MIN);
    r_hi = column_lower_bound(cols, r_lo, hi, x0 + lane + 1, INT_MIN);
  }
  u32 out = EMIT ? slab_begin[warp] : 0u, mpos = lo;
  for (;;) {
    const int y = r_lo < r_hi ? floor_div(contiguous_index(cols[r_lo].sy), k) : INT_MAX;
    const int Y = __reduce_min_sync(0xffffffffu, y);
    if (Y == INT_MAX) break;
    const u32 e = y == Y ? column_lower_bound(cols, r_lo, r_hi, x0 + lane, (Y + 1) * k) : r_lo;
    if (EMIT) {
      const u32 cnt = e - r_lo;
      u32 inc = cnt;  // inclusive scan over the lanes: rows in order
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const u32 t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
      }
      const u32 total = __shfl_sync(0xffffffffu, inc, 31);
      for (u32 j = r_lo; j < e; ++j) members[mpos + inc - cnt + (j - r_lo)] = j;
      if (lane == 0) {
        gndt_column c = {};
        c.sx = signed_index(X0 + (int)warp);
        c.sy = signed_index(Y);
        c.slope_begin = mpos;
        c.slope_count = total;
        ccols[out] = c;
      }
      mpos += total;
    }
    ++out;
    r_lo = e;
  }
  if (!EMIT && lane == 0) slab_count[warp] = out;
}

// first voxel of [lo, hi) (one column, sorted by cz) with cz >= z
__device__ __forceinline__ u32 voxel_lower_bound(const gndt_voxel *table, u32 lo, u32 hi, int z) {
  while (lo < hi) {
    const u32 mid = (lo + hi) >> 1;
    if (contiguous_index(table[mid].sz) < z) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// Level voxels, one thread per coarse column: its coarse cells bottom to top.  A cell's Gaussian is
// the binary64 Chan merge of its GNDT_F_FITTED records in ascending table index (map columns in
// table order, each bottom to top), scatter un-normalised (* n_i when normalize_cov); Sigma =
// S / (n - 1) and C as at the map level, usable when n >= 3.  Count pass: vcount[c].  Emit pass:
// the voxels at vbegin[c] and the column's voxel_begin / voxel_count; c = Sigma' when kCov.
template <bool EMIT, bool kCov = false>
__global__ void __launch_bounds__(256) ndt_level_voxels_kernel(const gndt_voxel *table, const gndt_column *cols, const u32 *members,
                                                               int k, int normalize_cov, gndt_column *ccols, u32 n_ccols,
                                                               u32 *vcount, const u32 *vbegin, NdtVoxel *out) {
  for (u32 c = blockIdx.x * blockDim.x + threadIdx.x; c < n_ccols; c += gridDim.x * blockDim.x) {
    const u32 mb = ccols[c].slope_begin, me = mb + ccols[c].slope_count;
    int Z = INT_MAX;
    for (u32 m = mb; m < me; ++m) Z = min(Z, floor_div(contiguous_index(table[cols[members[m]].voxel_begin].sz), k));
    const u32 o0 = EMIT ? vbegin[c] : 0u;
    u32 nv = 0;
    while (Z != INT_MAX) {
      int next = INT_MAX;
      double n = 0.0, mu[3] = {0.0, 0.0, 0.0}, S[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
      for (u32 m = mb; m < me; ++m) {
        const gndt_column mc = cols[members[m]];
        const u32 end = mc.voxel_begin + mc.voxel_count;
        for (u32 v = voxel_lower_bound(table, mc.voxel_begin, end, Z * k); v < end; ++v) {
          const gndt_voxel &r = table[v];
          const int cz = contiguous_index(r.sz);
          if (cz >= (Z + 1) * k) { next = min(next, floor_div(cz, k)); break; }
          if (!EMIT || !(r.flags & GNDT_F_FITTED)) continue;
          const double nb = (double)r.count, nn = n + nb, f = nb / nn, w = n * nb / nn;
          const double d[3] = {(double)r.mean[0] - mu[0], (double)r.mean[1] - mu[1], (double)r.mean[2] - mu[2]};
          const int ii[6] = {0, 0, 0, 1, 1, 2}, jj[6] = {0, 1, 2, 1, 2, 2};
#pragma unroll
          for (int j = 0; j < 6; ++j) S[j] += (normalize_cov ? (double)r.scatter[j] * nb : (double)r.scatter[j]) + d[ii[j]] * d[jj[j]] * w;
#pragma unroll
          for (int i = 0; i < 3; ++i) mu[i] += d[i] * f;
          n = nn;
        }
      }
      if (EMIT) {
        NdtVoxel o = {};
        o.cz = Z;
        if (n >= 3.0) {
          double s[6];
#pragma unroll
          for (int j = 0; j < 6; ++j) s[j] = S[j] / (n - 1.0);
          if (ndt_inverse_cov<kCov>(s, o.c)) {
            o.mu[0] = mu[0]; o.mu[1] = mu[1]; o.mu[2] = mu[2];
            o.count = (u32)n;
          }
        }
        out[o0 + nv] = o;
      }
      ++nv;
      Z = next;
    }
    if (EMIT) { ccols[c].voxel_begin = o0; ccols[c].voxel_count = nv; } else vcount[c] = nv;
  }
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
