// K7 — batched PnP on the GPU (SURVEY.md section 8f-2, the step right after the voting path).
//
// Stands in for the reference's host-side pnp()
// (/root/reference/casapose/pose_estimation/ransac_voting.py:13-57: cv2.solvePnPRansac(EPNP) as the initial
// guess, then cv2.solvePnP(ITERATIVE) on ALL points, flip if t_z < 0, zeros on failure) and its callers
// map_offsets / map_pnp (:487-514).  OpenCV's RANSAC draws random minimal sets, so it cannot be replayed
// bit for bit; what is reproduced is its structure — a robust initial pose from point subsets, then the
// Levenberg-Marquardt minimum of the reprojection error over all points, which is what the reference returns:
//   * candidates: the full point set, every leave-one-out and every leave-two-out subset (46 for 9 points);
//     each is solved by a normalised DLT (reduced to a 4x4 symmetric eigen-problem, or 3x3 for coplanar points),
//     projected on SO(3) by a polar iteration and polished by 5 LM steps; the candidate with the most points inside 12 px (cv2's
//     reprojectionError), then the smallest inlier cost, wins;
//   * final: LM over all points from the winner, float64 throughout.
// One warp per object, lanes = candidates.  oracle/pnp_np.py is the numpy restatement of this algorithm;
// tests compare both with the reference's cv2 sequence (identical ADD / ADD-S verdicts on the synthetic set).
#pragma once
#include "common.cuh"

namespace casa {

struct PnpParams {
  int n, vn;
  float reproj_px;  // 12: cv2.solvePnPRansac reprojectionError (:35)
};

__device__ __forceinline__ void mat3_inv_t(const double* R, double* out) {  // out = inverse(R)^T
  const double c00 = R[4] * R[8] - R[5] * R[7], c01 = R[5] * R[6] - R[3] * R[8], c02 = R[3] * R[7] - R[4] * R[6];
  const double c10 = R[2] * R[7] - R[1] * R[8], c11 = R[0] * R[8] - R[2] * R[6], c12 = R[1] * R[6] - R[0] * R[7];
  const double c20 = R[1] * R[5] - R[2] * R[4], c21 = R[2] * R[3] - R[0] * R[5], c22 = R[0] * R[4] - R[1] * R[3];
  const double det = R[0] * c00 + R[1] * c01 + R[2] * c02, id = 1.0 / det;
  out[0] = c00 * id; out[1] = c01 * id; out[2] = c02 * id;
  out[3] = c10 * id; out[4] = c11 * id; out[5] = c12 * id;
  out[6] = c20 * id; out[7] = c21 * id; out[8] = c22 * id;
}

__device__ __forceinline__ double mat3_det(const double* R) {
  return R[0] * (R[4] * R[8] - R[5] * R[7]) - R[1] * (R[3] * R[8] - R[5] * R[6]) + R[2] * (R[3] * R[7] - R[4] * R[6]);
}

// exp([w]x) (Rodrigues)
__device__ __forceinline__ void so3_exp(const double* w, double* E) {
  const double th = sqrt(w[0] * w[0] + w[1] * w[1] + w[2] * w[2]);
  double a, b;  // E = I + a K + b K^2 with K = [w]x
  if (th < 1e-12) {
    a = 1.0;
    b = 0.5;
  } else {
    a = sin(th) / th;
    b = (1.0 - cos(th)) / (th * th);
  }
  const double x = w[0], y = w[1], z = w[2];
  E[0] = 1.0 - b * (y * y + z * z); E[1] = -a * z + b * x * y;       E[2] = a * y + b * x * z;
  E[3] = a * z + b * x * y;         E[4] = 1.0 - b * (x * x + z * z); E[5] = -a * x + b * y * z;
  E[6] = -a * y + b * x * z;        E[7] = a * x + b * y * z;         E[8] = 1.0 - b * (x * x + y * y);
}

// smallest-eigenvalue eigenvector of the symmetric DxD matrix A (destroyed; D = 4 or 3 in the leading block), cyclic Jacobi
template <int D>
__device__ __forceinline__ void jacobi_smallest(double (&A)[4][4], double (&vec)[4]) {
  double V[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) V[i][j] = i == j ? 1.0 : 0.0;
  for (int sweep = 0; sweep < 30; ++sweep) {
    double off = 0.0, diag = 0.0;
#pragma unroll
    for (int i = 0; i < D; ++i) {
      diag += A[i][i] * A[i][i];
#pragma unroll
      for (int j = i + 1; j < D; ++j) off += A[i][j] * A[i][j];
    }
    if (off <= 1e-30 * diag || off == 0.0) break;
#pragma unroll
    for (int p = 0; p < D - 1; ++p)
#pragma unroll
      for (int q = p + 1; q < D; ++q) {
        const double apq = A[p][q];
        if (fabs(apq) < 1e-300) continue;
        const double theta = (A[q][q] - A[p][p]) / (2.0 * apq);
        const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
        const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
#pragma unroll
        for (int k = 0; k < D; ++k) {  // columns p, q
          const double akp = A[k][p], akq = A[k][q];
          A[k][p] = c * akp - s * akq;
          A[k][q] = s * akp + c * akq;
        }
#pragma unroll
        for (int k = 0; k < D; ++k) {  // rows p, q
          const double apk = A[p][k], aqk = A[q][k];
          A[p][k] = c * apk - s * aqk;
          A[q][k] = s * apk + c * aqk;
        }
#pragma unroll
        for (int k = 0; k < D; ++k) {
          const double vkp = V[k][p], vkq = V[k][q];
          V[k][p] = c * vkp - s * vkq;
          V[k][q] = s * vkp + c * vkq;
        }
      }
  }
  int best = 0;
#pragma unroll
  for (int i = 1; i < D; ++i)
    if (A[i][i] < A[best][best]) best = i;
#pragma unroll
  for (int k = 0; k < 4; ++k) vec[k] = best == 0 ? V[k][0] : best == 1 ? V[k][1] : best == 2 ? V[k][2] : V[k][3];
}

// Schur reduction of the DLT normal equations in the leading DxD block (D = 4: the 3x4 projection of general points,
// D = 3: the homography of coplanar points).  For fixed last row h3 the optimum is h1 = S^-1 Sx h3, h2 = S^-1 Sy h3,
// and h3 is the smallest eigenvector of M = Sq - Sx S^-1 Sx - Sy S^-1 Sy.  Rows go to p[0..D), p[4..4+D), p[8..8+D).
// False when a Cholesky pivot of S is not above 1e-14 times its diagonal entry (S singular for this D).
template <int D>
__device__ __forceinline__ bool dlt_reduce(const double (&S)[4][4], const double (&Sx)[4][4], const double (&Sy)[4][4],
                                           const double (&Sq)[4][4], double (&p)[12]) {
  double L[4][4];
#pragma unroll
  for (int j = 0; j < D; ++j) {
    double d = S[j][j];
#pragma unroll
    for (int k = 0; k < j; ++k) d -= L[j][k] * L[j][k];
    if (!(d > 1e-14 * S[j][j])) return false;
    L[j][j] = sqrt(d);
#pragma unroll
    for (int i = j + 1; i < D; ++i) {
      double v = S[i][j];
#pragma unroll
      for (int k = 0; k < j; ++k) v -= L[i][k] * L[j][k];
      L[i][j] = v / L[j][j];
    }
  }
  // Tx = S^-1 Sx, Ty = S^-1 Sy (column by column), M = Sq - Sx Tx - Sy Ty
  double Tx[4][4], Ty[4][4], M4[4][4];
#pragma unroll
  for (int col = 0; col < D; ++col) {
    double zx[4], zy[4];
#pragma unroll
    for (int i = 0; i < D; ++i) {
      double vx = Sx[i][col], vy = Sy[i][col];
#pragma unroll
      for (int k = 0; k < i; ++k) {
        vx -= L[i][k] * zx[k];
        vy -= L[i][k] * zy[k];
      }
      zx[i] = vx / L[i][i];
      zy[i] = vy / L[i][i];
    }
#pragma unroll
    for (int i = D - 1; i >= 0; --i) {
      double vx = zx[i], vy = zy[i];
#pragma unroll
      for (int k = i + 1; k < D; ++k) {
        vx -= L[k][i] * Tx[k][col];
        vy -= L[k][i] * Ty[k][col];
      }
      Tx[i][col] = vx / L[i][i];
      Ty[i][col] = vy / L[i][i];
    }
  }
#pragma unroll
  for (int a = 0; a < D; ++a)
#pragma unroll
    for (int b = 0; b < D; ++b) {
      double v = Sq[a][b];
#pragma unroll
      for (int k = 0; k < D; ++k) v -= Sx[a][k] * Tx[k][b] + Sy[a][k] * Ty[k][b];
      M4[a][b] = v;
    }
#pragma unroll
  for (int a = 0; a < D; ++a)
#pragma unroll
    for (int b = a + 1; b < D; ++b) M4[a][b] = M4[b][a] = 0.5 * (M4[a][b] + M4[b][a]);
  double p3[4];
  jacobi_smallest<D>(M4, p3);
#pragma unroll
  for (int a = 0; a < D; ++a) {
    double v1 = 0, v2 = 0;
#pragma unroll
    for (int k = 0; k < D; ++k) {
      v1 += Tx[a][k] * p3[k];
      v2 += Ty[a][k] * p3[k];
    }
    p[a] = v1;
    p[4 + a] = v2;
    p[8 + a] = p3[a];
  }
  return true;
}

constexpr double kPnpPlanarRtol = 1e-10;  // smallest / largest eigenvalue of the centred covariance below which the
                                          // points are solved as a plane: ~1e-14 from float32 rounding of planar
                                          // sets, ~1e-9 for +-1 um out of a 120 mm plane

// normalised DLT on the points whose bit is set in `sel`; X [vn][3] object points, xn [vn][2] normalised image points.
// The 12 unknowns (rows p1, p2, p3 of the 3x4 projection) are reduced to the last row (dlt_reduce<4>) with
// S = sum P P^T, Sx = sum x P P^T, Sy = sum y P P^T, Sq = sum (x^2 + y^2) P P^T (P = normalised homogeneous point).
// Coplanar points make S singular; they are solved as a plane instead, when the centred covariance is flat to
// kPnpPlanarRtol or a pivot of the general reduction fails: the normal n is the largest cross product of two rows of
// the centred covariance (a rank-2 matrix), (e1, e2, n) a right-handed basis, and the homography
// H ~ [r1 r2 t'] on Q = (P.e1, P.e2, 1) reduces the same way (dlt_reduce<3>).  Its sign puts the centroid in front
// (H_22 > 0); r3 = r1 x r2 and the 3x3 of the projection is [r1 r2 r3] [e1 e2 n]^T.  A candidate fails only when
// both reductions do (for example collinear points).
__device__ bool pnp_dlt(const double* X, const double* xn, int vn, unsigned sel, double* R, double* t) {
  double c[3] = {0, 0, 0};
  int m = 0;
  for (int i = 0; i < vn; ++i)
    if ((sel >> i) & 1u) {
      c[0] += X[3 * i]; c[1] += X[3 * i + 1]; c[2] += X[3 * i + 2];
      ++m;
    }
  if (m < 6) return false;
  c[0] /= m; c[1] /= m; c[2] /= m;
  double ms = 0;
  for (int i = 0; i < vn; ++i)
    if ((sel >> i) & 1u) {
      const double a = X[3 * i] - c[0], b = X[3 * i + 1] - c[1], d = X[3 * i + 2] - c[2];
      ms += a * a + b * b + d * d;
    }
  if (!(ms > 0)) return false;
  const double s = 1.0 / sqrt(ms / m);
  double S[4][4], Sx[4][4], Sy[4][4], Sq[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) S[a][b] = Sx[a][b] = Sy[a][b] = Sq[a][b] = 0.0;
  for (int i = 0; i < vn; ++i) {
    if (!((sel >> i) & 1u)) continue;
    const double P[4] = {(X[3 * i] - c[0]) * s, (X[3 * i + 1] - c[1]) * s, (X[3 * i + 2] - c[2]) * s, 1.0};
    const double x = xn[2 * i], y = xn[2 * i + 1], q = x * x + y * y;
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = a; b < 4; ++b) {
        const double pp = P[a] * P[b];
        S[a][b] += pp;
        Sx[a][b] += x * pp;
        Sy[a][b] += y * pp;
        Sq[a][b] += q * pp;
      }
  }
#pragma unroll
  for (int a = 1; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < a; ++b) {
      S[a][b] = S[b][a]; Sx[a][b] = Sx[b][a]; Sy[a][b] = Sy[b][a]; Sq[a][b] = Sq[b][a];
    }
  // rows of the centred covariance C = S[0..2][0..2]: the largest cross product of two rows is the plane normal of a
  // rank-2 C, and det C / (|that cross product| tr C) estimates the smallest eigenvalue over the largest within a factor
  // of 3 (the cross products are columns of adj C, whose eigenvalues are the pairwise products of C's)
  double nv[3] = {0, 0, 0}, nq = 0;
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int b = a + 1; b < 3; ++b) {
      const double v[3] = {S[a][1] * S[b][2] - S[a][2] * S[b][1], S[a][2] * S[b][0] - S[a][0] * S[b][2],
                           S[a][0] * S[b][1] - S[a][1] * S[b][0]};
      const double q = v[0] * v[0] + v[1] * v[1] + v[2] * v[2];
      if (q > nq) {
        nq = q;
        nv[0] = v[0]; nv[1] = v[1]; nv[2] = v[2];
      }
    }
  const double detC = S[0][0] * (S[1][1] * S[2][2] - S[1][2] * S[2][1]) - S[0][1] * (S[1][0] * S[2][2] - S[1][2] * S[2][0]) +
                      S[0][2] * (S[1][0] * S[2][1] - S[1][1] * S[2][0]);
  // coplanar after float32 rounding: the 4x4 system is singular whether or not its pivots fall under 1e-14
  const bool flat = detC <= kPnpPlanarRtol * sqrt(nq) * (S[0][0] + S[1][1] + S[2][2]);
  double p[12], M[9], p4[3];
  if (!flat && dlt_reduce<4>(S, Sx, Sy, Sq, p)) {
    for (int r = 0; r < 3; ++r) {
      for (int k = 0; k < 3; ++k) M[3 * r + k] = p[4 * r + k] * s;
      p4[r] = p[4 * r + 3] - (M[3 * r] * c[0] + M[3 * r + 1] * c[1] + M[3 * r + 2] * c[2]);
    }
  } else {  // coplanar points: planar DLT
    if (!(nq > 0) || !isfinite(nq)) return false;
    const double in = 1.0 / sqrt(nq);
    const double n[3] = {nv[0] * in, nv[1] * in, nv[2] * in};
    const double f0 = fabs(n[0]), f1 = fabs(n[1]), f2 = fabs(n[2]);
    const int ax = (f0 <= f1 && f0 <= f2) ? 0 : (f1 <= f2 ? 1 : 2);  // the axis least aligned with n
    double e1[3] = {ax == 0 ? 0.0 : (ax == 1 ? -n[2] : n[1]), ax == 0 ? n[2] : (ax == 1 ? 0.0 : -n[0]),
                    ax == 0 ? -n[1] : (ax == 1 ? n[0] : 0.0)};  // n x axis
    const double ie = 1.0 / sqrt(e1[0] * e1[0] + e1[1] * e1[1] + e1[2] * e1[2]);
    e1[0] *= ie; e1[1] *= ie; e1[2] *= ie;
    const double e2[3] = {n[1] * e1[2] - n[2] * e1[1], n[2] * e1[0] - n[0] * e1[2], n[0] * e1[1] - n[1] * e1[0]};
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b) S[a][b] = Sx[a][b] = Sy[a][b] = Sq[a][b] = 0.0;
    for (int i = 0; i < vn; ++i) {
      if (!((sel >> i) & 1u)) continue;
      const double P0 = (X[3 * i] - c[0]) * s, P1 = (X[3 * i + 1] - c[1]) * s, P2 = (X[3 * i + 2] - c[2]) * s;
      const double Q[3] = {P0 * e1[0] + P1 * e1[1] + P2 * e1[2], P0 * e2[0] + P1 * e2[1] + P2 * e2[2], 1.0};
      const double x = xn[2 * i], y = xn[2 * i + 1], q = x * x + y * y;
#pragma unroll
      for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int b = a; b < 3; ++b) {
          const double qq = Q[a] * Q[b];
          S[a][b] += qq;
          Sx[a][b] += x * qq;
          Sy[a][b] += y * qq;
          Sq[a][b] += q * qq;
        }
    }
#pragma unroll
    for (int a = 1; a < 3; ++a)
#pragma unroll
      for (int b = 0; b < a; ++b) {
        S[a][b] = S[b][a]; Sx[a][b] = Sx[b][a]; Sy[a][b] = Sy[b][a]; Sq[a][b] = Sq[b][a];
      }
    if (!dlt_reduce<3>(S, Sx, Sy, Sq, p)) return false;
    const double sg = p[10] < 0 ? -s : s;  // H = rows p[0..3), p[4..7), p[8..11); columns 0, 1 carry the scale s
    const double a1[3] = {p[0] * sg, p[4] * sg, p[8] * sg}, a2[3] = {p[1] * sg, p[5] * sg, p[9] * sg};
    const double l1 = sqrt(a1[0] * a1[0] + a1[1] * a1[1] + a1[2] * a1[2]);
    const double l2 = sqrt(a2[0] * a2[0] + a2[1] * a2[1] + a2[2] * a2[2]);
    const double il = 1.0 / sqrt(l1 * l2);
    const double a3[3] = {(a1[1] * a2[2] - a1[2] * a2[1]) * il, (a1[2] * a2[0] - a1[0] * a2[2]) * il,
                          (a1[0] * a2[1] - a1[1] * a2[0]) * il};
    for (int r = 0; r < 3; ++r) {
      for (int k = 0; k < 3; ++k) M[3 * r + k] = a1[r] * e1[k] + a2[r] * e2[k] + a3[r] * n[k];
      p4[r] = (p[10] < 0 ? -p[4 * r + 2] : p[4 * r + 2]) - (M[3 * r] * c[0] + M[3 * r + 1] * c[1] + M[3 * r + 2] * c[2]);
    }
  }
  double det = mat3_det(M);
  if (det < 0) {
    for (int k = 0; k < 9; ++k) M[k] = -M[k];
    for (int k = 0; k < 3; ++k) p4[k] = -p4[k];
    det = -det;
  }
  if (!(det > 0) || !isfinite(det)) return false;
  const double sc = cbrt(det);
  for (int k = 0; k < 9; ++k) R[k] = M[k] / sc;
  for (int it = 0; it < 30; ++it) {  // polar iteration: R <- (R + R^-T) / 2
    double Ri[9], dmax = 0;
    mat3_inv_t(R, Ri);
    for (int k = 0; k < 9; ++k) {
      const double rn = 0.5 * (R[k] + Ri[k]);
      dmax = fmax(dmax, fabs(rn - R[k]));
      R[k] = rn;
    }
    if (dmax < 1e-15) break;
  }
  for (int k = 0; k < 3; ++k) t[k] = p4[k] / sc;
  return isfinite(t[0]) && isfinite(t[1]) && isfinite(t[2]) && isfinite(R[0]);
}

// squared reprojection cost of the selected points; uv in pixels
__device__ __forceinline__ double pnp_cost(const double* X, const double* uv, int vn, unsigned sel, const double* K4,
                                           const double* R, const double* t) {
  double cost = 0;
  for (int i = 0; i < vn; ++i) {
    if (!((sel >> i) & 1u)) continue;
    const double x = R[0] * X[3 * i] + R[1] * X[3 * i + 1] + R[2] * X[3 * i + 2] + t[0];
    const double y = R[3] * X[3 * i] + R[4] * X[3 * i + 1] + R[5] * X[3 * i + 2] + t[1];
    const double z = R[6] * X[3 * i] + R[7] * X[3 * i + 1] + R[8] * X[3 * i + 2] + t[2];
    const double ru = K4[0] * x / z + K4[2] - uv[2 * i], rv = K4[1] * y / z + K4[3] - uv[2 * i + 1];
    cost += ru * ru + rv * rv;
  }
  return cost;
}

// Levenberg-Marquardt on (rotation, translation), left-multiplicative rotation update; K4 = (fx, fy, cx, cy)
__device__ void pnp_lm(const double* X, const double* uv, int vn, unsigned sel, const double* K4, double* R, double* t, int iters) {
  double lam = 1e-3;
  double cost = pnp_cost(X, uv, vn, sel, K4, R, t);
  for (int it = 0; it < iters; ++it) {
    double H[36], g[6];
    for (int k = 0; k < 36; ++k) H[k] = 0;
    for (int k = 0; k < 6; ++k) g[k] = 0;
    for (int i = 0; i < vn; ++i) {
      if (!((sel >> i) & 1u)) continue;
      const double rx = R[0] * X[3 * i] + R[1] * X[3 * i + 1] + R[2] * X[3 * i + 2];
      const double ry = R[3] * X[3 * i] + R[4] * X[3 * i + 1] + R[5] * X[3 * i + 2];
      const double rz = R[6] * X[3 * i] + R[7] * X[3 * i + 1] + R[8] * X[3 * i + 2];
      const double x = rx + t[0], y = ry + t[1], z = rz + t[2];
      const double iz = 1.0 / z;
      const double ru = K4[0] * x * iz + K4[2] - uv[2 * i], rv = K4[1] * y * iz + K4[3] - uv[2 * i + 1];
      // d proj / d Xc
      const double a0 = K4[0] * iz, a2 = -K4[0] * x * iz * iz, b1 = K4[1] * iz, b2 = -K4[1] * y * iz * iz;
      // d Xc / d w = -[RX]x ; columns: (0, -rz, ry), (rz, 0, -rx), (-ry, rx, 0)   (= e_j x RX)
      double Ju[6], Jv[6];
      Ju[0] = a2 * ry;              Ju[1] = a0 * rz - a2 * rx; Ju[2] = -a0 * ry;
      Jv[0] = -b1 * rz + b2 * ry;   Jv[1] = -b2 * rx;          Jv[2] = b1 * rx;
      Ju[3] = a0; Ju[4] = 0;  Ju[5] = a2;
      Jv[3] = 0;  Jv[4] = b1; Jv[5] = b2;
      for (int a = 0; a < 6; ++a) {
        g[a] += Ju[a] * ru + Jv[a] * rv;
        for (int b = a; b < 6; ++b) H[a * 6 + b] += Ju[a] * Ju[b] + Jv[a] * Jv[b];
      }
    }
    for (int a = 0; a < 6; ++a)
      for (int b = 0; b < a; ++b) H[a * 6 + b] = H[b * 6 + a];
    bool ok = false;
    double dmax = 0, dc = 0;
    for (int tries = 0; tries < 10 && !ok; ++tries) {
      double Lm[36], d[6];
      bool spd = true;
      for (int k = 0; k < 36; ++k) Lm[k] = H[k];
      for (int k = 0; k < 6; ++k) Lm[k * 6 + k] += lam * H[k * 6 + k];
      for (int j = 0; j < 6 && spd; ++j) {  // Cholesky, lower triangle in place
        double s = Lm[j * 6 + j];
        for (int k = 0; k < j; ++k) s -= Lm[j * 6 + k] * Lm[j * 6 + k];
        if (!(s > 0)) {
          spd = false;
          break;
        }
        const double l = sqrt(s);
        Lm[j * 6 + j] = l;
        for (int i = j + 1; i < 6; ++i) {
          double v = Lm[i * 6 + j];
          for (int k = 0; k < j; ++k) v -= Lm[i * 6 + k] * Lm[j * 6 + k];
          Lm[i * 6 + j] = v / l;
        }
      }
      if (!spd) {
        lam *= 10;
        continue;
      }
      for (int i = 0; i < 6; ++i) {  // L y = -g
        double v = -g[i];
        for (int k = 0; k < i; ++k) v -= Lm[i * 6 + k] * d[k];
        d[i] = v / Lm[i * 6 + i];
      }
      for (int i = 5; i >= 0; --i) {  // L^T d = y
        double v = d[i];
        for (int k = i + 1; k < 6; ++k) v -= Lm[k * 6 + i] * d[k];
        d[i] = v / Lm[i * 6 + i];
      }
      double E[9], R2[9], t2[3];
      so3_exp(d, E);
      for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) R2[3 * r + c] = E[3 * r] * R[c] + E[3 * r + 1] * R[3 + c] + E[3 * r + 2] * R[6 + c];
      for (int k = 0; k < 3; ++k) t2[k] = t[k] + d[3 + k];
      const double c2 = pnp_cost(X, uv, vn, sel, K4, R2, t2);
      if (c2 < cost) {
        for (int k = 0; k < 9; ++k) R[k] = R2[k];
        for (int k = 0; k < 3; ++k) t[k] = t2[k];
        dc = cost - c2;
        cost = c2;
        lam = fmax(lam / 10, 1e-12);
        dmax = 0;
        for (int k = 0; k < 6; ++k) dmax = fmax(dmax, fabs(d[k]));
        ok = true;
      } else {
        lam *= 10;
      }
    }
    if (!ok || dmax < 1e-12 || dc < 1e-14 * fmax(cost, 1e-30)) break;
  }
}

// transform_points_back_tf (:92-121) in float32, applied to one point
__device__ __forceinline__ float2 pnp_unmap(float2 p, const float* o) {
  // offsets: [0]=h_crop, [1]=w_crop, [8]=sx, [9]=sy, [4]=dx, [5]=dy, [6]=angle, [7]=scale   (:494-504)
  const float sx = o[8], sy = o[9];
  float x = __fadd_rn(__fdiv_rn(p.x, o[7]), o[1]);
  float y = __fadd_rn(__fdiv_rn(p.y, o[7]), o[0]);
  x = __fsub_rn(x, o[4]);
  y = __fsub_rn(y, o[5]);
  const float ang = __fmul_rn(-o[6], 0.017453292519943295f);
  const float a = cosf(ang), b = sinf(ang);
  const float cx = __fdiv_rn(sx, 2.0f), cy = __fdiv_rn(sy, 2.0f);
  const float c = __fsub_rn(__fmul_rn(__fsub_rn(1.0f, a), cx), __fmul_rn(b, cy));
  const float d = __fadd_rn(__fmul_rn(b, cx), __fmul_rn(__fsub_rn(1.0f, a), cy));
  return make_float2(__fadd_rn(__fadd_rn(__fmul_rn(a, x), __fmul_rn(b, y)), c),
                     __fadd_rn(__fadd_rn(__fmul_rn(-b, x), __fmul_rn(a, y)), d));
}

// one warp per object.  pts2d [n,vn,2] (x,y) px, pts3d [n,vn,3], cam [n,3,3] (zero skew), offsets [n,10] or NULL
__global__ void __launch_bounds__(128) k_pnp(PnpParams pp, const float* __restrict__ pts2d, const float* __restrict__ pts3d,
                                            const float* __restrict__ cam, const float* __restrict__ offsets,
                                            float* __restrict__ poses) {
  const int obj = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (obj >= pp.n) return;
  const int vn = pp.vn;
  double X[48], uv[32], xn[32];
  float sum = 0.f;
  for (int i = 0; i < vn; ++i) {
    float2 p = make_float2(pts2d[((size_t)obj * vn + i) * 2], pts2d[((size_t)obj * vn + i) * 2 + 1]);
    sum = __fadd_rn(sum, __fadd_rn(p.x, p.y));
    uv[2 * i] = p.x;
    uv[2 * i + 1] = p.y;
  }
  float* out = poses + (size_t)obj * 12;
  // map_offsets :489 / map_pnp :510; a NaN or inf keypoint (non-finite sum) also gives zeros, as in the reference, where
  // cv2 returns a NaN translation for it and pnp() returns zeros (:48-50)
  bool dead = fabsf(sum) < 0.01f || !isfinite(sum);
  if (!dead && offsets) {
    sum = 0.f;
    for (int i = 0; i < vn; ++i) {
      const float2 q = pnp_unmap(make_float2((float)uv[2 * i], (float)uv[2 * i + 1]), offsets + (size_t)obj * 10);
      uv[2 * i] = q.x;
      uv[2 * i + 1] = q.y;
      sum = __fadd_rn(sum, __fadd_rn(q.x, q.y));
    }
    dead = fabsf(sum) < 0.01f || !isfinite(sum);
  }
  if (dead) {
    if (lane < 12) out[lane] = 0.f;
    return;
  }
  const float* Kf = cam + (size_t)obj * 9;
  const double K4[4] = {Kf[0], Kf[4], Kf[2], Kf[5]};
  for (int i = 0; i < vn; ++i) {
    X[3 * i] = pts3d[((size_t)obj * vn + i) * 3];
    X[3 * i + 1] = pts3d[((size_t)obj * vn + i) * 3 + 1];
    X[3 * i + 2] = pts3d[((size_t)obj * vn + i) * 3 + 2];
    xn[2 * i] = (uv[2 * i] - K4[2]) / K4[0];
    xn[2 * i + 1] = (uv[2 * i + 1] - K4[3]) / K4[1];
  }
  // candidates: 0 = all points, 1..vn = leave one out, then leave two out (a < b)
  const unsigned full = vn >= 32 ? 0xffffffffu : ((1u << vn) - 1u);
  const int ncand = 1 + vn + vn * (vn - 1) / 2;
  double bestR[9], bestT[3], bestCost = 1e300;
  int bestInl = -1, bestIdx = 0x7fffffff;
  for (int cnd = lane; cnd < ncand; cnd += 32) {
    unsigned sel = full;
    if (cnd >= 1 && cnd <= vn) {
      sel &= ~(1u << (cnd - 1));
    } else if (cnd > vn) {
      int k = cnd - vn - 1, a = 0;
      while (k >= vn - 1 - a) {
        k -= vn - 1 - a;
        ++a;
      }
      sel &= ~(1u << a);
      sel &= ~(1u << (a + 1 + k));
    }
    double R[9], t[3];
    if (!pnp_dlt(X, xn, vn, sel, R, t)) continue;
    pnp_lm(X, uv, vn, sel, K4, R, t, 5);
    int ninl = 0;
    double cost = 0;
    bool front = true;
    for (int i = 0; i < vn; ++i) {
      const double x = R[0] * X[3 * i] + R[1] * X[3 * i + 1] + R[2] * X[3 * i + 2] + t[0];
      const double y = R[3] * X[3 * i] + R[4] * X[3 * i + 1] + R[5] * X[3 * i + 2] + t[1];
      const double z = R[6] * X[3 * i] + R[7] * X[3 * i + 1] + R[8] * X[3 * i + 2] + t[2];
      if (!(z > 0)) front = false;
      const double ru = K4[0] * x / z + K4[2] - uv[2 * i], rv = K4[1] * y / z + K4[3] - uv[2 * i + 1];
      const double e2 = ru * ru + rv * rv;
      if (e2 < (double)pp.reproj_px * pp.reproj_px) {
        ++ninl;
        cost += e2;
      }
    }
    if (!front || !isfinite(cost)) continue;
    if (ninl > bestInl || (ninl == bestInl && cost < bestCost)) {  // candidates come in ascending index per lane
      bestInl = ninl;
      bestCost = cost;
      bestIdx = cnd;
      for (int k = 0; k < 9; ++k) bestR[k] = R[k];
      for (int k = 0; k < 3; ++k) bestT[k] = t[k];
    }
  }
  // warp arg-max of (inliers, -cost, -index)
  int winner = lane;
  {
    int inl = bestInl, idx = bestIdx, who = lane;
    double cst = bestCost;
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      const int oi = __shfl_xor_sync(0xffffffffu, inl, o), ox = __shfl_xor_sync(0xffffffffu, idx, o);
      const int ow = __shfl_xor_sync(0xffffffffu, who, o);
      const double oc = __shfl_xor_sync(0xffffffffu, cst, o);
      const bool better = oi > inl || (oi == inl && (oc < cst || (oc == cst && ox < idx)));
      if (better) {
        inl = oi;
        idx = ox;
        who = ow;
        cst = oc;
      }
    }
    winner = who;
    bestInl = inl;
  }
  if (bestInl < 0) {  // no candidate produced a pose in front of the camera: the reference returns zeros on failure
    if (lane < 12) out[lane] = 0.f;
    return;
  }
  if (lane == winner) {
    pnp_lm(X, uv, vn, full, K4, bestR, bestT, 50);  // cv2.solvePnP(ITERATIVE, useExtrinsicGuess) on all points (:37-46)
    bool fin = true;
    for (int k = 0; k < 3; ++k) fin = fin && isfinite(bestT[k]);
    for (int k = 0; k < 9; ++k) fin = fin && isfinite(bestR[k]);
    const double sg = bestT[2] < 0 ? -1.0 : 1.0;  // :53-55
    for (int r = 0; r < 3; ++r) {
      for (int c = 0; c < 3; ++c) out[4 * r + c] = fin ? (float)(sg * bestR[3 * r + c]) : 0.f;
      out[4 * r + 3] = fin ? (float)(sg * bestT[r]) : 0.f;
    }
  }
}

// K10 — backward of PnP, BPnP_fast (Chen et al., CVPR 2020; the reference's bpnp_layers.py:138-277).
// The pose y is differentiated through the stationarity condition f(x, y) = C^T (pi(y) - x) = 0 with
// C = -2 dpi/dy detached at the forward pose, so that with J = dpi/dy (2vn x 6)
//   dy/dx = (J^T J)^-1 J^T   and   grad_x = J (J^T J)^-1 grad_y.
// J does not depend on the observed points x, and the result does not depend on how the rotation is parameterised:
// y is taken as the left-multiplicative tangent of pnp_lm (R <- exp([w]x) R, t <- t + dt), and the incoming gradient
// is mapped onto it.
//   pose_form 12: poses [n,3,4] = [R|t] as written by k_pnp / poses_pnp.  A t_z < 0 flip (-[R|t], ransac_voting.py:53-55)
//                 is recognised by det(R) < 0: the un-flipped pose is differentiated with the incoming gradient negated.
//                 g_w = vee(A - A^T) with A = G_R R^T, g_t = G_t.
//   pose_form 6:  poses [n,6] = (rvec, tvec) as returned by BPNP_fast; g_w = Jl(rvec)^-T g_rvec, where Jl is the left
//                 Jacobian of SO(3) (exp(r + dr) = exp([Jl dr]x) exp(r)), and g_t = g_tvec.
// Guards, each giving an exact zero gradient for the object instead of NaN / inf:
//   * an all-zero pose (dead object, failed solve, available = 0);
//   * a point at z <= 0 under the differentiated (un-flipped) pose, or any non-finite entry of J or of Jl^-T;
//   * a Cholesky pivot of J^T J that is not above kPnpPivotRtol times its diagonal entry (rank-deficient J, e.g.
//     collinear keypoints; the reference's torch.inverse would fail or return inf there).
// One warp per object, one lane per row of J (point i = lane / 2, coordinate lane % 2); the 21 entries of J^T J are
// warp-reduced and every lane factors the 6x6 system itself.  float64 inside, float32 in and out.
constexpr double kPnpPivotRtol = 1e-10;  // pivot^2 / diagonal; collinear float32 keypoints give ~1e-14

__global__ void __launch_bounds__(128) k_pnp_backward(int n, int vn, int pose_form, const float* __restrict__ pts3d,
                                                     const float* __restrict__ cam, const float* __restrict__ poses,
                                                     const float* __restrict__ grad_poses, float* __restrict__ grad2d) {
  const int obj = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (obj >= n) return;
  const int np = pose_form;  // floats per pose
  const float* P = poses + (size_t)obj * np;
  const float* Gp = grad_poses + (size_t)obj * np;
  bool dead = true;
  for (int k = 0; k < np; ++k) dead = dead && P[k] == 0.f;
  bool ok = !dead;
  double R[9], t[3], gw[3], gt[3];
  if (pose_form == 12) {
    for (int r = 0; r < 3; ++r) {
      for (int c = 0; c < 3; ++c) R[3 * r + c] = P[4 * r + c];
      t[r] = P[4 * r + 3];
    }
    const double sg = mat3_det(R) < 0 ? -1.0 : 1.0;
    double G[9];
    for (int r = 0; r < 3; ++r) {
      for (int c = 0; c < 3; ++c) {
        R[3 * r + c] *= sg;
        G[3 * r + c] = sg * Gp[4 * r + c];
      }
      t[r] *= sg;
      gt[r] = sg * Gp[4 * r + 3];
    }
    double A[9];  // A = G_R R^T
    for (int r = 0; r < 3; ++r)
      for (int c = 0; c < 3; ++c) A[3 * r + c] = G[3 * r] * R[3 * c] + G[3 * r + 1] * R[3 * c + 1] + G[3 * r + 2] * R[3 * c + 2];
    gw[0] = A[7] - A[5];
    gw[1] = A[2] - A[6];
    gw[2] = A[3] - A[1];
  } else {
    const double rv[3] = {P[0], P[1], P[2]}, gr[3] = {Gp[0], Gp[1], Gp[2]};
    for (int k = 0; k < 3; ++k) {
      t[k] = P[3 + k];
      gt[k] = Gp[3 + k];
    }
    // R = exp([r]x) = I + a K + b K^2 (Rodrigues, like so3_exp) from the half angle: a = 2 sh ch / th, b = 2 sh^2 / th^2.
    // Jl^-1 = I - [r]x / 2 + c [r]x^2, so Jl^-T g = g + r x g / 2 + c r x (r x g), c = 1/th^2 - cot(th/2) / (2 th)
    // (series below th = 1e-2; infinite at th = 2 pi, where the guard applies).  sincospi needs no argument-reduction
    // scratch in local memory, unlike sin / cos.
    const double th2 = rv[0] * rv[0] + rv[1] * rv[1] + rv[2] * rv[2], th = sqrt(th2);
    double sh, ch;
    sincospi(th * 0.15915494309189535, &sh, &ch);  // th / (2 pi)
    const double a = th < 1e-12 ? 1.0 : 2.0 * sh * ch / th, b = th < 1e-12 ? 0.5 : 2.0 * sh * sh / th2;
    const double x = rv[0], y = rv[1], z = rv[2];
    R[0] = 1.0 - b * (y * y + z * z); R[1] = -a * z + b * x * y;       R[2] = a * y + b * x * z;
    R[3] = a * z + b * x * y;         R[4] = 1.0 - b * (x * x + z * z); R[5] = -a * x + b * y * z;
    R[6] = -a * y + b * x * z;        R[7] = a * x + b * y * z;         R[8] = 1.0 - b * (x * x + y * y);
    const double cf = th2 < 1e-4 ? 1.0 / 12.0 + th2 * (1.0 / 720.0 + th2 / 30240.0) : 1.0 / th2 - ch / (2.0 * th * sh);
    const double rg[3] = {rv[1] * gr[2] - rv[2] * gr[1], rv[2] * gr[0] - rv[0] * gr[2], rv[0] * gr[1] - rv[1] * gr[0]};
    const double rrg[3] = {rv[1] * rg[2] - rv[2] * rg[1], rv[2] * rg[0] - rv[0] * rg[2], rv[0] * rg[1] - rv[1] * rg[0]};
    for (int k = 0; k < 3; ++k) gw[k] = gr[k] + 0.5 * rg[k] + cf * rrg[k];
    ok = ok && isfinite(cf);
  }
  // this lane's row of J
  const int pt = lane >> 1, coord = lane & 1;
  double Jr[6] = {0, 0, 0, 0, 0, 0};
  if (ok && pt < vn) {
    const float* Kf = cam + (size_t)obj * 9;
    const double f = coord ? Kf[4] : Kf[0];
    const float* Xf = pts3d + ((size_t)obj * vn + pt) * 3;
    const double X0 = Xf[0], X1 = Xf[1], X2 = Xf[2];
    const double rx = R[0] * X0 + R[1] * X1 + R[2] * X2, ry = R[3] * X0 + R[4] * X1 + R[5] * X2,
                 rz = R[6] * X0 + R[7] * X1 + R[8] * X2;
    const double z = rz + t[2], iz = 1.0 / z;
    // d pi_coord / d Xc = (f/z, 0, -f x/z^2) or (0, f/z, -f y/z^2); d Xc / d w = -[RX]x, so the w-part is RX x d
    const double d0 = coord ? 0.0 : f * iz, d1 = coord ? f * iz : 0.0, d2 = -f * (coord ? ry + t[1] : rx + t[0]) * iz * iz;
    Jr[0] = ry * d2 - rz * d1;
    Jr[1] = rz * d0 - rx * d2;
    Jr[2] = rx * d1 - ry * d0;
    Jr[3] = d0;
    Jr[4] = d1;
    Jr[5] = d2;
    bool good = z > 0;
#pragma unroll
    for (int a = 0; a < 6; ++a) good = good && isfinite(Jr[a]);
    ok = good;
  }
  ok = __all_sync(0xffffffffu, ok);
  // J^T J (lower triangle, row-major packed) summed over the warp
  double H[21];
  {
    int k = 0;
#pragma unroll
    for (int a = 0; a < 6; ++a)
#pragma unroll
      for (int b = 0; b <= a; ++b) H[k++] = Jr[a] * Jr[b];
  }
#pragma unroll
  for (int o = 16; o; o >>= 1)
#pragma unroll
    for (int k = 0; k < 21; ++k) H[k] += __shfl_xor_sync(0xffffffffu, H[k], o);
  // Cholesky H = L L^T in place, with the relative pivot test (fixed loop bounds so that H stays in registers)
#pragma unroll
  for (int j = 0; j < 6; ++j) {
    const int jj = j * (j + 1) / 2;
    double s = H[jj + j];
#pragma unroll
    for (int k = 0; k < 6; ++k)
      if (k < j) s -= H[jj + k] * H[jj + k];
    ok = ok && s > kPnpPivotRtol * H[jj + j];
    const double l = sqrt(fmax(s, 1e-300));
    H[jj + j] = l;
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      if (i <= j) continue;
      const int ii = i * (i + 1) / 2;
      double v = H[ii + j];
#pragma unroll
      for (int k = 0; k < 6; ++k)
        if (k < j) v -= H[ii + k] * H[jj + k];
      H[ii + j] = v / l;
    }
  }
  // s = H^-1 g_y: L u = g, L^T s = u
  double sv[6] = {gw[0], gw[1], gw[2], gt[0], gt[1], gt[2]};
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    const int ii = i * (i + 1) / 2;
#pragma unroll
    for (int k = 0; k < 6; ++k)
      if (k < i) sv[i] -= H[ii + k] * sv[k];
    sv[i] /= H[ii + i];
  }
#pragma unroll
  for (int i = 5; i >= 0; --i) {
#pragma unroll
    for (int k = 0; k < 6; ++k)
      if (k > i) sv[i] -= H[k * (k + 1) / 2 + i] * sv[k];
    sv[i] /= H[i * (i + 1) / 2 + i];
  }
  double g = 0;
#pragma unroll
  for (int a = 0; a < 6; ++a) g += Jr[a] * sv[a];
  if (pt < vn) grad2d[(size_t)obj * 2 * vn + lane] = ok ? (float)g : 0.f;
}

}  // namespace casa
