// cvf_math.cuh -- per-frame geometry shared by every kernel (and compiled for the host by
// tests/host_math_check.cpp so the numerics can be checked against the oracle without a GPU).
//
//  * cvf_rotation(): optimal proper rotation of the Kabsch problem  min_R sum |(x_i-c) R - ref_i|^2
//    from the 3x3 covariance H = (x_A-c)^T ref.  The reference path gets this from torch.linalg.svd
//    inside the third-party alignment layer (examples/dipeptide/main.ipynb:345); here: Horn's 4x4
//    quaternion matrix, cyclic Jacobi in fp32 registers, then Newton steps on the rotation in fp64
//    (the optimum is where M = R^T H is symmetric), which also yields K = tr(M) I - M whose inverse the
//    closed-form alignment Jacobian needs (SURVEY.md section 7.3-A).
//  * bond / angle / dihedral values with their gradient stencils.
#pragma once
#include <math.h>

// cyclic Jacobi sweeps on Horn's 4x4 matrix (fp32) and evaluations of M = R^T H in the fp64 polish (the last one only yields
// K^-1): oracle/rotation_budget.py measures the rotation error of every combination against an fp64 SVD.  Four sweeps leave
// the rotation within ~1e-6 even for noisy 10-atom subsets; ONE Newton step then gives <= 2e-11 (two evaluations), a second
// step changes nothing that survives the rounding of the output to float
#ifndef CVF_JACOBI_SWEEPS
#define CVF_JACOBI_SWEEPS 4
#endif
#ifndef CVF_NEWTON_EVALS
#define CVF_NEWTON_EVALS 2
#endif

#if defined(__CUDACC__)
#define CVF_HD __host__ __device__ __forceinline__
#else
#define CVF_HD inline
#endif

struct cvf_v3 {
  float x, y, z;
};
CVF_HD cvf_v3 v3(float x, float y, float z) { return cvf_v3{x, y, z}; }
CVF_HD cvf_v3 operator+(cvf_v3 a, cvf_v3 b) { return v3(a.x + b.x, a.y + b.y, a.z + b.z); }
CVF_HD cvf_v3 operator-(cvf_v3 a, cvf_v3 b) { return v3(a.x - b.x, a.y - b.y, a.z - b.z); }
CVF_HD cvf_v3 operator*(float s, cvf_v3 a) { return v3(s * a.x, s * a.y, s * a.z); }
CVF_HD float dot(cvf_v3 a, cvf_v3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
CVF_HD cvf_v3 cross(cvf_v3 a, cvf_v3 b) {
  return v3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
// row vector times 3x3 row-major matrix:  (a R)_b = sum_a a_a R[a][b]
CVF_HD cvf_v3 mul_rowvec(cvf_v3 a, const float* R) {
  return v3(a.x * R[0] + a.y * R[3] + a.z * R[6], a.x * R[1] + a.y * R[4] + a.z * R[7],
            a.x * R[2] + a.y * R[5] + a.z * R[8]);
}
// row vector times R^T
CVF_HD cvf_v3 mul_rowvec_T(cvf_v3 a, const float* R) {
  return v3(a.x * R[0] + a.y * R[1] + a.z * R[2], a.x * R[3] + a.y * R[4] + a.z * R[5],
            a.x * R[6] + a.y * R[7] + a.z * R[8]);
}
// symmetric 3x3 (xx,xy,xz,yy,yz,zz) times vector
CVF_HD cvf_v3 mul_sym(const float* S, cvf_v3 a) {
  return v3(S[0] * a.x + S[1] * a.y + S[2] * a.z, S[1] * a.x + S[3] * a.y + S[4] * a.z,
            S[2] * a.x + S[4] * a.y + S[5] * a.z);
}

// One Jacobi rotation in the (p,q) plane of the symmetric 4x4 `a`, accumulated into `v`.
template <int p, int q>
CVF_HD void cvf_jacobi_rot(float (&a)[4][4], float (&v)[4][4]) {
  const float apq = a[p][q];
  if (fabsf(apq) > 1e-30f) {
    const float theta = (a[q][q] - a[p][p]) / (2.0f * apq);
    const float t = copysignf(1.0f, theta) / (fabsf(theta) + sqrtf(theta * theta + 1.0f));
    const float c = 1.0f / sqrtf(t * t + 1.0f);
    const float s = t * c;
    a[p][p] -= t * apq;
    a[q][q] += t * apq;
    a[p][q] = 0.0f;
    a[q][p] = 0.0f;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      if (r != p && r != q) {
        const float arp = a[r][p], arq = a[r][q];
        a[r][p] = a[p][r] = c * arp - s * arq;
        a[r][q] = a[q][r] = s * arp + c * arq;
      }
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const float vrp = v[r][p], vrq = v[r][q];
      v[r][p] = c * vrp - s * vrq;
      v[r][q] = s * vrp + c * vrq;
    }
  }
}


// Reciprocal and reciprocal square root of a double from a float seed and ONE Newton step in double (relative error ~1e-13):
// a full-precision double division / square root is ~25-40 instructions on the fp64 pipe, which is the pipe the Kabsch kernels
// are bound by; none of their uses (K^-1 of a Newton step, the quaternion norm before the polish) needs the last bits.
CVF_HD double cvf_rcp_d(double x) {
  const double ax = fabs(x);
  if (!(ax > 1e-30 && ax < 1e30)) return 1.0 / x;
#if defined(__CUDA_ARCH__)
  const double r = (double)__frcp_rn((float)x);
#else
  const double r = (double)(1.0f / (float)x);
#endif
  return fma(r, fma(-x, r, 1.0), r);
}
CVF_HD double cvf_rsqrt_d(double x) {
  if (!(x > 1e-30 && x < 1e30)) return 1.0 / sqrt(x);
#if defined(__CUDA_ARCH__)
  const double r = (double)rsqrtf((float)x);
#else
  const double r = (double)(1.0f / sqrtf((float)x));
#endif
  return r * fma(-0.5 * x, r * r, 1.5);
}

// Largest eigenvalue / eigenvector of Horn's symmetric traceless 4x4 matrix `a` (entries O(1)) without iterating on the matrix:
// Newton on its characteristic polynomial  P(l) = l^4 + c2 l^2 + c1 l + c0  from an upper bound of the largest root (all roots are
// real, so the iteration descends monotonically onto it; Theobald 2005, "QCP"), then the eigenvector as the best-conditioned row
// of adj(a - l I) = const * q q^T.  ~250 instructions instead of the ~2 500 of four cyclic Jacobi sweeps; the result only has to
// be good to ~1e-4, the fp64 Newton polish of the rotation does the rest.  Returns false when the top eigenvalue is (nearly)
// degenerate -- adj(a - l I) vanishes -- and the caller falls back to the Jacobi sweeps.
CVF_HD bool cvf_top_quaternion_qcp(const float (&a)[4][4], float& q0, float& qx, float& qy, float& qz) {
  const double a00 = a[0][0], a01 = a[0][1], a02 = a[0][2], a03 = a[0][3], a11 = a[1][1], a12 = a[1][2], a13 = a[1][3], a22 = a[2][2],
               a23 = a[2][3], a33 = a[3][3];
  // coefficients from the invariants of a symmetric matrix with zero trace: c2 = -tr(a^2)/2, c1 = -tr(a^3)/3, c0 = det(a)
  const double s01 = a01 * a01, s02 = a02 * a02, s03 = a03 * a03, s12 = a12 * a12, s13 = a13 * a13, s23 = a23 * a23;
  const double c2 = -0.5 * (a00 * a00 + a11 * a11 + a22 * a22 + a33 * a33) - (s01 + s02 + s03 + s12 + s13 + s23);
  // 2x2 minors of rows 2,3 (columns i<j), shared by det(a) and by the cofactors below
  const double m01 = a02 * a13 - a03 * a12, m02 = a02 * a23 - a03 * a22, m03 = a02 * a33 - a03 * a23;
  const double m12 = a12 * a23 - a13 * a22, m13 = a12 * a33 - a13 * a23, m23 = a22 * a33 - a23 * a23;
  const double c0 = a00 * (a11 * m23 - a12 * m13 + a13 * m12) - a01 * (a01 * m23 - a12 * m03 + a13 * m02) +
                    a02 * (a01 * m13 - a11 * m03 + a13 * m01) - a03 * (a01 * m12 - a11 * m02 + a12 * m01);
  // tr(a^3) = sum_ijk a_ij a_jk a_ki
  const double t3 = a00 * a00 * a00 + a11 * a11 * a11 + a22 * a22 * a22 + a33 * a33 * a33 +
                    3.0 * (a00 * (s01 + s02 + s03) + a11 * (s01 + s12 + s13) + a22 * (s02 + s12 + s23) + a33 * (s03 + s13 + s23)) +
                    6.0 * (a01 * a02 * a12 + a01 * a03 * a13 + a02 * a03 * a23 + a12 * a13 * a23);
  const double c1 = t3 * (-1.0 / 3.0);
  // sum of squared roots = -2 c2, zero sum  =>  largest root <= sqrt(3/4 * (-2 c2))
  double l = (double)sqrtf((float)(-1.5 * c2)) * (1.0 + 1e-6);   // float square root, nudged up: it only has to stay an upper bound
  if (!(l > 0.0)) return false;
  for (int it = 0; it < 24; ++it) {
    const double l2 = l * l;
    const double P = (l2 + c2) * l2 + c1 * l + c0;
    const double dP = (4.0 * l2 + 2.0 * c2) * l + c1;
    if (!(dP > 0.0)) return false;
    const double step = P * (double)(1.0f / (float)dP);   // approximate reciprocal: still a contraction, 3 instructions
    l -= step;
    if (fabs(step) < 1e-8 * l) break;   // the eigenvector below is formed in fp32: nothing finer survives
  }
  // k = a - l I; cofactors of the symmetric 4x4 (adjugate entries), fp32 is enough
  const float k00 = (float)(a00 - l), k11 = (float)(a11 - l), k22 = (float)(a22 - l), k33 = (float)(a33 - l);
  const float k01 = a[0][1], k02 = a[0][2], k03 = a[0][3], k12 = a[1][2], k13 = a[1][3], k23 = a[2][3];
  // 2x2 minors of rows (2,3) and rows (0,1)
  const float p01 = k02 * k13 - k03 * k12, p02 = k02 * k23 - k03 * k22, p03 = k02 * k33 - k03 * k23;
  const float p12 = k12 * k23 - k13 * k22, p13 = k12 * k33 - k13 * k23, p23 = k22 * k33 - k23 * k23;
  const float r01 = k00 * k11 - k01 * k01, r02 = k00 * k12 - k01 * k02, r03 = k00 * k13 - k01 * k03;
  const float r12 = k01 * k12 - k11 * k02, r13 = k01 * k13 - k11 * k03, r23 = k02 * k13 - k12 * k03;
  // adj_ij (symmetric); rows (2,3) minors p serve rows 0,1 of the adjugate, rows (0,1) minors r serve rows 2,3
  const float A00 = k11 * p23 - k12 * p13 + k13 * p12;
  const float A01 = -(k01 * p23 - k12 * p03 + k13 * p02);
  const float A02 = k01 * p13 - k11 * p03 + k13 * p01;
  const float A03 = -(k01 * p12 - k11 * p02 + k12 * p01);
  const float A11 = k00 * p23 - k02 * p03 + k03 * p02;
  const float A12 = -(k00 * p13 - k01 * p03 + k03 * p01);
  const float A13 = k00 * p12 - k01 * p02 + k02 * p01;
  const float A22 = k33 * r01 - k13 * r03 + k03 * r13;
  const float A23 = -(k23 * r01 - k13 * r02 + k03 * r12);
  const float A33 = k22 * r01 - k12 * r02 + k02 * r12;
  // the row with the largest diagonal entry |const| q_i^2 is the best-conditioned multiple of q
  float best = fabsf(A00);
  q0 = A00, qx = A01, qy = A02, qz = A03;
  if (fabsf(A11) > best) best = fabsf(A11), q0 = A01, qx = A11, qy = A12, qz = A13;
  if (fabsf(A22) > best) best = fabsf(A22), q0 = A02, qx = A12, qy = A22, qz = A23;
  if (fabsf(A33) > best) best = fabsf(A33), q0 = A03, qx = A13, qy = A23, qz = A33;
  (void)r23;
  // |adj| ~ product of the gaps to the other three eigenvalues (entries of a are O(1)): tiny means a degenerate top eigenvalue
  return best > 1e-6f;
}

// H[9] row-major covariance (x_A-c)^T ref in double.  Outputs R[9] (row-major, y = (x-c) R) and,
// if Kinv != nullptr, the inverse of K = tr(M) I - M, M = sym(R^T H), as (xx,xy,xz,yy,yz,zz).
CVF_HD void cvf_rotation(const double* H, float* R, float* Kinv, double* Rd_out = nullptr) {
  // Horn (1987) 4x4 matrix; its top eigenvector is the unit quaternion of the column-convention rotation R^T.
  float a[4][4], v[4][4];
  {
    const float Sxx = (float)H[0], Sxy = (float)H[1], Sxz = (float)H[2];
    const float Syx = (float)H[3], Syy = (float)H[4], Syz = (float)H[5];
    const float Szx = (float)H[6], Szy = (float)H[7], Szz = (float)H[8];
    // scale to O(1) so the Jacobi thresholds are meaningful for any unit system
    float sc = fabsf(Sxx) + fabsf(Sxy) + fabsf(Sxz) + fabsf(Syx) + fabsf(Syy) + fabsf(Syz) + fabsf(Szx) + fabsf(Szy) + fabsf(Szz);
    sc = sc > 0.0f ? 1.0f / sc : 1.0f;
    a[0][0] = sc * (Sxx + Syy + Szz);
    a[0][1] = a[1][0] = sc * (Syz - Szy);
    a[0][2] = a[2][0] = sc * (Szx - Sxz);
    a[0][3] = a[3][0] = sc * (Sxy - Syx);
    a[1][1] = sc * (Sxx - Syy - Szz);
    a[1][2] = a[2][1] = sc * (Sxy + Syx);
    a[1][3] = a[3][1] = sc * (Szx + Sxz);
    a[2][2] = sc * (-Sxx + Syy - Szz);
    a[2][3] = a[3][2] = sc * (Syz + Szy);
    a[3][3] = sc * (-Sxx - Syy + Szz);
  }
  float q0, qx, qy, qz;
  if (!cvf_top_quaternion_qcp(a, q0, qx, qy, qz)) {
    // (nearly) degenerate top eigenvalue: cyclic Jacobi on the 4x4 (rare; the two paths may diverge inside a warp)
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int c = 0; c < 4; ++c) v[r][c] = (r == c) ? 1.0f : 0.0f;
    for (int sweep = 0; sweep < CVF_JACOBI_SWEEPS; ++sweep) {
      cvf_jacobi_rot<0, 1>(a, v);
      cvf_jacobi_rot<0, 2>(a, v);
      cvf_jacobi_rot<0, 3>(a, v);
      cvf_jacobi_rot<1, 2>(a, v);
      cvf_jacobi_rot<1, 3>(a, v);
      cvf_jacobi_rot<2, 3>(a, v);
    }
    // column of the largest eigenvalue (branch-free select keeps v in registers)
    float best = a[0][0];
    q0 = v[0][0], qx = v[1][0], qy = v[2][0], qz = v[3][0];
#pragma unroll
    for (int c = 1; c < 4; ++c) {
      const bool take = a[c][c] > best;
      best = take ? a[c][c] : best;
      q0 = take ? v[0][c] : q0;
      qx = take ? v[1][c] : qx;
      qy = take ? v[2][c] : qy;
      qz = take ? v[3][c] : qz;
    }
  }
  double Rd[9];
  {
    const double n = cvf_rsqrt_d((double)q0 * q0 + (double)qx * qx + (double)qy * qy + (double)qz * qz);
    const double w = q0 * n, x = qx * n, y = qy * n, z = qz * n;
    // R = (column-convention rotation of q)^T
    Rd[0] = w * w + x * x - y * y - z * z;
    Rd[3] = 2.0 * (x * y - w * z);
    Rd[6] = 2.0 * (x * z + w * y);
    Rd[1] = 2.0 * (y * x + w * z);
    Rd[4] = w * w - x * x + y * y - z * z;
    Rd[7] = 2.0 * (y * z - w * x);
    Rd[2] = 2.0 * (z * x - w * y);
    Rd[5] = 2.0 * (z * y + w * x);
    Rd[8] = w * w - x * x - y * y + z * z;
  }
  double Ki[6] = {0, 0, 0, 0, 0, 0};
  double last_th2 = 0.0;   // squared size of the previous Newton step (0 before the first)
  // Newton on the rotation: R <- R exp([d]x),  K d = axial(M - M^T),  M = R^T H.  Error e -> O(e^2).
  for (int it = 0; it < CVF_NEWTON_EVALS + 2; ++it) {
    double M[9];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j) M[3 * i + j] = Rd[i] * H[j] + Rd[3 + i] * H[3 + j] + Rd[6 + i] * H[6 + j];
    const double sxy = 0.5 * (M[1] + M[3]), sxz = 0.5 * (M[2] + M[6]), syz = 0.5 * (M[5] + M[7]);
    const double tr = M[0] + M[4] + M[8];
    const double kxx = tr - M[0], kyy = tr - M[4], kzz = tr - M[8], kxy = -sxy, kxz = -sxz, kyz = -syz;
    const double c00 = kyy * kzz - kyz * kyz, c01 = kxz * kyz - kxy * kzz, c02 = kxy * kyz - kxz * kyy;
    const double c11 = kxx * kzz - kxz * kxz, c12 = kxy * kxz - kxx * kyz, c22 = kxx * kyy - kxy * kxy;
    const double det = kxx * c00 + kxy * c01 + kxz * c02;
    const double idet = det != 0.0 ? cvf_rcp_d(det) : 0.0;
    Ki[0] = c00 * idet, Ki[1] = c01 * idet, Ki[2] = c02 * idet, Ki[3] = c11 * idet, Ki[4] = c12 * idet, Ki[5] = c22 * idet;
    // K^-1 of the polished rotation is what the Jacobian uses: stop after the planned evaluations once the last step was tiny
    // (a step of size th leaves an error O(th^2): after a step below 1e-5 rad the rotation is good to ~1e-10)
    if (it >= CVF_NEWTON_EVALS - 1 && (it == CVF_NEWTON_EVALS + 1 || last_th2 < 1e-10)) break;
    const double t0 = M[7] - M[5], t1 = M[2] - M[6], t2 = M[3] - M[1];
    double d0 = Ki[0] * t0 + Ki[1] * t1 + Ki[2] * t2;
    double d1 = Ki[1] * t0 + Ki[3] * t1 + Ki[4] * t2;
    double d2 = Ki[2] * t0 + Ki[4] * t1 + Ki[5] * t2;
    const double th2 = d0 * d0 + d1 * d1 + d2 * d2;
    if (!(th2 < 0.01)) break;   // degenerate frame (K singular): keep the starting rotation
    last_th2 = th2;
    const double A = 1.0 - th2 * (1.0 / 6.0) + th2 * th2 * (1.0 / 120.0);     // sin(th)/th
    const double Bc = 0.5 - th2 * (1.0 / 24.0) + th2 * th2 * (1.0 / 720.0);   // (1-cos th)/th^2
    // E = I + A [d]x + B [d]x^2
    double E[9];
    E[0] = 1.0 - Bc * (d1 * d1 + d2 * d2);
    E[4] = 1.0 - Bc * (d0 * d0 + d2 * d2);
    E[8] = 1.0 - Bc * (d0 * d0 + d1 * d1);
    E[1] = -A * d2 + Bc * d0 * d1;
    E[3] = A * d2 + Bc * d0 * d1;
    E[2] = A * d1 + Bc * d0 * d2;
    E[6] = -A * d1 + Bc * d0 * d2;
    E[5] = -A * d0 + Bc * d1 * d2;
    E[7] = A * d0 + Bc * d1 * d2;
    double Rn[9];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j) Rn[3 * i + j] = Rd[3 * i] * E[j] + Rd[3 * i + 1] * E[3 + j] + Rd[3 * i + 2] * E[6 + j];
#pragma unroll
    for (int i = 0; i < 9; ++i) Rd[i] = Rn[i];
  }
#pragma unroll
  for (int i = 0; i < 9; ++i) R[i] = (float)Rd[i];
  if (Rd_out) {
#pragma unroll
    for (int i = 0; i < 9; ++i) Rd_out[i] = Rd[i];
  }
  if (Kinv) {
#pragma unroll
    for (int i = 0; i < 6; ++i) Kinv[i] = (float)Ki[i];
  }
}

// y = (x - c) R evaluated in double and rounded once: keeps aligned coordinates within 1 ulp of the exact
// value (the float32 rounding of a 15 A centroid alone would cost 5e-7 A).
CVF_HD cvf_v3 cvf_transform(float px, float py, float pz, double cx, double cy, double cz, const double* Rd) {
  const double dx = px - cx, dy = py - cy, dz = pz - cz;
  return v3((float)(dx * Rd[0] + dy * Rd[3] + dz * Rd[6]), (float)(dx * Rd[1] + dy * Rd[4] + dz * Rd[7]),
            (float)(dx * Rd[2] + dy * Rd[5] + dz * Rd[8]));
}

// the same with the centroid folded in once per frame, t = c R:  y = x R - t.  One subtraction per coordinate fewer, and the
// only conversions left are x -> double and y -> float (the terms are O(|x|), the cancellation costs ~1e-15 in double)
CVF_HD cvf_v3 cvf_transform_t(float px, float py, float pz, double tx, double ty, double tz, const double* Rd) {
  const double dx = px, dy = py, dz = pz;
  return v3((float)fma(dx, Rd[0], fma(dy, Rd[3], fma(dz, Rd[6], -tx))), (float)fma(dx, Rd[1], fma(dy, Rd[4], fma(dz, Rd[7], -ty))),
            (float)fma(dx, Rd[2], fma(dy, Rd[5], fma(dz, Rd[8], -tz))));
}

// ---- feature stencils (values + gradient w.r.t. the atoms of the feature) -------------------------
// bond |b-a|: gradient w.r.t. b is g, w.r.t. a is -g
CVF_HD float cvf_bond(cvf_v3 a, cvf_v3 b, cvf_v3& g) {
  const cvf_v3 d = b - a;
  const float n = sqrtf(dot(d, d));
  g = (1.0f / n) * d;
  return n;
}
// cos of the angle at m between (a-m) and (c-m); gradients ga (atom a), gc (atom c); atom m gets -(ga+gc)
CVF_HD float cvf_angle(cvf_v3 a, cvf_v3 m, cvf_v3 c, cvf_v3& ga, cvf_v3& gc) {
  const cvf_v3 u = a - m, w = c - m;
  const float inu = 1.0f / sqrtf(dot(u, u)), inw = 1.0f / sqrtf(dot(w, w));
  const cvf_v3 uh = inu * u, wh = inw * w;
  const float cs = dot(uh, wh);
  ga = inu * (wh - cs * uh);
  gc = inw * (uh - cs * wh);
  return cs;
}
// dihedral of atoms (p0,p1,p2,p3): returns cos, sin and the gradient of the ANGLE phi w.r.t. each atom;
// d cos = -sin * dphi, d sin = cos * dphi.
CVF_HD void cvf_dihedral(cvf_v3 p0, cvf_v3 p1, cvf_v3 p2, cvf_v3 p3, float& cs, float& sn, cvf_v3 (&g)[4]) {
  const cvf_v3 r12 = p1 - p0, r23 = p2 - p1, r34 = p3 - p2;
  const cvf_v3 n1 = cross(r12, r23), n2 = cross(r23, r34);
  const float n1s = dot(n1, n1), n2s = dot(n2, n2), l23s = dot(r23, r23);
  const float l23 = sqrtf(l23s);
  const float iden = 1.0f / sqrtf(n1s * n2s);
  cs = dot(n1, n2) * iden;
  sn = dot(n1, r34) * l23 * iden;
  g[0] = (-l23 / n1s) * n1;
  g[3] = (l23 / n2s) * n2;
  const float p = dot(r12, r23) / l23s, q = dot(r34, r23) / l23s;
  g[1] = (-1.0f - p) * g[0] + q * g[3];
  g[2] = p * g[0] + (-1.0f - q) * g[3];
}
// ---- adjoints (vector-Jacobian products) of one frame -----------------------------------------------------
// Coordinate c of atom a of a frame sits at p[(3 a + c) * st]: st = 1 for a frame stored contiguously, the tile width for a
// frame held as a column of a frame-minor tile.

// Kabsch alignment y = (x - c) R (SURVEY 7.3-A, DESIGN §3): g holds G = dg/dy of the n atoms on entry and dg/dx on return,
//   tau = sum_j G_j x y_j,  q = K^-1 tau,  dg/dx_j = (G_j - 1_A(j) (sum_j G_j / n_A + ref_j x q)) R^T
// with A the alignment atoms aidx[0..n_align) (indices into the n atoms), ref their centred reference positions, R and K^-1
// what cvf_rotation returns for the frame.  No SVD derivative: the rotation's response to x is the K^-1 solve.
CVF_HD void cvf_align_vjp_frame(const float* y, float* g, int n, int st, const int* aidx, int n_align, const float* ref,
                                const float* R, const float* Kinv) {
  double t0 = 0, t1 = 0, t2 = 0, s0 = 0, s1 = 0, s2 = 0;
  for (int a = 0; a < n; ++a) {
    const float* p = y + 3 * a * st;
    const float* q = g + 3 * a * st;
    const double yx = p[0], yy = p[st], yz = p[2 * st], gx = q[0], gy = q[st], gz = q[2 * st];
    t0 += gy * yz - gz * yy, t1 += gz * yx - gx * yz, t2 += gx * yy - gy * yx;
    s0 += gx, s1 += gy, s2 += gz;
  }
  const cvf_v3 q = mul_sym(Kinv, v3((float)t0, (float)t1, (float)t2));
  const double inv = 1.0 / n_align;
  const cvf_v3 s = v3((float)(s0 * inv), (float)(s1 * inv), (float)(s2 * inv));
  for (int a = 0; a < n_align; ++a) {
    float* p = g + 3 * aidx[a] * st;
    const cvf_v3 d = s + cross(v3(ref[3 * a], ref[3 * a + 1], ref[3 * a + 2]), q);
    p[0] -= d.x, p[st] -= d.y, p[2 * st] -= d.z;
  }
  for (int a = 0; a < n; ++a) {
    float* p = g + 3 * a * st;
    const cvf_v3 o = mul_rowvec_T(v3(p[0], p[st], p[2 * st]), R);
    p[0] = o.x, p[st] = o.y, p[2 * st] = o.z;
  }
}

// Feature records (include/cvf.h: type, then up to 4 atom positions) evaluated on y: G += (dr/dy)^T u.  u[j * ust] is the
// cotangent of output column j; G must hold zeros (or earlier contributions) on entry.  The stencils are the forward's.
CVF_HD void cvf_features_vjp_frame(const float* y, float* G, int st, const int* feat, int n_feat, const float* u, int ust) {
  auto ld = [&](int a) { return v3(y[3 * a * st], y[(3 * a + 1) * st], y[(3 * a + 2) * st]); };
  auto add = [&](int a, cvf_v3 v) {
    float* p = G + 3 * a * st;
    p[0] += v.x, p[st] += v.y, p[2 * st] += v.z;
  };
  int col = 0;
  for (int j = 0; j < n_feat; ++j) {
    const int* fr = feat + 5 * j;
    const int type = fr[0];
    if (type == 0) {   // CVF_FEAT_POSITION
      add(fr[1], v3(u[col * ust], u[(col + 1) * ust], u[(col + 2) * ust]));
      col += 3;
    } else if (type == 1) {   // CVF_FEAT_BOND
      cvf_v3 gb;
      cvf_bond(ld(fr[1]), ld(fr[2]), gb);
      const cvf_v3 v = u[col * ust] * gb;
      add(fr[2], v), add(fr[1], -1.0f * v);
      col += 1;
    } else if (type == 2) {   // CVF_FEAT_ANGLE
      cvf_v3 ga, gc;
      cvf_angle(ld(fr[1]), ld(fr[2]), ld(fr[3]), ga, gc);
      const float w = u[col * ust];
      add(fr[1], w * ga), add(fr[3], w * gc), add(fr[2], -w * (ga + gc));
      col += 1;
    } else {   // CVF_FEAT_DIHEDRAL: d cos = -sin dphi, d sin = cos dphi
      float cs, sn;
      cvf_v3 gp[4];
      cvf_dihedral(ld(fr[1]), ld(fr[2]), ld(fr[3]), ld(fr[4]), cs, sn, gp);
      const float w = cs * u[(col + 1) * ust] - sn * u[col * ust];
      add(fr[1], w * gp[0]), add(fr[2], w * gp[1]), add(fr[3], w * gp[2]), add(fr[4], w * gp[3]);
      col += 2;
    }
  }
}

// the same with the two middle gradients left implicit: g[1] = (-1-p) g0 + q g3, g[2] = p g0 + (-1-q) g3
CVF_HD void cvf_dihedral_compact(cvf_v3 p0, cvf_v3 p1, cvf_v3 p2, cvf_v3 p3, float& cs, float& sn, cvf_v3& g0, cvf_v3& g3, float& p,
                                 float& q) {
  const cvf_v3 r12 = p1 - p0, r23 = p2 - p1, r34 = p3 - p2;
  const cvf_v3 n1 = cross(r12, r23), n2 = cross(r23, r34);
  const float n1s = dot(n1, n1), n2s = dot(n2, n2), l23s = dot(r23, r23);
  const float l23 = sqrtf(l23s);
  const float iden = 1.0f / sqrtf(n1s * n2s);
  cs = dot(n1, n2) * iden;
  sn = dot(n1, r34) * l23 * iden;
  g0 = (-l23 / n1s) * n1;
  g3 = (l23 / n2s) * n2;
  p = dot(r12, r23) / l23s;
  q = dot(r34, r23) / l23s;
}
