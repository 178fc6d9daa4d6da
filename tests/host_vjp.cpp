// Host build of the per-frame adjoints of colvars-finder_b200/csrc/cvf_math.cuh for the CPU tests (tests/test_preproc_vjp_host.py).
// The frame loops below are the ones the backward kernels of csrc/cvf_align.cu run per thread, with the frame stored
// contiguously (stride 1); compiling them with g++ lets the tests check them against oracle/closed_form.py without a GPU.
#include "../colvars-finder_b200/csrc/cvf_math.cuh"

// g_x = (dy/dx)^T g_y of the Kabsch alignment, B frames of n atoms: centroid, covariance and rotation as the kernels form them
extern "C" void host_align_vjp(const float* x, int B, int n, const int* aidx, int n_align, const float* ref, const float* g_y,
                               float* g_x) {
  float* y = new float[3 * n];
  for (int b = 0; b < B; ++b) {
    const float* fr = x + (size_t)3 * n * b;
    double c[3] = {0, 0, 0};
    for (int a = 0; a < n_align; ++a)
      for (int k = 0; k < 3; ++k) c[k] += fr[3 * aidx[a] + k];
    for (int k = 0; k < 3; ++k) c[k] /= n_align;
    double H[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (int a = 0; a < n_align; ++a)
      for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) H[3 * i + j] += (fr[3 * aidx[a] + i] - c[i]) * (double)ref[3 * a + j];
    float R[9], Kinv[6];
    double Rd[9];
    cvf_rotation(H, R, Kinv, Rd);
    for (int a = 0; a < n; ++a) {
      const cvf_v3 p = cvf_transform(fr[3 * a], fr[3 * a + 1], fr[3 * a + 2], c[0], c[1], c[2], Rd);
      y[3 * a] = p.x, y[3 * a + 1] = p.y, y[3 * a + 2] = p.z;
    }
    float* g = g_x + (size_t)3 * n * b;
    for (int i = 0; i < 3 * n; ++i) g[i] = g_y[(size_t)3 * n * b + i];
    cvf_align_vjp_frame(y, g, n, 1, aidx, n_align, ref, R, Kinv);
  }
  delete[] y;
}

// G = (dr/dy)^T u of the feature records feat [n_feat,5] on frames y [B,n,3]; u [B,d_r]
extern "C" void host_features_vjp(const float* y, int B, int n, const int* feat, int n_feat, int d_r, const float* u, float* G) {
  for (int b = 0; b < B; ++b) {
    float* g = G + (size_t)3 * n * b;
    for (int i = 0; i < 3 * n; ++i) g[i] = 0.0f;
    cvf_features_vjp_frame(y + (size_t)3 * n * b, g, 1, feat, n_feat, u + (size_t)d_r * b, 1);
  }
}
