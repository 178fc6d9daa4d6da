// cvf_align.cu -- batched Kabsch alignment and the whole-trajectory feature pre-pass on sm_100a.
//
// Replaces the alignment / feature half of the caller's pp_layer (core.py:65,122) when it runs on its own:
//   core.py:635   self._feature_traj = self.preprocessing_layer(trajectory)   (AutoEncoderTask pre-pass)
// The reference has no source for it (molann.ann.AlignmentLayer / FeatureLayer, examples/dipeptide/main.ipynb:335-348).
//
// This path is HBM-bound (12 N bytes read + 12 N written per frame, ~1.5 kflop): frame tiles are staged
// through shared memory with 1-D bulk async copies (TMA, cp.async.bulk + mbarrier) in both directions, a
// thread owns one frame while it is in shared memory, and several CTAs per SM overlap copy and math.
// Large molecules (a tile would not fit) use one warp per frame with coalesced loads instead.
//
// The backward of both (cvf_align_vjp, cvf_features_vjp) is the autograd backward of utils.Align / FeatureMap / Preprocessing:
// it stands where the reference differentiates molann's layers inside torch.autograd.grad(y, X) (core.py:424).  Same kernel
// shapes as the forwards, 36 N bytes per frame for the alignment; the rotation and K^-1 are recomputed from x.
#include <string.h>

#include "cvf_common.cuh"
#include "cvf_math.cuh"
#include "cvf_tma.cuh"

namespace cvf {

// One frame held at `fr` (3N floats, stride 1): align in place; K^-1 of the rotation goes to `Kinv` when it is not null.
// `off` = 3 * atom index and `refd` = reference positions in double, both shared-memory tables built once per CTA: the per-atom
// loops cost one broadcast LDS where they used to load from global memory, scale and convert.
__device__ __forceinline__ void align_frame_inplace(float* fr, int n_atoms, const int* __restrict__ off, int n_align,
                                                    const double* __restrict__ refd, float* R9, float* c3,
                                                    float* Kinv = nullptr) {
  // one sweep over the alignment atoms (a coordinate is converted to double once): centroid and H = sum x (x) ref, then
  // (x_A - c)^T ref = sum x (x) ref - c (x) sum ref, with sum ref (refd[3 n_align ..]) the rounding residue of the centred reference
  double cx = 0, cy = 0, cz = 0;
  double H[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll 2
  for (int a = 0; a < n_align; ++a) {
    const float* p = fr + off[a];
    const double px = p[0], py = p[1], pz = p[2];
    const double rx = refd[3 * a], ry = refd[3 * a + 1], rz = refd[3 * a + 2];
    cx += px, cy += py, cz += pz;
    H[0] = fma(px, rx, H[0]), H[1] = fma(px, ry, H[1]), H[2] = fma(px, rz, H[2]);
    H[3] = fma(py, rx, H[3]), H[4] = fma(py, ry, H[4]), H[5] = fma(py, rz, H[5]);
    H[6] = fma(pz, rx, H[6]), H[7] = fma(pz, ry, H[7]), H[8] = fma(pz, rz, H[8]);
  }
  const double inv = 1.0 / n_align;
  cx *= inv, cy *= inv, cz *= inv;
  {
    const double sx = refd[3 * n_align], sy = refd[3 * n_align + 1], sz = refd[3 * n_align + 2];
    H[0] = fma(-cx, sx, H[0]), H[1] = fma(-cx, sy, H[1]), H[2] = fma(-cx, sz, H[2]);
    H[3] = fma(-cy, sx, H[3]), H[4] = fma(-cy, sy, H[4]), H[5] = fma(-cy, sz, H[5]);
    H[6] = fma(-cz, sx, H[6]), H[7] = fma(-cz, sy, H[7]), H[8] = fma(-cz, sz, H[8]);
  }
  float R[9];
  double Rd[9];
  cvf_rotation(H, R, Kinv, Rd);
  const float fx = (float)cx, fy = (float)cy, fz = (float)cz;
  const double tx = cx * Rd[0] + cy * Rd[3] + cz * Rd[6], ty = cx * Rd[1] + cy * Rd[4] + cz * Rd[7],
               tz = cx * Rd[2] + cy * Rd[5] + cz * Rd[8];
#pragma unroll 2
  for (int a = 0; a < n_atoms; ++a) {
    float* p = fr + 3 * a;
    const cvf_v3 y = cvf_transform_t(p[0], p[1], p[2], tx, ty, tz, Rd);
    p[0] = y.x, p[1] = y.y, p[2] = y.z;
  }
#pragma unroll
  for (int i = 0; i < 9; ++i) R9[i] = R[i];
  c3[0] = fx, c3[1] = fy, c3[2] = fz;
}

// Thread per frame, tile of `tile_f` frames staged in shared memory (frame-major, stride = 3N floats).
__global__ void __launch_bounds__(128, 6)
align_tile_kernel(const float* __restrict__ x, long long B, int n_atoms, const int32_t* __restrict__ aidx, int n_align,
                  const float* __restrict__ ref, float* __restrict__ y, float* __restrict__ R_out, float* __restrict__ c_out,
                  int tile_f, int use_tma) {
  extern __shared__ __align__(128) float stage[];
  __shared__ __align__(8) uint64_t bar;
  const int tid = threadIdx.x, nt = blockDim.x;
  const int fl = 3 * n_atoms;
  const long long n_tiles = (B + tile_f - 1) / tile_f;
  // tables behind the frame tile (tile_f * fl floats, rounded up to 8 bytes)
  double* s_ref = reinterpret_cast<double*>(stage + (((size_t)tile_f * fl + 1) & ~(size_t)1));
  int* s_off = reinterpret_cast<int*>(s_ref + 3 * n_align + 3);
  for (int a = tid; a < n_align; a += nt) {
    s_off[a] = 3 * aidx[a];
    s_ref[3 * a] = ref[3 * a], s_ref[3 * a + 1] = ref[3 * a + 1], s_ref[3 * a + 2] = ref[3 * a + 2];
  }
  if (tid < 3) {
    double t = 0.0;
    for (int a = 0; a < n_align; ++a) t += (double)ref[3 * a + tid];
    s_ref[3 * n_align + tid] = t;
  }
  if (tid == 0) {
    mbar_init(&bar, 1);
    fence_barrier_init();
  }
  __syncthreads();
  uint32_t phase = 0;
  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const long long f0 = tile * tile_f;
    const int nf = (int)min((long long)tile_f, B - f0);
    const size_t bytes = (size_t)nf * fl * sizeof(float);
    const float* src = x + (size_t)f0 * fl;
    float* dst = y + (size_t)f0 * fl;
    const bool tma = use_tma && (bytes % 16 == 0);
    if (tma) {
      if (tid == 0) {
        mbar_expect_tx(&bar, (uint32_t)bytes);
        bulk_g2s(stage, src, (uint32_t)bytes, &bar);
      }
      mbar_wait(&bar, phase);
      phase ^= 1;
    } else {
      for (int i = tid; i < nf * fl; i += nt) stage[i] = src[i];
      __syncthreads();
    }
    if (tid < nf) {
      float R9[9], c3[3];
      align_frame_inplace(stage + (size_t)tid * fl, n_atoms, s_off, n_align, s_ref, R9, c3);
      if (R_out) {
#pragma unroll
        for (int i = 0; i < 9; ++i) R_out[(f0 + tid) * 9 + i] = R9[i];
      }
      if (c_out) {
        c_out[(f0 + tid) * 3 + 0] = c3[0], c_out[(f0 + tid) * 3 + 1] = c3[1], c_out[(f0 + tid) * 3 + 2] = c3[2];
      }
    }
    if (tma) {
      fence_proxy_async();   // make the generic-proxy writes to `stage` visible to the bulk copy engine
      __syncthreads();
      if (tid == 0) {
        bulk_s2g(dst, stage, (uint32_t)bytes);
        bulk_wait_read();    // `stage` may be overwritten once the engine has read it
      }
      __syncthreads();
    } else {
      __syncthreads();
      for (int i = tid; i < nf * fl; i += nt) dst[i] = stage[i];
      __syncthreads();
    }
  }
}

// Warp per frame for large molecules: coalesced strided loads, warp-shuffle sums, every lane solves the 3x3.
__global__ void __launch_bounds__(256)
align_warp_kernel(const float* __restrict__ x, long long B, int n_atoms, const int32_t* __restrict__ aidx, int n_align,
                  const float* __restrict__ ref, float* __restrict__ y, float* __restrict__ R_out, float* __restrict__ c_out) {
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
  const int fl = 3 * n_atoms;
  for (long long f = warp; f < B; f += n_warps) {
    const float* fr = x + (size_t)f * fl;
    double s[3] = {0, 0, 0};
    for (int a = lane; a < n_align; a += 32) {
      const float* p = fr + 3 * aidx[a];
      s[0] += p[0], s[1] += p[1], s[2] += p[2];
    }
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s[i] += __shfl_xor_sync(0xffffffffu, s[i], o);
    const double inv = 1.0 / n_align;
    const double cx = s[0] * inv, cy = s[1] * inv, cz = s[2] * inv;
    double H[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (int a = lane; a < n_align; a += 32) {
      const float* p = fr + 3 * aidx[a];
      const double px = p[0] - cx, py = p[1] - cy, pz = p[2] - cz;
      const double rx = ref[3 * a], ry = ref[3 * a + 1], rz = ref[3 * a + 2];
      H[0] += px * rx, H[1] += px * ry, H[2] += px * rz;
      H[3] += py * rx, H[4] += py * ry, H[5] += py * rz;
      H[6] += pz * rx, H[7] += pz * ry, H[8] += pz * rz;
    }
#pragma unroll
    for (int i = 0; i < 9; ++i)
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) H[i] += __shfl_xor_sync(0xffffffffu, H[i], o);
    float R[9];
    double Rd[9];
    cvf_rotation(H, R, nullptr, Rd);
    const float c[3] = {(float)cx, (float)cy, (float)cz};
    float* out = y + (size_t)f * fl;
    // coalesced: lane handles coordinate j of atom j/3; output coordinate b = sum_a (x_a - c_a) R[a][b]
    for (int j = lane; j < fl; j += 32) {
      const int a = j / 3, b = j - 3 * a;
      const float* p = fr + 3 * a;
      out[j] = (float)((p[0] - cx) * Rd[b] + (p[1] - cy) * Rd[3 + b] + (p[2] - cz) * Rd[6 + b]);
    }
    if (lane < 9 && R_out) R_out[f * 9 + lane] = R[lane];
    if (lane < 3 && c_out) c_out[f * 3 + lane] = c[lane];
  }
}

// ---- backward of the alignment: g_x = (dy/dx)^T g_y ----------------------------------------------------------------------
// Centroid, H and the rotation are recomputed from x exactly as the forward computes them (nothing is kept between the two
// calls); K^-1 comes out of the same Newton polish.  36 N bytes per frame: x and g_y read, g_x written.
__device__ __forceinline__ void align_rotation_warp(const float* fr, int lane, const int32_t* __restrict__ aidx, int n_align,
                                                    const float* __restrict__ ref, double& cx, double& cy, double& cz,
                                                    double* Rd, float* R, float* Kinv) {
  double s[3] = {0, 0, 0};
  for (int a = lane; a < n_align; a += 32) {
    const float* p = fr + 3 * aidx[a];
    s[0] += p[0], s[1] += p[1], s[2] += p[2];
  }
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s[i] += __shfl_xor_sync(0xffffffffu, s[i], o);
  const double inv = 1.0 / n_align;
  cx = s[0] * inv, cy = s[1] * inv, cz = s[2] * inv;
  double H[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  for (int a = lane; a < n_align; a += 32) {
    const float* p = fr + 3 * aidx[a];
    const double px = p[0] - cx, py = p[1] - cy, pz = p[2] - cz;
    const double rx = ref[3 * a], ry = ref[3 * a + 1], rz = ref[3 * a + 2];
    H[0] += px * rx, H[1] += px * ry, H[2] += px * rz;
    H[3] += py * rx, H[4] += py * ry, H[5] += py * rz;
    H[6] += pz * rx, H[7] += pz * ry, H[8] += pz * rz;
  }
#pragma unroll
  for (int i = 0; i < 9; ++i)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) H[i] += __shfl_xor_sync(0xffffffffu, H[i], o);
  cvf_rotation(H, R, Kinv, Rd);
}

// Thread per frame: the x tile and the g_y tile arrive by bulk copies, each thread aligns its frame of the x tile in place
// (the forward's arithmetic, so y is the forward's y), turns its g_y frame into g_x in place, and the g_x tile leaves by one
// bulk copy.  Plain loads / stores when a pointer is not 16-byte aligned.
__global__ void __launch_bounds__(128, 4)
align_vjp_tile_kernel(const float* __restrict__ x, const float* __restrict__ gy, long long B, int n_atoms,
                      const int32_t* __restrict__ aidx, int n_align, const float* __restrict__ ref, float* __restrict__ gx,
                      int tile_f, int use_tma) {
  extern __shared__ __align__(128) float stage[];
  __shared__ __align__(8) uint64_t bar;
  const int tid = threadIdx.x, nt = blockDim.x;
  const int fl = 3 * n_atoms;
  const long long n_tiles = (B + tile_f - 1) / tile_f;
  float* sx = stage;                                   // [tile_f][fl]
  float* sg = stage + (size_t)tile_f * fl;             // [tile_f][fl], 16-byte aligned (tile_f % 4 == 0)
  double* s_ref = reinterpret_cast<double*>(sg + (((size_t)tile_f * fl + 1) & ~(size_t)1));
  int* s_off = reinterpret_cast<int*>(s_ref + 3 * n_align + 3);
  int* s_idx = s_off + n_align;
  float* s_reff = reinterpret_cast<float*>(s_idx + n_align);
  for (int a = tid; a < n_align; a += nt) {
    s_off[a] = 3 * aidx[a];
    s_idx[a] = aidx[a];
    s_ref[3 * a] = ref[3 * a], s_ref[3 * a + 1] = ref[3 * a + 1], s_ref[3 * a + 2] = ref[3 * a + 2];
    s_reff[3 * a] = ref[3 * a], s_reff[3 * a + 1] = ref[3 * a + 1], s_reff[3 * a + 2] = ref[3 * a + 2];
  }
  if (tid < 3) {
    double t = 0.0;
    for (int a = 0; a < n_align; ++a) t += (double)ref[3 * a + tid];
    s_ref[3 * n_align + tid] = t;
  }
  if (tid == 0) {
    mbar_init(&bar, 1);
    fence_barrier_init();
  }
  __syncthreads();
  uint32_t phase = 0;
  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const long long f0 = tile * tile_f;
    const int nf = (int)min((long long)tile_f, B - f0);
    const size_t bytes = (size_t)nf * fl * sizeof(float);
    const size_t off = (size_t)f0 * fl;
    const bool tma = use_tma && (bytes % 16 == 0);
    if (tma) {
      if (tid == 0) {
        mbar_expect_tx(&bar, (uint32_t)(2 * bytes));
        bulk_g2s(sx, x + off, (uint32_t)bytes, &bar);
        bulk_g2s(sg, gy + off, (uint32_t)bytes, &bar);
      }
      mbar_wait(&bar, phase);
      phase ^= 1;
    } else {
      for (int i = tid; i < nf * fl; i += nt) sx[i] = x[off + i], sg[i] = gy[off + i];
      __syncthreads();
    }
    if (tid < nf) {
      float R[9], Kinv[6], c3[3];
      float* fr = sx + (size_t)tid * fl;
      align_frame_inplace(fr, n_atoms, s_off, n_align, s_ref, R, c3, Kinv);
      cvf_align_vjp_frame(fr, sg + (size_t)tid * fl, n_atoms, 1, s_idx, n_align, s_reff, R, Kinv);
    }
    if (tma) {
      fence_proxy_async();
      __syncthreads();
      if (tid == 0) {
        bulk_s2g(gx + off, sg, (uint32_t)bytes);
        bulk_wait_read();
      }
      __syncthreads();
    } else {
      __syncthreads();
      for (int i = tid; i < nf * fl; i += nt) gx[off + i] = sg[i];
      __syncthreads();
    }
  }
}

// Warp per frame for molecules whose tiles do not fit shared memory.  Lanes stride over atoms for tau and sum G (the frame's
// x and g_y come from HBM once; the second pass re-reads g_y from L1/L2), then write g_x = G R^T coalesced by coordinate;
// the alignment atoms' correction is added afterwards by atomics (an atom listed twice in align_idx gets both).
__global__ void __launch_bounds__(256)
align_vjp_warp_kernel(const float* __restrict__ x, const float* __restrict__ gy, long long B, int n_atoms,
                      const int32_t* __restrict__ aidx, int n_align, const float* __restrict__ ref, float* __restrict__ gx) {
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
  const int fl = 3 * n_atoms;
  for (long long f = warp; f < B; f += n_warps) {
    const float* fr = x + (size_t)f * fl;
    const float* g = gy + (size_t)f * fl;
    float* out = gx + (size_t)f * fl;
    double cx, cy, cz, Rd[9];
    float R[9], Kinv[6];
    align_rotation_warp(fr, lane, aidx, n_align, ref, cx, cy, cz, Rd, R, Kinv);
    const double tx = cx * Rd[0] + cy * Rd[3] + cz * Rd[6], ty = cx * Rd[1] + cy * Rd[4] + cz * Rd[7],
                 tz = cx * Rd[2] + cy * Rd[5] + cz * Rd[8];
    double t[6] = {0, 0, 0, 0, 0, 0};   // tau, sum G
    for (int a = lane; a < n_atoms; a += 32) {
      const float* p = fr + 3 * a;
      const cvf_v3 y = cvf_transform_t(p[0], p[1], p[2], tx, ty, tz, Rd);
      const double gx0 = g[3 * a], gy0 = g[3 * a + 1], gz0 = g[3 * a + 2];
      t[0] += gy0 * y.z - gz0 * y.y, t[1] += gz0 * y.x - gx0 * y.z, t[2] += gx0 * y.y - gy0 * y.x;
      t[3] += gx0, t[4] += gy0, t[5] += gz0;
    }
#pragma unroll
    for (int i = 0; i < 6; ++i)
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) t[i] += __shfl_xor_sync(0xffffffffu, t[i], o);
    for (int j = lane; j < fl; j += 32) {
      const int a = j / 3, b = j - 3 * a;
      out[j] = g[3 * a] * R[3 * b] + g[3 * a + 1] * R[3 * b + 1] + g[3 * a + 2] * R[3 * b + 2];
    }
    const cvf_v3 q = mul_sym(Kinv, v3((float)t[0], (float)t[1], (float)t[2]));
    const double inv = 1.0 / n_align;
    const cvf_v3 s = v3((float)(t[3] * inv), (float)(t[4] * inv), (float)(t[5] * inv));
    __syncwarp();
    for (int a = lane; a < n_align; a += 32) {
      const cvf_v3 d = mul_rowvec_T(s + cross(v3(ref[3 * a], ref[3 * a + 1], ref[3 * a + 2]), q), R);
      float* p = out + 3 * aidx[a];
      atomicAdd(p, -d.x), atomicAdd(p + 1, -d.y), atomicAdd(p + 2, -d.z);
    }
  }
}

// ---- whole-trajectory feature pre-pass (general features): thread per frame ---------------------------
struct FeatPlan {
  int n_atoms, n_used, n_align, n_feat, d_r;
  const int32_t* used_atoms;
  const int32_t* align_used;
  const float* ref;
  const int32_t* feat;
};

__global__ void __launch_bounds__(128)
features_kernel(const FeatPlan P, const float* __restrict__ x, long long B, float* __restrict__ r_out) {
  // shared: per thread a private column of 3*n_used coordinates and d_r outputs, stride blockDim (+1 pad via odd stride)
  extern __shared__ float sm[];
  const int tid = threadIdx.x, nt = blockDim.x;
  const int S = nt + 1;
  float* Y = sm;                          // [3 n_used][S]
  float* O = sm + 3 * P.n_used * S;       // [d_r][S]
  const long long n_tiles = (B + nt - 1) / nt;
  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const long long f0 = tile * nt;
    const int nf = (int)min((long long)nt, B - f0);
    const int nu3 = 3 * P.n_used;
    for (int idx = tid; idx < nf * nu3; idx += nt) {
      const int f = idx / nu3, j = idx - f * nu3;
      const int a = j / 3, c = j - 3 * a;
      Y[j * S + f] = x[(size_t)(f0 + f) * 3 * P.n_atoms + 3 * P.used_atoms[a] + c];
    }
    __syncthreads();
    if (tid < nf) {
      const int f = tid;
      auto ld = [&](int atom) { return v3(Y[(3 * atom) * S + f], Y[(3 * atom + 1) * S + f], Y[(3 * atom + 2) * S + f]); };
      if (P.n_align > 0) {
        double cx = 0, cy = 0, cz = 0;
        for (int a = 0; a < P.n_align; ++a) {
          const cvf_v3 p = ld(P.align_used[a]);
          cx += p.x, cy += p.y, cz += p.z;
        }
        const double inv = 1.0 / P.n_align;
        cx *= inv, cy *= inv, cz *= inv;
        double H[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
        for (int a = 0; a < P.n_align; ++a) {
          const cvf_v3 p = ld(P.align_used[a]);
          const double px = p.x - cx, py = p.y - cy, pz = p.z - cz;
          const double rx = P.ref[3 * a], ry = P.ref[3 * a + 1], rz = P.ref[3 * a + 2];
          H[0] += px * rx, H[1] += px * ry, H[2] += px * rz;
          H[3] += py * rx, H[4] += py * ry, H[5] += py * rz;
          H[6] += pz * rx, H[7] += pz * ry, H[8] += pz * rz;
        }
        float R[9];
        double Rd[9];
        cvf_rotation(H, R, nullptr, Rd);
        for (int a = 0; a < P.n_used; ++a) {
          const cvf_v3 p = ld(a);
          const cvf_v3 q = cvf_transform(p.x, p.y, p.z, cx, cy, cz, Rd);
          Y[(3 * a) * S + f] = q.x, Y[(3 * a + 1) * S + f] = q.y, Y[(3 * a + 2) * S + f] = q.z;
        }
      }
      int col = 0;
      for (int j = 0; j < P.n_feat; ++j) {
        const int32_t* fr = P.feat + 5 * j;
        const int type = fr[0];
        if (type == CVF_FEAT_POSITION) {
          const cvf_v3 p = ld(fr[1]);
          O[col * S + f] = p.x, O[(col + 1) * S + f] = p.y, O[(col + 2) * S + f] = p.z;
          col += 3;
        } else if (type == CVF_FEAT_BOND) {
          cvf_v3 g;
          O[col * S + f] = cvf_bond(ld(fr[1]), ld(fr[2]), g);
          col += 1;
        } else if (type == CVF_FEAT_ANGLE) {
          cvf_v3 ga, gc;
          O[col * S + f] = cvf_angle(ld(fr[1]), ld(fr[2]), ld(fr[3]), ga, gc);
          col += 1;
        } else {
          float cs, sn;
          cvf_v3 g[4];
          cvf_dihedral(ld(fr[1]), ld(fr[2]), ld(fr[3]), ld(fr[4]), cs, sn, g);
          O[col * S + f] = cs, O[(col + 1) * S + f] = sn;
          col += 2;
        }
      }
    }
    __syncthreads();
    for (int idx = tid; idx < nf * P.d_r; idx += nt) {
      const int f = idx / P.d_r, j = idx - f * P.d_r;
      r_out[(size_t)(f0 + f) * P.d_r + j] = O[j * S + f];
    }
    __syncthreads();
  }
}

// Backward of features_kernel: g_x = (dr/dx)^T g_r.  Same staging (a frame-minor column per thread, stride nt + 1): the used
// atoms' coordinates, their gradient G and the frame's g_r row.  A thread aligns its column exactly as the forward does, adds
// the feature stencils times g_r into G, applies the Kabsch adjoint, and the whole [nf, N, 3] g_x tile is written coalesced
// through an atom -> used-slot table; atoms no record reads get exact zeros.
__global__ void __launch_bounds__(128)
features_vjp_kernel(const FeatPlan P, const float* __restrict__ x, const float* __restrict__ g_r, long long B,
                    float* __restrict__ g_x) {
  extern __shared__ float sm[];
  const int tid = threadIdx.x, nt = blockDim.x;
  const int S = nt + 1;
  const int nu3 = 3 * P.n_used, fl = 3 * P.n_atoms;
  float* Y = sm;                      // [3 n_used][S]
  float* G = Y + nu3 * S;             // [3 n_used][S]
  float* U = G + nu3 * S;             // [d_r][S]
  int* slot = reinterpret_cast<int*>(U + P.d_r * S);   // [n_atoms]: used slot of an atom, -1 if no record reads it
  for (int a = tid; a < P.n_atoms; a += nt) slot[a] = -1;
  __syncthreads();
  for (int u = tid; u < P.n_used; u += nt) slot[P.used_atoms[u]] = u;
  __syncthreads();
  const long long n_tiles = (B + nt - 1) / nt;
  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const long long f0 = tile * nt;
    const int nf = (int)min((long long)nt, B - f0);
    for (int idx = tid; idx < nf * nu3; idx += nt) {
      const int f = idx / nu3, j = idx - f * nu3;
      const int a = j / 3, c = j - 3 * a;
      Y[j * S + f] = x[(size_t)(f0 + f) * fl + 3 * P.used_atoms[a] + c];
    }
    for (int idx = tid; idx < nf * P.d_r; idx += nt) {
      const int f = idx / P.d_r, j = idx - f * P.d_r;
      U[j * S + f] = g_r[(size_t)(f0 + f) * P.d_r + j];
    }
    __syncthreads();
    if (tid < nf) {
      const int f = tid;
      float R[9], Kinv[6];
      if (P.n_align > 0) {
        auto ld = [&](int atom) { return v3(Y[(3 * atom) * S + f], Y[(3 * atom + 1) * S + f], Y[(3 * atom + 2) * S + f]); };
        double cx = 0, cy = 0, cz = 0;
        for (int a = 0; a < P.n_align; ++a) {
          const cvf_v3 p = ld(P.align_used[a]);
          cx += p.x, cy += p.y, cz += p.z;
        }
        const double inv = 1.0 / P.n_align;
        cx *= inv, cy *= inv, cz *= inv;
        double H[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
        for (int a = 0; a < P.n_align; ++a) {
          const cvf_v3 p = ld(P.align_used[a]);
          const double px = p.x - cx, py = p.y - cy, pz = p.z - cz;
          const double rx = P.ref[3 * a], ry = P.ref[3 * a + 1], rz = P.ref[3 * a + 2];
          H[0] += px * rx, H[1] += px * ry, H[2] += px * rz;
          H[3] += py * rx, H[4] += py * ry, H[5] += py * rz;
          H[6] += pz * rx, H[7] += pz * ry, H[8] += pz * rz;
        }
        double Rd[9];
        cvf_rotation(H, R, Kinv, Rd);
        for (int a = 0; a < P.n_used; ++a) {
          const cvf_v3 p = ld(a);
          const cvf_v3 q = cvf_transform(p.x, p.y, p.z, cx, cy, cz, Rd);
          Y[(3 * a) * S + f] = q.x, Y[(3 * a + 1) * S + f] = q.y, Y[(3 * a + 2) * S + f] = q.z;
        }
      }
      for (int j = 0; j < nu3; ++j) G[j * S + f] = 0.0f;
      cvf_features_vjp_frame(Y + f, G + f, S, P.feat, P.n_feat, U + f, S);
      if (P.n_align > 0) cvf_align_vjp_frame(Y + f, G + f, P.n_used, S, P.align_used, P.n_align, P.ref, R, Kinv);
    }
    __syncthreads();
    for (int idx = tid; idx < nf * fl; idx += nt) {
      const int f = idx / fl, j = idx - f * fl;
      const int a = j / 3, c = j - 3 * a;
      const int u = slot[a];
      g_x[(size_t)f0 * fl + idx] = u >= 0 ? G[(3 * u + c) * S + f] : 0.0f;
    }
    __syncthreads();
  }
}

}  // namespace cvf

using namespace cvf;

extern "C" int cvf_align_fwd(const float* x, int64_t B, int32_t n_atoms, const int32_t* align_idx, int32_t n_align,
                             const float* ref_centred, float* y_out, float* R_out, float* c_out, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (!x || !y_out || !align_idx || !ref_centred || B < 1 || n_atoms < 1 || n_align < 3 || n_align > n_atoms) {
    set_error("cvf_align_fwd: bad argument (B=%lld, n_atoms=%d, n_align=%d)", (long long)B, n_atoms, n_align);
    return CVF_E_ARG;
  }
  const size_t frame_bytes = (size_t)n_atoms * 12;
  int tile_f = 0;
  for (int t = 128; t >= 32; t >>= 1)
    if ((size_t)t * frame_bytes <= 56 * 1024) {
      tile_f = t;
      break;
    }
  if (tile_f > 0) {
    const size_t smem = (((size_t)tile_f * frame_bytes + 7) & ~(size_t)7) + (size_t)n_align * (3 * sizeof(double) + sizeof(int)) + 3 * sizeof(double);
    CVF_CUDA(cudaFuncSetAttribute(align_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const long long n_tiles = (B + tile_f - 1) / tile_f;
    const int per_sm = (int)((size_t)max_smem_optin() / (smem + 1024));
    long long grid = (long long)sm_count() * (per_sm < 1 ? 1 : (per_sm > 8 ? 8 : per_sm));
    if (n_tiles < grid) grid = n_tiles;
    // frames are 16-byte aligned in global memory iff the base is and tile_f * 12 N is a multiple of 16 (tile_f % 4 == 0)
    const int use_tma = (((uintptr_t)x | (uintptr_t)y_out) & 15) == 0 ? 1 : 0;
    CVF_LAUNCH(K_ALIGN, stream, align_tile_kernel<<<(int)grid, tile_f, smem, stream>>>(x, B, n_atoms, align_idx, n_align, ref_centred, y_out, R_out, c_out,
                                                          tile_f, use_tma));
  } else {
    long long grid = (long long)sm_count() * 8;
    const long long need = (B + 7) / 8;
    if (need < grid) grid = need;
    CVF_LAUNCH(K_ALIGN, stream, align_warp_kernel<<<(int)grid, 256, 0, stream>>>(x, B, n_atoms, align_idx, n_align, ref_centred, y_out, R_out, c_out));
  }
  CVF_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int cvf_features_fwd(const float* x, int64_t B, const cvf_preproc* pp, float* r_out, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (!x || !pp || !r_out || B < 1) {
    set_error("cvf_features_fwd: bad argument");
    return CVF_E_ARG;
  }
  if (pp->kind != 1 || pp->n_atoms < 1 || pp->n_used < 1 || !pp->used_atoms || pp->n_feat < 1 || !pp->feat || pp->d_r < 1 ||
      (pp->n_align > 0 && (pp->n_align < 3 || !pp->align_used || !pp->ref))) {
    set_error("cvf_features_fwd: molecular pre-processing descriptor inconsistent");
    return CVF_E_ARG;
  }
  FeatPlan P;
  P.n_atoms = pp->n_atoms, P.n_used = pp->n_used, P.n_align = pp->n_align, P.n_feat = pp->n_feat, P.d_r = pp->d_r;
  P.used_atoms = pp->used_atoms, P.align_used = pp->align_used, P.ref = pp->ref, P.feat = pp->feat;
  int nt = 128;
  size_t smem = 0;
  for (; nt >= 32; nt >>= 1) {
    smem = (size_t)(3 * P.n_used + P.d_r) * (nt + 1) * sizeof(float);
    if (smem <= (size_t)max_smem_optin()) break;
  }
  if (nt < 32) {
    set_error("cvf_features_fwd: %d used atoms + %d features do not fit shared memory", P.n_used, P.d_r);
    return CVF_E_UNSUPPORTED;
  }
  CVF_CUDA(cudaFuncSetAttribute(features_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const long long n_tiles = (B + nt - 1) / nt;
  const int per_sm = (int)((size_t)max_smem_optin() / (smem + 1024));
  long long grid = (long long)sm_count() * (per_sm < 1 ? 1 : (per_sm > 8 ? 8 : per_sm));
  if (n_tiles < grid) grid = n_tiles;
  CVF_LAUNCH(K_FEATURES, stream, features_kernel<<<(int)grid, nt, smem, stream>>>(P, x, B, r_out));
  CVF_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int cvf_align_vjp(const float* x, int64_t B, int32_t n_atoms, const int32_t* align_idx, int32_t n_align,
                             const float* ref_centred, const float* g_y, float* g_x, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (!x || !g_y || !g_x || !align_idx || !ref_centred || B < 1 || n_atoms < 1 || n_align < 3 || n_align > n_atoms) {
    set_error("cvf_align_vjp: bad argument (B=%lld, n_atoms=%d, n_align=%d)", (long long)B, n_atoms, n_align);
    return CVF_E_ARG;
  }
  // two tiles (x and g_y) of tile_f frames within the forward's 56 kB: the same number of CTAs per SM keeps copies in flight
  const size_t frame_bytes = (size_t)n_atoms * 12;
  int tile_f = 0;
  for (int t = 128; t >= 32; t >>= 1)
    if ((size_t)2 * t * frame_bytes <= 56 * 1024) {
      tile_f = t;
      break;
    }
  if (tile_f > 0) {
    const size_t smem = (((size_t)2 * tile_f * frame_bytes + 7) & ~(size_t)7) + (size_t)n_align * (3 * sizeof(double) + 2 * sizeof(int) + 3 * sizeof(float)) +
                        3 * sizeof(double);
    CVF_CUDA(cudaFuncSetAttribute(align_vjp_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const long long n_tiles = (B + tile_f - 1) / tile_f;
    const int per_sm = (int)((size_t)max_smem_optin() / (smem + 1024));
    long long grid = (long long)sm_count() * (per_sm < 1 ? 1 : (per_sm > 8 ? 8 : per_sm));
    if (n_tiles < grid) grid = n_tiles;
    const int use_tma = (((uintptr_t)x | (uintptr_t)g_y | (uintptr_t)g_x) & 15) == 0 ? 1 : 0;
    CVF_LAUNCH(K_ALIGN_VJP, stream, align_vjp_tile_kernel<<<(int)grid, tile_f, smem, stream>>>(x, g_y, B, n_atoms, align_idx, n_align,
                                                                                               ref_centred, g_x, tile_f, use_tma));
  } else {
    long long grid = (long long)sm_count() * 8;
    const long long need = (B + 7) / 8;
    if (need < grid) grid = need;
    CVF_LAUNCH(K_ALIGN_VJP, stream, align_vjp_warp_kernel<<<(int)grid, 256, 0, stream>>>(x, g_y, B, n_atoms, align_idx, n_align, ref_centred, g_x));
  }
  CVF_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int cvf_features_vjp(const float* x, int64_t B, const cvf_preproc* pp, const float* g_r, float* g_x, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (!x || !pp || !g_r || !g_x || B < 1) {
    set_error("cvf_features_vjp: bad argument");
    return CVF_E_ARG;
  }
  if (pp->kind != 1 || pp->n_atoms < 1 || pp->n_used < 1 || !pp->used_atoms || pp->n_feat < 1 || !pp->feat || pp->d_r < 1 ||
      (pp->n_align > 0 && (pp->n_align < 3 || !pp->align_used || !pp->ref))) {
    set_error("cvf_features_vjp: molecular pre-processing descriptor inconsistent");
    return CVF_E_ARG;
  }
  FeatPlan P;
  P.n_atoms = pp->n_atoms, P.n_used = pp->n_used, P.n_align = pp->n_align, P.n_feat = pp->n_feat, P.d_r = pp->d_r;
  P.used_atoms = pp->used_atoms, P.align_used = pp->align_used, P.ref = pp->ref, P.feat = pp->feat;
  int nt = 128;
  size_t smem = 0;
  for (; nt >= 32; nt >>= 1) {
    smem = (size_t)(6 * P.n_used + P.d_r) * (nt + 1) * sizeof(float) + (size_t)P.n_atoms * sizeof(int);
    if (smem <= (size_t)max_smem_optin()) break;
  }
  if (nt < 32) {
    set_error("cvf_features_vjp: %d used atoms + %d features + %d atoms do not fit shared memory", P.n_used, P.d_r, P.n_atoms);
    return CVF_E_UNSUPPORTED;
  }
  CVF_CUDA(cudaFuncSetAttribute(features_vjp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const long long n_tiles = (B + nt - 1) / nt;
  const int per_sm = (int)((size_t)max_smem_optin() / (smem + 1024));
  long long grid = (long long)sm_count() * (per_sm < 1 ? 1 : (per_sm > 8 ? 8 : per_sm));
  if (n_tiles < grid) grid = n_tiles;
  CVF_LAUNCH(K_FEATURES_VJP, stream, features_vjp_kernel<<<(int)grid, nt, smem, stream>>>(P, x, g_r, B, g_x));
  CVF_CUDA(cudaGetLastError());
  return 0;
}
