// cvf_common.cuh -- error plumbing, launch helpers and the shared-memory "row engine" used by the
// eigenfunction and autoencoder step kernels.
//
// Data layout inside a CTA.  A tile is F frames (F = 32, 64 or 128).  Every per-frame quantity lives in
// shared memory as a ROW of F floats (row stride FS = F + 4 floats, so rows stay 16-byte aligned and rows
// r, r+1, .. r+7 start in different bank groups): row[unit][frame].  A lane owns 4 consecutive frames
// (one LDS.128 / STS.128 per row access).  All the small dense layers are evaluated as register-tiled
// products over these rows:
//     forward     out[o][f] = sum_i W[o][i] * in[i][f]      thread tile: 4 outputs x 4 frames
//     transposed  out[i][f] = sum_o W[o][i] * in[o][f]      thread tile: 4 inputs  x 4 frames
//     outer       dW[o][i] += sum_f X[o][f] * Z[i][f]       thread tile: 4 x 4 weights, loop over frames
// with the weights W resident in shared memory in torch's [out][in] layout, `in` padded to a multiple
// of 4 with zeros.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/cvf.h"

namespace cvf {

void set_error(const char* fmt, ...);
int check_cuda(cudaError_t e, const char* what);
int sm_count();
int max_smem_optin();

#define CVF_STR2(x) #x
#define CVF_STR(x) CVF_STR2(x)
#define CVF_CUDA(call)                                                          \
  do {                                                                          \
    int _e = cvf::check_cuda((call), #call " at " __FILE__ ":" CVF_STR(__LINE__)); \
    if (_e) return _e;                                                          \
  } while (0)

// Launch accounting (cvf_api.cu): every kernel launch of the library goes through CVF_LAUNCH, which counts it and, while
// profiling is switched on with cvf_profile_enable(1), brackets it with CUDA events on the launching stream.
enum KernelId {
  K_ALIGN = 0, K_FEATURES, K_EIGEN_STATS, K_EIGEN_GRAD, K_EIGEN_COMBINE, K_REDUCE, K_AE_STEP, K_FAST_PACK, K_FAST_PREP,
  K_FAST_PASS1, K_FAST_STATS, K_FAST_PASS2A, K_FAST_PASS2B, K_FMA_PROBE, K_FAST_JJT, K_AE_FAST_PREP, K_AE_FAST_MAIN, K_AE_FAST_DW,
  K_WEIGHTS, K_ALIGN_VJP, K_FEATURES_VJP, K_COUNT
};
void prof_begin(int id, cudaStream_t stream);
void prof_end(int id, cudaStream_t stream);
#define CVF_LAUNCH(id, stream, ...)   \
  do {                                \
    cvf::prof_begin((id), (stream));  \
    __VA_ARGS__;                      \
    cvf::prof_end((id), (stream));    \
  } while (0)

constexpr int kMaxLayers = CVF_MAX_LAYERS;
constexpr int kMaxK = CVF_MAX_K;

// Shape and shared-memory placement of one Linear+activation chain.
struct NetPlan {
  int L;
  int dims[kMaxLayers + 1];
  int act[kMaxLayers];
  int ld[kMaxLayers];      // padded input width of layer l (multiple of 4)
  int w_off[kMaxLayers];   // float offset of W_l inside the shared-memory parameter block of one net
  int b_off[kMaxLayers];
  int gw_off[kMaxLayers];  // float offset of W_l inside the caller's flat parameter vector (torch order)
  int gb_off[kMaxLayers];
  int n_params;            // per net, unpadded
  int smem_floats;         // per net, padded (multiple of 4)
};

inline int round4(int v) { return (v + 3) & ~3; }

inline int make_net_plan(const cvf_mlp* net, NetPlan* p) {
  if (!net || net->n_layers < 1 || net->n_layers > kMaxLayers) {
    set_error("cvf_mlp: n_layers must be in [1,%d]", kMaxLayers);
    return CVF_E_UNSUPPORTED;
  }
  p->L = net->n_layers;
  int so = 0, go = 0;
  for (int l = 0; l <= p->L; ++l) {
    if (net->dims[l] < 1) {
      set_error("cvf_mlp: dims[%d] = %d", l, net->dims[l]);
      return CVF_E_ARG;
    }
    p->dims[l] = net->dims[l];
  }
  for (int l = 0; l < p->L; ++l) {
    if (net->act[l] < CVF_ACT_NONE || net->act[l] > CVF_ACT_RELU) {
      set_error("cvf_mlp: unknown activation kind %d after layer %d", net->act[l], l);
      return CVF_E_UNSUPPORTED;
    }
    p->act[l] = net->act[l];
    p->ld[l] = round4(p->dims[l]);
    p->w_off[l] = so;
    so += p->dims[l + 1] * p->ld[l];
    p->b_off[l] = so;
    so += round4(p->dims[l + 1]);
    p->gw_off[l] = go;
    go += p->dims[l + 1] * p->dims[l];
    p->gb_off[l] = go;
    go += p->dims[l + 1];
  }
  p->n_params = go;
  p->smem_floats = so;
  return 0;
}

#if defined(__CUDACC__)

// ---- device helpers --------------------------------------------------------------------------------
__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }

// copy one net's parameters from the caller's flat vector into the padded shared-memory block
__device__ inline void load_net_params(const NetPlan& np, const float* __restrict__ g, float* s, int tid, int nt) {
  for (int i = tid; i < np.smem_floats; i += nt) s[i] = 0.0f;
  __syncthreads();
  for (int l = 0; l < np.L; ++l) {
    const int nin = np.dims[l], nout = np.dims[l + 1];
    for (int i = tid; i < nin * nout; i += nt) s[np.w_off[l] + (i / nin) * np.ld[l] + (i % nin)] = g[np.gw_off[l] + i];
    for (int i = tid; i < nout; i += nt) s[np.b_off[l] + i] = g[np.gb_off[l] + i];
  }
}

// ---- vectors of FPL consecutive frames (FPL = 2: LDS.64, FPL = 4: LDS.128) ----------------------------
template <int N> struct FVec;
template <> struct FVec<2> {
  float v[2];
  __device__ __forceinline__ static FVec ld(const float* p) { const float2 t = *reinterpret_cast<const float2*>(p); return FVec{{t.x, t.y}}; }
  __device__ __forceinline__ void st(float* p) const { *reinterpret_cast<float2*>(p) = make_float2(v[0], v[1]); }
};
template <> struct FVec<4> {
  float v[4];
  __device__ __forceinline__ static FVec ld(const float* p) { const float4 t = *reinterpret_cast<const float4*>(p); return FVec{{t.x, t.y, t.z, t.w}}; }
  __device__ __forceinline__ void st(float* p) const { *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]); }
};

// tanh with <= ~3 ulp error and no divergent slow path: odd minimax polynomial below 0.55, 1 - 2/(e^{2|x|}+1)
// with ex2.approx / rcp.approx above (tanh.approx's 2^-11 error would break the 1e-5 parity target).
__device__ __forceinline__ float cvf_tanh(float x) {
  const float ax = fabsf(x), s = x * x;
  float p = fmaf(-0.00622109929f, s, 0.0210381374f);
  p = fmaf(p, s, -0.0538453273f);
  p = fmaf(p, s, 0.133325338f);
  p = fmaf(p, s, -0.333333164f);
  const float small = fmaf(x * s, p, x);
  float e, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(ax * 2.885390082f));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(e + 1.0f));
  const float big = copysignf(fmaf(-2.0f, r, 1.0f), x);
  return ax < 0.55f ? small : big;
}

// packed f32x2 arithmetic (Blackwell FFMA2 / FMUL2 / FADD2: two fp32 lanes per issue slot)
typedef unsigned long long cvf_u64;
__device__ __forceinline__ float2 cvf_ffma2(float2 a, float2 b, float2 c) {
  cvf_u64 d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;"
      : "=l"(d)
      : "l"(*reinterpret_cast<cvf_u64*>(&a)), "l"(*reinterpret_cast<cvf_u64*>(&b)), "l"(*reinterpret_cast<cvf_u64*>(&c)));
  return *reinterpret_cast<float2*>(&d);
}
__device__ __forceinline__ float2 cvf_fmul2(float2 a, float2 b) {
  cvf_u64 d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(*reinterpret_cast<cvf_u64*>(&a)), "l"(*reinterpret_cast<cvf_u64*>(&b)));
  return *reinterpret_cast<float2*>(&d);
}
__device__ __forceinline__ float2 cvf_fadd2(float2 a, float2 b) {
  cvf_u64 d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(*reinterpret_cast<cvf_u64*>(&a)), "l"(*reinterpret_cast<cvf_u64*>(&b)));
  return *reinterpret_cast<float2*>(&d);
}
// cvf_tanh on two values at once: the same operations in the same order -- bit-identical results -- with the polynomial, the
// scaling and the final 1 - 2r as packed f32x2 instructions (10 instead of 16 issue slots per value)
__device__ __forceinline__ float2 cvf_tanh2(float2 x) {
  const float2 s = cvf_fmul2(x, x);
  float2 p = cvf_ffma2(make_float2(-0.00622109929f, -0.00622109929f), s, make_float2(0.0210381374f, 0.0210381374f));
  p = cvf_ffma2(p, s, make_float2(-0.0538453273f, -0.0538453273f));
  p = cvf_ffma2(p, s, make_float2(0.133325338f, 0.133325338f));
  p = cvf_ffma2(p, s, make_float2(-0.333333164f, -0.333333164f));
  const float2 small = cvf_ffma2(cvf_fmul2(x, s), p, x);
  const float2 ax = make_float2(fabsf(x.x), fabsf(x.y));
  const float2 t = cvf_fmul2(ax, make_float2(2.885390082f, 2.885390082f));
  float2 e, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e.x) : "f"(t.x));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e.y) : "f"(t.y));
  const float2 e1 = cvf_fadd2(e, make_float2(1.0f, 1.0f));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r.x) : "f"(e1.x));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r.y) : "f"(e1.y));
  const float2 b = cvf_ffma2(make_float2(-2.0f, -2.0f), r, make_float2(1.0f, 1.0f));
  return make_float2(ax.x < 0.55f ? small.x : copysignf(b.x, x.x), ax.y < 0.55f ? small.y : copysignf(b.y, x.y));
}

// ---- activations of the general kernels: value, f'(z) and f''(z) / f'(z), the last two as functions of the OUTPUT a = f(z) ----
__device__ __forceinline__ float cvf_act(int kind, float z) {
  switch (kind) {
    case CVF_ACT_TANH: return cvf_tanh(z);
    case CVF_ACT_SIGMOID: return 1.0f / (1.0f + expf(-z));
    case CVF_ACT_SOFTPLUS: return z > 20.0f ? z : fmaxf(z, 0.0f) + log1pf(expf(-fabsf(z)));   // torch.nn.Softplus(beta=1, threshold=20)
    case CVF_ACT_ELU: return z > 0.0f ? z : expm1f(z);
    case CVF_ACT_RELU: return fmaxf(z, 0.0f);
    default: return z;
  }
}
__device__ __forceinline__ float cvf_act_d1(int kind, float a) {
  switch (kind) {
    case CVF_ACT_TANH: return fmaf(-a, a, 1.0f);
    case CVF_ACT_SIGMOID: return a * (1.0f - a);
    case CVF_ACT_SOFTPLUS: return a > 20.0f ? 1.0f : -expm1f(-a);   // sigmoid(z) = 1 - exp(-softplus(z))
    case CVF_ACT_ELU: return a > 0.0f ? 1.0f : a + 1.0f;
    case CVF_ACT_RELU: return a > 0.0f ? 1.0f : 0.0f;
    default: return 1.0f;
  }
}
__device__ __forceinline__ float cvf_act_r2(int kind, float a) {
  switch (kind) {
    case CVF_ACT_TANH: return -2.0f * a;
    case CVF_ACT_SIGMOID: return fmaf(-2.0f, a, 1.0f);
    case CVF_ACT_SOFTPLUS: return a > 20.0f ? 0.0f : expf(-a);       // 1 - sigmoid(z)
    case CVF_ACT_ELU: return a > 0.0f ? 0.0f : 1.0f;
    default: return 0.0f;
  }
}

// acc[j][f] = sum_i W[o0+j][i] * in[i][f0+f]      (rows of W clamped to n_out-1 for the tail block)
template <int FPL>
__device__ __forceinline__ void tile_fwd(float (&acc)[4][FPL], const float* __restrict__ W, int ld, int o0, int n_out,
                                         int n_in, const float* __restrict__ in, int FS, int f0) {
#pragma unroll
  for (int j = 0; j < 4; ++j)
#pragma unroll
    for (int f = 0; f < FPL; ++f) acc[j][f] = 0.0f;
  const float* wr[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) wr[j] = W + min(o0 + j, n_out - 1) * ld;
  const float* a = in + f0;
  int i = 0;
#pragma unroll 2
  for (; i + 4 <= n_in; i += 4) {
    float4 wv[4];
    FVec<FPL> av[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) wv[j] = ld4(wr[j] + i);
#pragma unroll
    for (int q = 0; q < 4; ++q) av[q] = FVec<FPL>::ld(a + (i + q) * FS);
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int f = 0; f < FPL; ++f) {
        acc[j][f] = fmaf(wv[j].x, av[0].v[f], acc[j][f]);
        acc[j][f] = fmaf(wv[j].y, av[1].v[f], acc[j][f]);
        acc[j][f] = fmaf(wv[j].z, av[2].v[f], acc[j][f]);
        acc[j][f] = fmaf(wv[j].w, av[3].v[f], acc[j][f]);
      }
  }
  for (; i < n_in; ++i) {
    const FVec<FPL> av = FVec<FPL>::ld(a + i * FS);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float wj = wr[j][i];
#pragma unroll
      for (int f = 0; f < FPL; ++f) acc[j][f] = fmaf(wj, av.v[f], acc[j][f]);
    }
  }
}

// acc[j][f] = sum_o W[o][i0+j] * in[o][f0+f]
template <int FPL>
__device__ __forceinline__ void tile_tr(float (&acc)[4][FPL], const float* __restrict__ W, int ld, int i0, int n_out,
                                        const float* __restrict__ in, int FS, int f0) {
#pragma unroll
  for (int j = 0; j < 4; ++j)
#pragma unroll
    for (int f = 0; f < FPL; ++f) acc[j][f] = 0.0f;
  const float* wp = W + i0;
  const float* a = in + f0;
#pragma unroll 4
  for (int o = 0; o < n_out; ++o) {
    const float4 wv = ld4(wp + o * ld);
    const FVec<FPL> av = FVec<FPL>::ld(a + o * FS);
#pragma unroll
    for (int f = 0; f < FPL; ++f) {
      acc[0][f] = fmaf(wv.x, av.v[f], acc[0][f]);
      acc[1][f] = fmaf(wv.y, av.v[f], acc[1][f]);
      acc[2][f] = fmaf(wv.z, av.v[f], acc[2][f]);
      acc[3][f] = fmaf(wv.w, av.v[f], acc[3][f]);
    }
  }
}

__device__ __forceinline__ float dot4(float4 a, float4 b) { return fmaf(a.x, b.x, fmaf(a.y, b.y, fmaf(a.z, b.z, a.w * b.w))); }

// Outer-product accumulation for one layer:  dW[o][i] += sum_f X1[o][f] Z1[i][f] (+ X2[o][f] Z2[i][f]),
// db[o] += sum_f X1[o][f].  A work item is a 4x4 block of weights (rows 4 ob .. 4 ob+3, columns 4 ib .. 4 ib+3)
// handled by a QUAD of adjacent lanes: lane q of the quad takes the 16-byte frame chunks q, q+4, q+8, ... of every
// row, the quad butterfly-reduces its 16 sums with shuffles, and each lane then adds one row of the block to the
// CTA's fp64 partial vector `part_w` (torch parameter order) with a fire-and-forget reduction: every address has one
// writer per phase and phases are ordered by CTA barriers, so the sum order -- and the result -- is deterministic.  `slot` = item * 4 + q; every lane of a warp must
// call this together (slots past the end compute on clamped rows and write nothing).
__device__ __forceinline__ void outer_quad(int slot, int n_items, int n_out, int n_in, const float* __restrict__ X1,
                                           const float* __restrict__ Z1, const float* __restrict__ X2,
                                           const float* __restrict__ Z2, int FS, int F, double* __restrict__ part_w,
                                           double* __restrict__ part_b) {
  const int q = slot & 3;
  const int item = min(slot >> 2, n_items - 1);
  const bool valid = (slot >> 2) < n_items;
  const int nib = (n_in + 3) >> 2;
  const int ob = item / nib, ib = item - ob * nib;
  int orow[4], irow[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    orow[j] = min(4 * ob + j, n_out - 1);
    irow[j] = min(4 * ib + j, n_in - 1);
  }
  float acc[4][4];
  float bacc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int j = 0; j < 4; ++j)
#pragma unroll
    for (int i = 0; i < 4; ++i) acc[j][i] = 0.0f;
#pragma unroll 2
  for (int f = 4 * q; f < F; f += 16) {
    float4 x[4], z[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      x[j] = ld4(X1 + orow[j] * FS + f);
      z[j] = ld4(Z1 + irow[j] * FS + f);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      bacc[j] += (x[j].x + x[j].y) + (x[j].z + x[j].w);
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[j][i] += dot4(x[j], z[i]);
    }
    if (X2 != nullptr) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        x[j] = ld4(X2 + orow[j] * FS + f);
        z[j] = ld4(Z2 + irow[j] * FS + f);
      }
#pragma unroll
      for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int i = 0; i < 4; ++i) acc[j][i] += dot4(x[j], z[i]);
    }
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      acc[j][i] += __shfl_xor_sync(0xffffffffu, acc[j][i], 1);
      acc[j][i] += __shfl_xor_sync(0xffffffffu, acc[j][i], 2);
    }
    bacc[j] += __shfl_xor_sync(0xffffffffu, bacc[j], 1);
    bacc[j] += __shfl_xor_sync(0xffffffffu, bacc[j], 2);
  }
  if (!valid) return;
  // lane q of the quad owns row 4 ob + q of the block
  float row[4] = {0.f, 0.f, 0.f, 0.f};
  float brow = 0.f;
#pragma unroll
  for (int j = 0; j < 4; ++j)
    if (j == q) {
#pragma unroll
      for (int i = 0; i < 4; ++i) row[i] = acc[j][i];
      brow = bacc[j];
    }
  const int o = 4 * ob + q;
  if (o < n_out) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int ii = 4 * ib + i;
      if (ii < n_in) atomicAdd(&part_w[o * n_in + ii], (double)row[i]);   // result unused -> RED.ADD.F64, no stall
    }
    if (ib == 0 && part_b != nullptr) atomicAdd(&part_b[o], (double)brow);
  }
}

// Run the outer-product items of one layer over the whole CTA.  `slot0` rotates the starting thread so that the
// layers of one phase land on different warps; returns the next rotation.  Warp-uniform control flow.
__device__ __forceinline__ int outer_layer(int slot0, int tid, int nt, int n_out, int n_in, const float* X1, const float* Z1,
                                           const float* X2, const float* Z2, int FS, int F, double* part_w, double* part_b) {
  const int n_items = ((n_out + 3) >> 2) * ((n_in + 3) >> 2);
  const int n_slots = 4 * n_items;
  // thread t handles slots (t - slot0) mod nt, + nt, ...; slot0 is kept a multiple of 32 so warps stay whole
  const int rel = (tid - slot0 + nt) % nt;
  for (int base = 0; base < n_slots; base += nt) {
    const int warp_first = base + (rel & ~31);
    if (warp_first >= n_slots) continue;
    outer_quad(base + rel, n_items, n_out, n_in, X1, Z1, X2, Z2, FS, F, part_w, part_b);
  }
  return (slot0 + ((n_slots + 31) & ~31)) % nt;
}

// deterministic sum of per-CTA fp64 partial vectors: out[i] = sum_b part[b * stride + off + i], i < n
static __global__ void reduce_partials_kernel(const double* __restrict__ part, int n_blocks, int stride, int off, int n,
                                              double* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double s = 0.0;
  for (int b = 0; b < n_blocks; ++b) s += part[(size_t)b * stride + off + i];
  out[i] = s;
}

#endif  // __CUDACC__

}  // namespace cvf
