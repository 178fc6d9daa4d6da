// cvf_eigen_fast.cu -- the EigenFunctionTask step for the common network shape (every hidden layer H wide, H % 4 == 0)
// on Identity or aligned-position pre-processing, organised around what the B200 SM can sustain (profiles/micro/mv_probe.cu):
//
//   * a 128-bit shared-memory load costs two cycles of the SM's shared-memory pipe even when every lane reads the same
//     address, so a weight has to be used at least twice per load; packed FFMA2 (fma.rn.f32x2) halves the issue slots
//     of the FMAs so the loads ride along.  A thread that owns TWO input vectors (two frames, or the primal and the
//     tangent of one frame) and all H outputs reaches ~100 of the 128 fp32 FMA/clk/SM; anything with less reuse is
//     shared-memory bound at <= 64;
//   * therefore every dense layer is evaluated THREAD-PRIVATELY (weights broadcast from shared memory, activations in
//     registers, no barrier between layers), and the only cross-frame work -- the weight-gradient outer products --
//     is a warp-level register-tiled product over the 32 frames the warp has just processed.
//
// Per mini-batch (reference file:line under colvarsfinder/):
//   prep   : Kabsch alignment of every frame (pp_layer, core.py:403), written frame-minor ("SoA": row = coordinate,
//            column = frame) with the 3x3 K^-1 of the alignment Jacobian;  Identity pp: a transpose
//   pass 1 : y = model(r) (core.py:403), u = grad_r y (core.py:424) by a reverse sweep, Dirichlet density
//            D = |J_r^T u|^2 (core.py:426) and the four 3-vectors of the alignment Jacobian applied to u;  2 frames / thread.
//            The hidden activations A_l stay in global memory for pass 2
//   stats  : fp64 batch sums (core.py:406-410,426)
//   pass 2 : d loss / d theta (core.py:517): tangent forward sweep (direction v = J_r J_r^T u, SURVEY 7.3-B; the primal
//            activations are pass 1's), reverse sweep of (G, s) fused, outer products per layer;  1 frame / lane.
//            Bound by the shared-memory pipe (operand loads of the outer products, weight broadcasts), not by the FMA count
#include <math.h>
#include <string.h>

#include "cvf_common.cuh"
#include "cvf_math.cuh"
#include "cvf_tma.cuh"

namespace cvf {
namespace fast {

typedef unsigned long long u64;
constexpr int kRowPad = 36;   // floats per 32-frame row of the pass-2 operand rows (16-byte aligned, bank-group skew 1 per row)

__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
  u64 d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;"
      : "=l"(d)
      : "l"(*reinterpret_cast<u64*>(&a)), "l"(*reinterpret_cast<u64*>(&b)), "l"(*reinterpret_cast<u64*>(&c)));
  return *reinterpret_cast<float2*>(&d);
}
__device__ __forceinline__ float2 dup(float x) { return make_float2(x, x); }
__device__ __forceinline__ float2 lds2(const float* p) { return *reinterpret_cast<const float2*>(p); }
// 4-byte asynchronous global -> shared copy (LDGSTS): no register staging, any number in flight
__device__ __forceinline__ void cp_async4(float* dst, const float* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}
// 16-byte variant (bypasses L1): a 4-byte LDGSTS costs as much issue / shared-memory time as a 16-byte one
__device__ __forceinline__ void cp_async16(float* dst, const float* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait_group() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
// warp-cooperative staging of `nrows` frame-minor row segments (32 frames = 128 B each) into padded shared-memory rows:
// lane -> (row mod 4, 16-byte chunk); `src` points at the first frame of the tile in row 0
__device__ __forceinline__ void stage_rows(float* dst, const float* src, int nrows, long long Bp, int lane) {
  const int c4 = 4 * (lane & 7);
#pragma unroll 4
  for (int r = lane >> 3; r < nrows; r += 4) cp_async16(dst + r * kRowPad + c4, src + (size_t)r * Bp + c4);
}
// the reverse: padded shared-memory rows -> frame-minor global rows, 16 bytes per lane
__device__ __forceinline__ void store_rows(float* dst, const float* src, int nrows, long long Bp, int lane) {
  const int c4 = 4 * (lane & 7);
#pragma unroll 4
  for (int r = lane >> 3; r < nrows; r += 4)
    *reinterpret_cast<float4*>(dst + (size_t)r * Bp + c4) = *reinterpret_cast<const float4*>(src + r * kRowPad + c4);
}
// bounded mbarrier wait: a byte count that does not add up must trap, not hang the GPU
__device__ __forceinline__ void mbar_wait_bounded(uint64_t* bar, uint32_t parity) {
  uint32_t done = 0;
  for (int spin = 0; spin < (1 << 24); ++spin) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    if (done) return;
  }
  __trap();
}
__device__ __forceinline__ void prefetch_l2_line(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
// the 128-byte line at p (aligned) will not be read again: L2 may drop it without writing it back to HBM
__device__ __forceinline__ void discard_l2_line(const void* p) { asm volatile("discard.global.L2 [%0], 128;" ::"l"(p) : "memory"); }
// warp prefetch of `nrows` row segments (one 128-byte line each: 32 frames of a frame-minor row)
__device__ __forceinline__ void prefetch_rows(const float* base, int nrows, long long Bp, int lane) {
  for (int r = lane; r < nrows; r += 32) prefetch_l2_line(base + (size_t)r * Bp);
}

constexpr int kP1Frames = 512, kP1Threads = 256;
// columns of dW_1 formed per pass over the warp's 32 frames (pass 2): 24, or 28 when that divides the padded input width
// (C4: 84 = 3 x 28, so that three networks' totals fit the 256 tensor-memory columns of a warp)
__host__ __device__ constexpr int dw1_chunk_of(int drp) { return drp % 28 == 0 ? 28 : 24; }
constexpr int kP2MaxWarps = 8, kP2MinWarps = 4;

// Shared-memory image of one network (floats; every block 16-byte aligned because H % 4 == 0 and d_rp % 12 == 0):
//   W1T [d_rp][H] (k-major)  b1 [H]  { WlT [H][H]  bl [H] } l=2..NH   Wout [H]  bout [4]   { Wl [H][H] natural } l=2..NH
//   -- pass 2 reads up to here --   W1 [H][d_rp] natural
template <int H, int NH>
struct Img {
  __host__ __device__ static int b1(int drp) { return drp * H; }
  __host__ __device__ static int wt(int drp, int l) { return drp * H + H + (l - 2) * (H * H + H); }   // l = 2..NH
  __host__ __device__ static int bl(int drp, int l) { return wt(drp, l) + H * H; }
  __host__ __device__ static int wout(int drp) { return drp * H + H + (NH - 1) * (H * H + H); }
  __host__ __device__ static int bout(int drp) { return wout(drp) + H; }
  __host__ __device__ static int wn(int drp, int l) { return bout(drp) + 4 + (l - 2) * H * H; }        // l = 2..NH
  __host__ __device__ static int p2_floats(int drp) { return bout(drp) + 4 + (NH - 1) * H * H; }
  __host__ __device__ static int w1n(int drp) { return p2_floats(drp); }
  __host__ __device__ static int floats(int drp) { return p2_floats(drp) + H * drp; }
};

struct FastPlan {
  int k, d_r, d_rp, kind;        // kind 0: identity on [B,d_r];  1: aligned positions of all n_atoms atoms (d_r = 3 n_atoms);
                                 // 2: feature map (position / bond / angle / dihedral records) on the raw frame, no alignment
  int n_atoms, n_align;
  int n_used, n_feat, n_st, n_adj;   // kind 2: atoms the features read, records, bounds on the stencil rows per frame and
                                     // on the (atom, record) pairs (the actual counts are in the table header)
  int n_self, n_shared;              // kind 2: self rows the builder may hand out; bound on the atoms in the CSR
  int tile_rows;                 // rows of the pass-1 frame tile: d_rp for kind 1 (the Jacobian sums read whole atoms), else d_r
  const int32_t* used_atoms;     // kind 2: [n_used] atom index
  const int32_t* feat;           // kind 2: [n_feat][5] type + positions in used_atoms
  int* tab;                      // kind 2: tables built by pack_kernel (layout: tab_* below)
  float* ST;                     // kind 2: [n_st][Bp] gradient stencils of every record (prep -> jjt)
  int img_floats, img2_floats, geo_floats, n_params;
  int gw_off[kMaxLayers], gb_off[kMaxLayers];   // torch-order offsets inside one network's parameters
  long long B, Bp;
  const int32_t* align_idx;      // [n_align] atom index
  const float* ref;              // [n_align][3] centred
  const float* diag;             // kind 0: [d_r] or null
  float* img;                    // [k][img_floats] followed by geo [geo_floats]
  float* Y;                      // [d_rp][Bp]
  float* Kinv;                   // [6][Bp]
  float* A;                      // [k][NH * H][Bp] hidden activations A_l of pass 1, read back by pass 2 (which only propagates tangents)
  float* U;                      // [k][d_rp][Bp]
  float* JQ;                     // [k][12][Bp]   gm, q, dc, om
  float* Dq;                     // [k][Bp]
  float* Ys;                     // [k][Bp]
  double* part;                  // per-CTA / per-warp partial sums
};

// geo block (floats): kind 1: refA [d_rp] (reference position of the atom a coordinate belongs to, 0 if not aligned),
// inA [d_rp] (1 if aligned), Iref [6] (sum |ref|^2 I - ref ref^T), nA, 1/nA;   kind 0: diag [d_rp], unused [d_rp], ...
__host__ __device__ inline int geo_floats_of(int drp) { return 2 * drp + 8; }

// ---- kind 2 tables (ints, built on the device by pack_kernel because the record list lives in device memory):
//   header    [4]            pairs in adj, atoms in the CSR, stencil rows per frame, 1 if the tables do not fit the host's bounds
//   finfo     [n_feat][12]   type | self mask << 8, first output row, first stencil row, self row or -1,
//                            atom index of each of up to 4 atoms, position in used_atoms of each
//   adj_start [n_used + 1]   CSR over the atoms that need one (padded to a multiple of 4 ints)
//   catom     [n_used]       position in used_atoms of CSR atom c (padded)
//   adj       [n_adj][4]     (kind, byte offset of the output row, byte offset of the stencil row, 0) of every (atom, record)
//                            pair, offsets inside 32-frame tiles (row = 128 bytes)
//   rstart    [n_feat + 1]   the same pairs grouped by record (padded)
//   radj      [n_adj][4]     (kind, byte offset of the atom's first row in the per-atom gradient block, byte offset of the stencil
//                            row, 0); kind 0 = position record (its three outputs are the atom's gradient itself)
//   scratch   [2 n_used]     of the builder
// Stencil rows of a record (floats per frame, written by prep_feat_kernel): bond 3 (unit vector a -> b), angle 6 (d cos / d a,
// d cos / d c), dihedral 10 (d phi / d p0, d phi / d p3, p, q, cos, sin; d phi / d p1 = (-1-p) g0 + q g3,
// d phi / d p2 = p g0 + (-1-q) g3 -- cvf_dihedral in cvf_math.cuh), position 0; then one "self" row for a record with atoms
// that no other record reads: m = sum over those atoms of stencil . (a stencil), so that their whole contribution is
// vhat_f += m u_f, D += m u_f^2 and they stay out of the CSR.  jjt_kernel appends 5 constant rows (0,0,1,0,0) to its staged
// tile: a position record is three pairs whose "stencils" are the unit vectors found there.
// adj kinds: 1 stencil times the sign in the fourth field, 3 angle apex -(s + s'), 4 dihedral p1, 5 dihedral p2.
constexpr int kTabHdr = 4, kFinfoInts = 12;
__host__ __device__ inline int tab_finfo() { return kTabHdr; }
__host__ __device__ inline int tab_adj_start(int n_feat) { return kTabHdr + kFinfoInts * n_feat; }
__host__ __device__ inline int tab_catom(int n_feat, int n_used) { return tab_adj_start(n_feat) + ((n_used + 1 + 3) & ~3); }
__host__ __device__ inline int tab_adj(int n_feat, int n_used) { return tab_catom(n_feat, n_used) + ((n_used + 3) & ~3); }
__host__ __device__ inline int tab_rstart(int n_feat, int n_used, int n_adj) { return tab_adj(n_feat, n_used) + 4 * (n_adj > 0 ? n_adj : 1); }
__host__ __device__ inline int tab_radj(int n_feat, int n_used, int n_adj) { return tab_rstart(n_feat, n_used, n_adj) + ((n_feat + 1 + 3) & ~3); }
__host__ __device__ inline int tab_scratch(int n_feat, int n_used, int n_adj) { return tab_radj(n_feat, n_used, n_adj) + 4 * (n_adj > 0 ? n_adj : 1); }
__host__ __device__ inline int tab_ints(int n_feat, int n_used, int n_adj) { return tab_scratch(n_feat, n_used, n_adj) + 2 * n_used; }
constexpr int kStBond = 3, kStAngle = 6, kStDihedral = 10, kStConstRows = 5;
__host__ __device__ inline int feat_atoms(int type) {
  return type == CVF_FEAT_POSITION ? 1 : type == CVF_FEAT_BOND ? 2 : type == CVF_FEAT_ANGLE ? 3 : 4;
}
__host__ __device__ inline int feat_rows(int type) {
  return type == CVF_FEAT_BOND ? kStBond : type == CVF_FEAT_ANGLE ? kStAngle : type == CVF_FEAT_DIHEDRAL ? kStDihedral : 0;
}

__device__ void build_feature_tables(const FastPlan& P) {
  int* hdr = P.tab;
  int* finfo = P.tab + tab_finfo();
  int* start = P.tab + tab_adj_start(P.n_feat);
  int* catom = P.tab + tab_catom(P.n_feat, P.n_used);
  int* adj = P.tab + tab_adj(P.n_feat, P.n_used);
  int* reads = P.tab + tab_scratch(P.n_feat, P.n_used, P.n_adj);   // records reading each used atom (a position record counts 2)
  int* slot = reads + P.n_used;                                    // pairs of the atom, then its fill cursor
  for (int a = 0; a < P.n_used; ++a) reads[a] = slot[a] = 0;
  for (int i = 0; i < P.n_feat; ++i) {
    const int* rec = P.feat + 5 * i;
    for (int j = 0; j < feat_atoms(rec[0]); ++j) reads[rec[1 + j]] += rec[0] == CVF_FEAT_POSITION ? 2 : 1;
  }
  int fo = 0, sr = 0, n_self = 0;
  for (int i = 0; i < P.n_feat; ++i) {
    const int* rec = P.feat + 5 * i;
    const int type = rec[0], na = feat_atoms(type);
    int mask = 0;
    if (type != CVF_FEAT_POSITION)
      for (int j = 0; j < na; ++j)
        if (reads[rec[1 + j]] == 1) mask |= 1 << j;
    int self_row = -1;
    if (mask != 0 && n_self < P.n_self) self_row = sr + feat_rows(type), ++n_self;
    else mask = 0;
    int* fi = finfo + kFinfoInts * i;
    fi[0] = type | (mask << 8), fi[1] = fo, fi[2] = sr, fi[3] = self_row;
    for (int j = 0; j < 4; ++j) fi[4 + j] = j < na ? P.used_atoms[rec[1 + j]] : 0, fi[8 + j] = j < na ? rec[1 + j] : 0;
    for (int j = 0; j < na; ++j)
      if (!((mask >> j) & 1)) slot[rec[1 + j]] += type == CVF_FEAT_POSITION ? 3 : 1;
    fo += type == CVF_FEAT_POSITION ? 3 : type == CVF_FEAT_DIHEDRAL ? 2 : 1;
    sr += feat_rows(type) + (self_row >= 0 ? 1 : 0);
  }
  int nc = 0, acc = 0;
  for (int a = 0; a < P.n_used; ++a)
    if (slot[a] > 0) {
      const int cnt = slot[a];
      catom[nc] = a, start[nc] = acc, slot[a] = acc, acc += cnt, ++nc;
    }
  start[nc] = acc;
  hdr[0] = acc, hdr[1] = nc, hdr[2] = sr, hdr[3] = (nc > P.n_shared || sr > P.n_st || acc > P.n_adj || fo != P.d_r) ? 1 : 0;
  if (hdr[3]) {   // the descriptor's sizing fields do not cover this record list: jjt_kernel poisons its output
    hdr[0] = hdr[1] = 0;
    return;
  }
  int* rstart = P.tab + tab_rstart(P.n_feat, P.n_used, P.n_adj);
  int* radj = P.tab + tab_radj(P.n_feat, P.n_used, P.n_adj);
  for (int a = 0; a < P.n_used; ++a) reads[a] = -1;          // reuse: CSR index of the used atom
  for (int c = 0; c < nc; ++c) reads[catom[c]] = c;
  {
    int racc = 0;
    for (int i = 0; i < P.n_feat; ++i) {
      const int* rec = P.feat + 5 * i;
      const int* fi = finfo + kFinfoInts * i;
      const int type = fi[0] & 0xff, mask = fi[0] >> 8, sr_i = fi[2];
      rstart[i] = racc;
      for (int j = 0; j < feat_atoms(type); ++j) {
        if ((mask >> j) & 1) continue;
        int kind, srj = sr_i;
        if (type == CVF_FEAT_POSITION) kind = 0;
        else if (type == CVF_FEAT_BOND) kind = j == 0 ? 2 : 1;
        else if (type == CVF_FEAT_ANGLE) kind = j == 1 ? 3 : 1, srj = sr_i + (j == 2 ? 3 : 0);
        else kind = j == 0 || j == 3 ? 1 : (j == 1 ? 4 : 5), srj = sr_i + (j == 3 ? 3 : 0);
        int* e = radj + 4 * racc++;
        e[0] = kind == 2 ? 1 : kind, e[1] = 128 * 3 * reads[rec[1 + j]], e[2] = 128 * srj, e[3] = __float_as_int(kind == 2 ? -1.0f : 1.0f);
      }
    }
    rstart[P.n_feat] = racc;
  }
  for (int i = 0; i < P.n_feat; ++i) {
    const int* rec = P.feat + 5 * i;
    const int* fi = finfo + kFinfoInts * i;
    const int type = fi[0] & 0xff, mask = fi[0] >> 8, fo_i = fi[1], sr_i = fi[2];
    if (type == CVF_FEAT_POSITION) {
      for (int c = 0; c < 3; ++c) {
        int* e = adj + 4 * slot[rec[1]]++;
        e[0] = 1, e[1] = 128 * (fo_i + c), e[2] = 128 * (sr + 2 - c), e[3] = __float_as_int(1.0f);
      }
      continue;
    }
    for (int j = 0; j < feat_atoms(type); ++j) {
      if ((mask >> j) & 1) continue;
      int kind, srj = sr_i;
      if (type == CVF_FEAT_BOND) kind = j == 0 ? 2 : 1;
      else if (type == CVF_FEAT_ANGLE) kind = j == 1 ? 3 : 1, srj = sr_i + (j == 2 ? 3 : 0);
      else kind = j == 0 || j == 3 ? 1 : (j == 1 ? 4 : 5), srj = sr_i + (j == 3 ? 3 : 0);
      int* e = adj + 4 * slot[rec[1 + j]]++;
      e[0] = kind == 2 ? 1 : kind, e[1] = 128 * fo_i, e[2] = 128 * srj, e[3] = __float_as_int(kind == 2 ? -1.0f : 1.0f);
    }
  }
}

// ------------------------------------------------------------------------------------------------ pack
template <int H, int NH>
__global__ void pack_kernel(const FastPlan P, const float* __restrict__ params) {
  const int drp = P.d_rp, d_r = P.d_r;
  typedef Img<H, NH> I;
  if (blockIdx.x == (unsigned)P.k + 1) {   // kind 2: record / adjacency tables
    if (threadIdx.x == 0) build_feature_tables(P);
    return;
  }
  if (blockIdx.x == (unsigned)P.k) {   // geometry block
    float* g = P.img + (size_t)P.k * P.img_floats;
    for (int i = threadIdx.x; i < P.geo_floats; i += blockDim.x) g[i] = 0.0f;
    __syncthreads();
    if (P.kind == 2) {
      for (int i = threadIdx.x; i < d_r; i += blockDim.x) g[i] = 1.0f;   // diag_coeff is applied by jjt_kernel
    } else if (P.kind == 0) {
      for (int i = threadIdx.x; i < d_r; i += blockDim.x) g[i] = P.diag ? P.diag[i] : 1.0f;
    } else {
      for (int j = threadIdx.x; j < P.n_align; j += blockDim.x) {
        const int a = P.align_idx[j];
        for (int c = 0; c < 3; ++c) g[3 * a + c] = P.ref[3 * j + c], g[drp + 3 * a + c] = 1.0f;
      }
      if (threadIdx.x == 0) {
        double xx = 0, xy = 0, xz = 0, yy = 0, yz = 0, zz = 0;
        for (int j = 0; j < P.n_align; ++j) {
          const double x = P.ref[3 * j], y = P.ref[3 * j + 1], z = P.ref[3 * j + 2], n2 = x * x + y * y + z * z;
          xx += n2 - x * x, yy += n2 - y * y, zz += n2 - z * z, xy -= x * y, xz -= x * z, yz -= y * z;
        }
        float* t = g + 2 * drp;
        t[0] = (float)xx, t[1] = (float)xy, t[2] = (float)xz, t[3] = (float)yy, t[4] = (float)yz, t[5] = (float)zz;
        t[6] = (float)P.n_align, t[7] = 1.0f / (float)P.n_align;
      }
    }
    return;
  }
  const float* src = params + (size_t)blockIdx.x * P.n_params;
  float* dst = P.img + (size_t)blockIdx.x * P.img_floats;
  for (int i = threadIdx.x; i < P.img_floats; i += blockDim.x) {
    float v = 0.0f;
    if (i < I::b1(drp)) {
      const int kk = i / H, o = i - kk * H;
      if (kk < d_r) v = src[P.gw_off[0] + o * d_r + kk];
    } else if (i < I::b1(drp) + H) {
      v = src[P.gb_off[0] + i - I::b1(drp)];
    } else if (i < I::wout(drp)) {
      const int r = i - (I::b1(drp) + H), l = 2 + r / (H * H + H), q = r - (l - 2) * (H * H + H);
      if (q < H * H) {
        const int kk = q / H, o = q - kk * H;
        v = src[P.gw_off[l - 1] + o * H + kk];
      } else {
        v = src[P.gb_off[l - 1] + q - H * H];
      }
    } else if (i < I::bout(drp)) {
      v = src[P.gw_off[NH] + i - I::wout(drp)];
    } else if (i < I::bout(drp) + 4) {
      if (i == I::bout(drp)) v = src[P.gb_off[NH]];
    } else if (i < I::p2_floats(drp)) {
      const int r = i - (I::bout(drp) + 4), l = 2 + r / (H * H), q = r - (l - 2) * H * H;
      v = src[P.gw_off[l - 1] + q];
    } else {
      const int r = i - I::w1n(drp), o = r / drp, kk = r - o * drp;
      if (kk < d_r) v = src[P.gw_off[0] + o * d_r + kk];
    }
    dst[i] = v;
  }
}

// ------------------------------------------------------------------------------------------------ prep
// kind 1: Kabsch per frame (thread per frame on a coalesced shared-memory tile), frame-minor output.
__global__ void __launch_bounds__(128, 6) prep_align_kernel(const FastPlan P, const float* __restrict__ x, int bulk) {
  extern __shared__ __align__(128) float st[];
  __shared__ __align__(8) uint64_t bar;
  const int tid = threadIdx.x;
  // bulk (TMA): a full tile of 128 raw frames is one contiguous block of global memory (128 * 12 N bytes, a multiple of 16) and
  // arrives by ONE cp.async.bulk into rows of stride 3N; otherwise (tail tile, unaligned x) cooperative loads into rows of odd stride
  const int fl = 3 * P.n_atoms, S = bulk ? fl : (fl | 1);
  float* kin = st + 128 * (fl | 1);           // [6][128]
  // the alignment set as shared-memory tables (offset of the atom inside a frame, reference position in double): the per-atom
  // loops then cost one broadcast LDS where they used to load, scale and convert
  double* s_ref = reinterpret_cast<double*>(kin + 6 * 128);   // [n_align][3]; 512 (fl|1) + 3072 bytes into the buffer: 8-byte aligned
  int* s_off = reinterpret_cast<int*>(s_ref + 3 * P.n_align + 3);                       // [n_align]
  for (int a = tid; a < P.n_align; a += 128) {
    s_off[a] = 3 * P.align_idx[a];
    s_ref[3 * a] = P.ref[3 * a], s_ref[3 * a + 1] = P.ref[3 * a + 1], s_ref[3 * a + 2] = P.ref[3 * a + 2];
  }
  if (tid < 3) {   // sum of the reference positions (zero up to the rounding of the centred reference), fixed order
    double t = 0.0;
    for (int a = 0; a < P.n_align; ++a) t += (double)P.ref[3 * a + tid];
    s_ref[3 * P.n_align + tid] = t;
  }
  if (tid == 0) {
    mbar_init(&bar, 1);
    fence_barrier_init();
  }
  __syncthreads();
  const int n_align = P.n_align, n_atoms = P.n_atoms;
  uint32_t phase = 0;
  const long long n_tiles = P.Bp / 128;
  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const long long f0 = tile * 128;
    if (bulk && f0 + 128 <= P.B) {
      if (tid == 0) {
        const uint32_t bytes = (uint32_t)(128 * fl * sizeof(float));
        fence_proxy_async();   // the previous tile's ordinary reads / writes of the buffer precede the copy
        mbar_expect_tx(&bar, bytes);
        bulk_g2s(st, x + (size_t)f0 * fl, bytes, &bar);
      }
      mbar_wait_bounded(&bar, phase);
      phase ^= 1;
    } else {
      for (int i = tid; i < 128 * fl; i += 128) {
        const int f = i / fl;
        const long long fr = min(f0 + f, P.B - 1);   // padding frames repeat the last frame (their weight is 0)
        st[f * S + (i - f * fl)] = __ldg(x + (size_t)fr * fl + (i - f * fl));
      }
      __syncthreads();
    }
    {
      float* fr = st + tid * S;
      // ONE sweep over the alignment atoms: every coordinate becomes a double once (the float <-> double conversions are what
      // the fp64 pipe spends most of its time on here) and feeds both the centroid and H = sum x (x) ref; the centroid leaves H
      // as  (x_A - c)^T ref = sum x (x) ref - c (x) sum ref  (sum ref is the rounding residue of the centred reference)
      double cx = 0, cy = 0, cz = 0;
      double Hm[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll 2
      for (int a = 0; a < n_align; ++a) {
        const float* p = fr + s_off[a];
        const double px = p[0], py = p[1], pz = p[2];
        const double rx = s_ref[3 * a], ry = s_ref[3 * a + 1], rz = s_ref[3 * a + 2];
        cx += px, cy += py, cz += pz;
        Hm[0] = fma(px, rx, Hm[0]), Hm[1] = fma(px, ry, Hm[1]), Hm[2] = fma(px, rz, Hm[2]);
        Hm[3] = fma(py, rx, Hm[3]), Hm[4] = fma(py, ry, Hm[4]), Hm[5] = fma(py, rz, Hm[5]);
        Hm[6] = fma(pz, rx, Hm[6]), Hm[7] = fma(pz, ry, Hm[7]), Hm[8] = fma(pz, rz, Hm[8]);
      }
      const double inv = 1.0 / n_align;
      cx *= inv, cy *= inv, cz *= inv;
      {
        const double sx = s_ref[3 * n_align], sy = s_ref[3 * n_align + 1], sz = s_ref[3 * n_align + 2];
        Hm[0] = fma(-cx, sx, Hm[0]), Hm[1] = fma(-cx, sy, Hm[1]), Hm[2] = fma(-cx, sz, Hm[2]);
        Hm[3] = fma(-cy, sx, Hm[3]), Hm[4] = fma(-cy, sy, Hm[4]), Hm[5] = fma(-cy, sz, Hm[5]);
        Hm[6] = fma(-cz, sx, Hm[6]), Hm[7] = fma(-cz, sy, Hm[7]), Hm[8] = fma(-cz, sz, Hm[8]);
      }
      float R[9], Ki[6];
      double Rd[9];
      cvf_rotation(Hm, R, Ki, Rd);
      const double tx = cx * Rd[0] + cy * Rd[3] + cz * Rd[6], ty = cx * Rd[1] + cy * Rd[4] + cz * Rd[7],
                   tz = cx * Rd[2] + cy * Rd[5] + cz * Rd[8];
#pragma unroll 2
      for (int a = 0; a < n_atoms; ++a) {
        float* p = fr + 3 * a;
        const cvf_v3 q = cvf_transform_t(p[0], p[1], p[2], tx, ty, tz, Rd);
        p[0] = q.x, p[1] = q.y, p[2] = q.z;
      }
#pragma unroll
      for (int i = 0; i < 6; ++i) kin[i * 128 + tid] = Ki[i];
    }
    __syncthreads();
    for (int r = 0; r < P.d_rp; ++r) P.Y[(size_t)r * P.Bp + f0 + tid] = r < fl ? st[tid * S + r] : 0.0f;
#pragma unroll
    for (int i = 0; i < 6; ++i) P.Kinv[(size_t)i * P.Bp + f0 + tid] = kin[i * 128 + tid];
    __syncthreads();
  }
}

// kind 0: [B][d] -> [d_rp][Bp]
__global__ void __launch_bounds__(256) prep_transpose_kernel(const FastPlan P, const float* __restrict__ x) {
  const long long n = P.Bp;
  for (long long f = (long long)blockIdx.x * blockDim.x + threadIdx.x; f < n; f += (long long)gridDim.x * blockDim.x) {
    const long long fr = min(f, P.B - 1);
    for (int r = 0; r < P.d_rp; ++r) P.Y[(size_t)r * P.Bp + f] = r < P.d_r ? __ldg(x + (size_t)fr * P.d_r + r) : 0.0f;
  }
}

// kind 2: feature values and their gradient stencils from the raw frame (the pp_layer of core.py:403 without alignment:
// _ops.py drops the Kabsch step when every record is invariant under it).  A CTA holds up to four groups of four warps; a group
// owns one staging buffer of 32 consecutive frames -- one contiguous block of global memory, fetched by a single 1-D bulk
// asynchronous copy (TMA) that completes on the group's mbarrier -- and then lane = frame, the group's warps taking every
// fourth record.  Groups run out of phase, so the copies of some overlap the arithmetic and the stores of the others.
// bulk = 0 (x not 16-byte aligned, or a frame length that would put every lane in the same bank): cooperative loads into
// rows of odd stride.
__global__ void __launch_bounds__(512) prep_feat_kernel(const FastPlan P, const float* __restrict__ x, int bulk) {
  extern __shared__ __align__(16) float st[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, grp = warp >> 2, wg = warp & 3, ng = blockDim.x >> 7;
  const int fl = 3 * P.n_atoms, S = bulk ? fl : (fl | 1);
  uint64_t* bars = reinterpret_cast<uint64_t*>(st);
  int4* finfo = reinterpret_cast<int4*>(st + 32);
  float* my = st + 32 + kFinfoInts * P.n_feat + (size_t)grp * ((32 * S + 3) & ~3);
  if (tid == 0) {
    for (int g = 0; g < ng; ++g) mbar_init(&bars[g], 1);
    fence_barrier_init();
  }
  if (P.tab[3] != 0) return;   // tables rejected by the builder (see jjt_kernel)
  for (int i = tid; i < 3 * P.n_feat; i += blockDim.x) finfo[i] = reinterpret_cast<const int4*>(P.tab + tab_finfo())[i];
  __syncthreads();
  uint32_t phase = 0;
  const long long n_tiles = P.Bp / 32;
  for (long long t = (long long)blockIdx.x * ng + grp; t < n_tiles; t += (long long)gridDim.x * ng) {
    const long long f0 = t * 32;
    if (bulk && f0 + 32 <= P.B) {
      if (wg == 0 && lane == 0) {
        const uint32_t bytes = (uint32_t)(32 * fl * sizeof(float));
        mbar_expect_tx(&bars[grp], bytes);
        bulk_g2s(my, x + (size_t)f0 * fl, bytes, &bars[grp]);
      }
      mbar_wait(&bars[grp], phase);
      phase ^= 1;
    } else {
      for (int i = wg * 32 + lane; i < 32 * fl; i += 128) {
        const int f = i / fl, j = i - f * fl;
        const long long fr = min(f0 + f, P.B - 1);   // padding frames repeat the last frame (their weight is 0)
        my[f * S + j] = __ldg(x + (size_t)fr * fl + j);
      }
      named_barrier(1 + grp, 128);
    }
    const float* fr = my + lane * S;
    float* Yt = P.Y + f0 + lane;
    float* St = P.ST + f0 + lane;
    for (int i = wg; i < P.n_feat; i += 4) {
      const int4 fa = finfo[3 * i], fb = finfo[3 * i + 1], fc = finfo[3 * i + 2];
      const int type = fa.x & 0xff, mask = fa.x >> 8;
      float* yo = Yt + (size_t)fa.y * P.Bp;
      float* so = St + (size_t)fa.z * P.Bp;
      // self term of an atom that only this record reads: stencil . (a stencil)
      auto self = [&](int j, int up, cvf_v3 sv) -> float {
        if (!((mask >> j) & 1)) return 0.0f;
        if (!P.diag) return dot(sv, sv);
        return __ldg(P.diag + 3 * up) * sv.x * sv.x + __ldg(P.diag + 3 * up + 1) * sv.y * sv.y + __ldg(P.diag + 3 * up + 2) * sv.z * sv.z;
      };
      const cvf_v3 p0 = v3(fr[3 * fb.x], fr[3 * fb.x + 1], fr[3 * fb.x + 2]);
      if (type == CVF_FEAT_POSITION) {
        yo[0] = p0.x, yo[P.Bp] = p0.y, yo[2 * P.Bp] = p0.z;
        continue;
      }
      float* mo = St + (size_t)fa.w * P.Bp;   // self row (only written when fa.w >= 0)
      const cvf_v3 p1 = v3(fr[3 * fb.y], fr[3 * fb.y + 1], fr[3 * fb.y + 2]);
      if (type == CVF_FEAT_BOND) {
        cvf_v3 g;
        yo[0] = cvf_bond(p0, p1, g);
        so[0] = g.x, so[P.Bp] = g.y, so[2 * P.Bp] = g.z;
        if (fa.w >= 0) mo[0] = self(0, fc.x, g) + self(1, fc.y, g);
        continue;
      }
      const cvf_v3 p2 = v3(fr[3 * fb.z], fr[3 * fb.z + 1], fr[3 * fb.z + 2]);
      if (type == CVF_FEAT_ANGLE) {
        cvf_v3 ga, gc;
        yo[0] = cvf_angle(p0, p1, p2, ga, gc);
        so[0] = ga.x, so[P.Bp] = ga.y, so[2 * P.Bp] = ga.z, so[3 * P.Bp] = gc.x, so[4 * P.Bp] = gc.y, so[5 * P.Bp] = gc.z;
        if (fa.w >= 0) mo[0] = self(0, fc.x, ga) + self(1, fc.y, ga + gc) + self(2, fc.z, gc);
        continue;
      }
      const cvf_v3 p3 = v3(fr[3 * fb.w], fr[3 * fb.w + 1], fr[3 * fb.w + 2]);
      float cs, sn, pc, qc;
      cvf_v3 g0, g3;
      cvf_dihedral_compact(p0, p1, p2, p3, cs, sn, g0, g3, pc, qc);
      yo[0] = cs, yo[P.Bp] = sn;
      so[0] = g0.x, so[P.Bp] = g0.y, so[2 * P.Bp] = g0.z, so[3 * P.Bp] = g3.x, so[4 * P.Bp] = g3.y, so[5 * P.Bp] = g3.z;
      so[6 * P.Bp] = pc, so[7 * P.Bp] = qc, so[8 * P.Bp] = cs, so[9 * P.Bp] = sn;
      if (fa.w >= 0)
        mo[0] = self(0, fc.x, g0) + self(1, fc.y, (-1.0f - pc) * g0 + qc * g3) + self(2, fc.z, pc * g0 + (-1.0f - qc) * g3) +
                self(3, fc.w, g3);
    }
    named_barrier(1 + grp, 128);   // every warp of the group has finished reading the buffer
  }
}

// kind 2, between pass 1 and the batch sums: for every network, vhat = J diag(a) J^T u (the tangent direction of pass 2,
// SURVEY 7.3-B) and the Dirichlet density D = u^T J diag(a) J^T u (core.py:426), where J = d r / d x is assembled from the
// stencils prep_feat_kernel left.  One CTA per 32-frame tile (lane = frame); the stencil tile is staged once and shared by
// the networks, and W warps work on each network.  Atoms that a single record reads are folded into that record's self row by
// prep_feat_kernel (vhat_f += m u_f, D += m u_f^2).  For the others:
//   phase 1, atom-major (a warp takes every W-th atom): g = sum over the atom's records of u_f * stencil, D += a |g|^2, and a g
//            goes to the network's per-atom gradient rows;
//   phase 2, record-major (a warp takes every W-th record): vhat_f = m u_f + sum over the record's atoms of stencil . (a g),
//            written in place of u_f.
// Every sum has one owner and a fixed order: the result is deterministic.  vhat replaces u in P.U.
struct JjtLoad {
  cvf_v3 s0, s1;
  float p, q;
};
__device__ __forceinline__ void jjt_issue(JjtLoad& L, const int4 en, const char* STl) {
  const float* sp = reinterpret_cast<const float*>(STl + en.z);
  L.s0 = v3(sp[0], sp[32], sp[64]);
  if (en.x >= 3) {
    L.s1 = v3(sp[96], sp[128], sp[160]);
    if (en.x >= 4) L.p = sp[192], L.q = sp[224];
  }
}
// stencil of kinds >= 3 (kind 1 is s0 times the pair's sign, applied by the caller to the scalar factor)
__device__ __forceinline__ cvf_v3 jjt_combine(const JjtLoad& L, int kind) {
  float c0 = -1.0f, c1 = -1.0f;
  if (kind == 4) c0 = -1.0f - L.p, c1 = L.q;
  if (kind == 5) c0 = L.p, c1 = -1.0f - L.q;
  return c0 * L.s0 + c1 * L.s1;
}

__global__ void __launch_bounds__(384, 2) jjt_kernel(const FastPlan P, int W) {
  extern __shared__ __align__(16) float sm[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nt = blockDim.x;
  const int n = warp / W, q = warp - n * W;   // network, warp of the network
  const int d_r = P.d_r, n_used = P.n_used, n_feat = P.n_feat;
  const bool poisoned = P.tab[3] != 0;   // the record list does not fit the descriptor's sizing fields: D = NaN, nothing else
  const int n_adj = P.tab[0], nc = P.tab[1], n_st = poisoned ? 0 : P.tab[2];   // actual counts (<= the host-side bounds)
  const int adj_cap = P.n_adj > 0 ? P.n_adj : 1;
  int* s_start = reinterpret_cast<int*>(sm);                          // [n_shared + 1]
  int* s_catom = s_start + ((P.n_shared + 1 + 3) & ~3);               // [n_shared]
  int* s_rstart = s_catom + ((P.n_shared + 3) & ~3);                  // [n_feat + 1]
  int4* s_adj = reinterpret_cast<int4*>(s_rstart + ((n_feat + 1 + 3) & ~3));
  int4* s_radj = s_adj + adj_cap;
  int4* s_fi = s_radj + adj_cap;
  float* s_dg = reinterpret_cast<float*>(s_fi + n_feat);             // [3 n_shared] diag_coeff of the CSR atoms
  float* STs = s_dg + ((3 * P.n_shared + 3) & ~3);
  const int net_floats = (d_r + 3 * P.n_shared + W) * 32;
  float* Su = STs + (size_t)(P.n_st + kStConstRows) * 32 + (size_t)n * net_floats;   // [d_r][32]  u, then vhat
  float* Sg = Su + (size_t)d_r * 32;                                                  // [3 nc][32] a g of every CSR atom
  float* Sd = Sg + (size_t)3 * P.n_shared * 32;                                       // [W][32]    partial D
  {
    const int* g_start = P.tab + tab_adj_start(n_feat);
    const int* g_catom = P.tab + tab_catom(n_feat, n_used);
    const int* g_rstart = P.tab + tab_rstart(n_feat, n_used, P.n_adj);
    const int4* g_adj = reinterpret_cast<const int4*>(P.tab + tab_adj(n_feat, n_used));
    const int4* g_radj = reinterpret_cast<const int4*>(P.tab + tab_radj(n_feat, n_used, P.n_adj));
    const int4* g_fi = reinterpret_cast<const int4*>(P.tab + tab_finfo());
    for (int i = tid; i <= nc; i += nt) s_start[i] = g_start[i];
    for (int i = tid; i < nc; i += nt) {
      const int a = g_catom[i];
      s_catom[i] = a;
      for (int c = 0; c < 3; ++c) s_dg[3 * i + c] = P.diag ? P.diag[3 * a + c] : 1.0f;
    }
    for (int i = tid; i <= n_feat; i += nt) s_rstart[i] = poisoned ? 0 : g_rstart[i];
    for (int i = tid; i < n_adj; i += nt) s_adj[i] = g_adj[i], s_radj[i] = g_radj[i];
    for (int i = tid; i < n_feat; i += nt) {
      const int4 v = g_fi[3 * i];
      s_fi[i] = make_int4(v.x & 0xff, 128 * v.y, 128 * v.z, v.w >= 0 ? 128 * v.w : -1);
    }
    for (int i = tid; i < kStConstRows * 32; i += nt) STs[n_st * 32 + i] = (i >> 5) == 2 ? 1.0f : 0.0f;
  }
  const int c4 = 4 * (lane & 7);
  const char* STl = reinterpret_cast<const char*>(STs + lane);
  char* Sul = reinterpret_cast<char*>(Su + lane);
  char* Sgl = reinterpret_cast<char*>(Sg + lane);
  const int bar_id = 1 + n, bar_n = 32 * W;
  const long long n_tiles = P.Bp / 32;
  for (long long t = blockIdx.x; t < n_tiles; t += gridDim.x) {
    __syncthreads();   // tables loaded / the previous tile's stencils are no longer read
    for (int r = tid >> 3; r < n_st; r += nt >> 3) cp_async16(STs + r * 32 + 4 * (tid & 7), P.ST + (size_t)r * P.Bp + t * 32 + 4 * (tid & 7));
    float* Un = P.U + ((size_t)n * P.d_rp) * P.Bp + t * 32;
    for (int r = 4 * q + (lane >> 3); r < d_r; r += 4 * W) cp_async16(Su + r * 32 + c4, Un + (size_t)r * P.Bp + c4);
    {
      const long long tn = t + gridDim.x;
      if (tn < n_tiles) {
        for (int r = tid; r < n_st; r += nt) prefetch_l2_line(P.ST + (size_t)r * P.Bp + tn * 32);
        for (int r = 32 * q + lane; r < d_r; r += 32 * W) prefetch_l2_line(P.U + ((size_t)n * P.d_rp + r) * P.Bp + tn * 32);
      }
    }
    cp_async_wait_all();
    __syncthreads();
    // phase 0: dihedral records, (u_cos, u_sin) -> u_phi = -sin u_cos + cos u_sin (d cos = -sin d phi, d sin = cos d phi)
    const int n_rec = poisoned ? 0 : n_feat;
    for (int i = q; i < n_rec; i += W) {
      const int4 fi = s_fi[i];
      if (fi.x != CVF_FEAT_DIHEDRAL) continue;
      const float* sp = reinterpret_cast<const float*>(STl + fi.z);
      float* up = reinterpret_cast<float*>(Sul + fi.y);
      up[0] = fmaf(sp[8 * 32], up[32], -sp[9 * 32] * up[0]);
    }
    named_barrier(bar_id, bar_n);
    // phase 1: per-atom gradients
    float D = 0.0f;
    for (int c = q; c < nc; c += W) {
      const int e_end = s_start[c + 1];
      cvf_v3 g = v3(0.f, 0.f, 0.f);
      for (int e = s_start[c]; e < e_end; ++e) {
        const int4 en = s_adj[e];
        const float u = *reinterpret_cast<const float*>(Sul + en.y);
        if (en.x == 1) {
          const float* sp = reinterpret_cast<const float*>(STl + en.z);
          g = g + (__int_as_float(en.w) * u) * v3(sp[0], sp[32], sp[64]);
        } else {
          JjtLoad L;
          jjt_issue(L, en, STl);
          g = g + u * jjt_combine(L, en.x);
        }
      }
      const cvf_v3 dg = v3(s_dg[3 * c], s_dg[3 * c + 1], s_dg[3 * c + 2]);
      D = fmaf(dg.x * g.x, g.x, fmaf(dg.y * g.y, g.y, fmaf(dg.z * g.z, g.z, D)));
      float* gp = reinterpret_cast<float*>(Sgl + 128 * 3 * c);
      gp[0] = dg.x * g.x, gp[32] = dg.y * g.y, gp[64] = dg.z * g.z;
    }
    named_barrier(bar_id, bar_n);
    // phase 2: vhat per record, in place of u
    for (int i = q; i < n_rec; i += W) {
      const int4 fi = s_fi[i];
      float* up = reinterpret_cast<float*>(Sul + fi.y);
      int e = s_rstart[i];
      const int e_end = s_rstart[i + 1];
      if (fi.x == CVF_FEAT_POSITION) {
        if (e < e_end) {
          const float* gp = reinterpret_cast<const float*>(Sgl + s_radj[e].y);
          up[0] = gp[0], up[32] = gp[32], up[64] = gp[64];
        }
        continue;
      }
      const float u = up[0];
      float v = 0.0f;
      if (fi.w >= 0) {
        v = *reinterpret_cast<const float*>(STl + fi.w) * u;
        D = fmaf(v, u, D);
      }
      for (; e < e_end; ++e) {
        const int4 en = s_radj[e];
        const float* gp = reinterpret_cast<const float*>(Sgl + en.y);
        const cvf_v3 gv = v3(gp[0], gp[32], gp[64]);
        if (en.x == 1) {
          const float* sp = reinterpret_cast<const float*>(STl + en.z);
          v = fmaf(__int_as_float(en.w), dot(v3(sp[0], sp[32], sp[64]), gv), v);
        } else {
          JjtLoad L;
          jjt_issue(L, en, STl);
          v += dot(jjt_combine(L, en.x), gv);
        }
      }
      if (fi.x == CVF_FEAT_DIHEDRAL) {
        const float* sp = reinterpret_cast<const float*>(STl + fi.z);
        up[0] = -sp[9 * 32] * v, up[32] = sp[8 * 32] * v;
      } else {
        up[0] = v;
      }
    }
    Sd[q * 32 + lane] = D;
    named_barrier(bar_id, bar_n);
    for (int r = 4 * q + (lane >> 3); r < d_r; r += 4 * W)
      *reinterpret_cast<float4*>(Un + (size_t)r * P.Bp + c4) = *reinterpret_cast<const float4*>(Su + r * 32 + c4);
    if (q == 0) {
      float Dt = Sd[lane];
      for (int w = 1; w < W; ++w) Dt += Sd[w * 32 + lane];
      P.Dq[(size_t)n * P.Bp + t * 32 + lane] = poisoned ? __int_as_float(0x7fc00000) : Dt;
    }
  }
}

// ------------------------------------------------------------------------------------------------ pass 1
// One CTA per SM, 256 threads, tiles of 512 frames; thread t owns frames 2t, 2t+1 of the tile.
template <int H, int NH>
__global__ void __launch_bounds__(kP1Threads, 1) pass1_kernel(const FastPlan P, float* __restrict__ y_out, int net_split) {
  extern __shared__ __align__(16) float sm[];
  typedef Img<H, NH> I;
  constexpr int F = kP1Frames, HP = H / 2;
  const int tid = threadIdx.x, drp = P.d_rp, d_r = P.d_r, k = P.k;
  float* wsm = sm;
  float* geo = wsm + k * P.img_floats;
  float* tile = geo + P.geo_floats;   // [drp][F]
  for (int i = tid; i < k * P.img_floats + P.geo_floats; i += kP1Threads) sm[i] = P.img[i];
  const long long n_tiles = P.Bp / F;
  const int c0 = 2 * tid;
  // work items: a tile with all its networks, or -- small batches, net_split -- one (tile, network) pair, so that a batch of a few
  // dozen tiles still spreads over the SMs instead of running k networks in sequence on a quarter of them
  const long long n_items = net_split ? n_tiles * k : n_tiles;
  for (long long q = blockIdx.x; q < n_items; q += gridDim.x) {
    const long long t = net_split ? q / k : q;
    const int n_begin = net_split ? (int)(q - t * k) : 0, n_end = net_split ? n_begin + 1 : k;
    const long long f0 = t * F;
    __syncthreads();
    {
      const int nv = P.tile_rows * (F / 4);
      for (int i = tid; i < nv; i += kP1Threads) {
        const int r = i / (F / 4), c4 = i - r * (F / 4);
        st4(tile + r * F + 4 * c4, __ldg(reinterpret_cast<const float4*>(P.Y + (size_t)r * P.Bp + f0) + c4));
      }
    }
    __syncthreads();
    for (int n = n_begin; n < n_end; ++n) {
      const float* W = wsm + n * P.img_floats;
      float om[NH][2][H];   // 1 - A_l^2
      float a[2][H];        // current activations
      float* An = P.A + ((size_t)n * NH * H) * P.Bp + f0 + c0;   // A_l rows kept for pass 2
      // ---- layer 1: z = W1 r + b1 (nn.py:52-57), both frames share every weight load
      {
        float2 z[2][HP];
#pragma unroll
        for (int j = 0; j < HP; ++j) z[0][j] = z[1][j] = lds2(W + I::b1(drp) + 2 * j);
#pragma unroll 2
        for (int kk = 0; kk < d_r; ++kk) {
          const float2 x = lds2(tile + kk * F + c0);
          const float2 x0 = dup(x.x), x1 = dup(x.y);
          const float* wr = W + kk * H;
#pragma unroll
          for (int q = 0; q < H / 4; ++q) {
            const float4 wv = ld4(wr + 4 * q);
            z[0][2 * q] = ffma2(make_float2(wv.x, wv.y), x0, z[0][2 * q]);
            z[0][2 * q + 1] = ffma2(make_float2(wv.z, wv.w), x0, z[0][2 * q + 1]);
            z[1][2 * q] = ffma2(make_float2(wv.x, wv.y), x1, z[1][2 * q]);
            z[1][2 * q + 1] = ffma2(make_float2(wv.z, wv.w), x1, z[1][2 * q + 1]);
          }
        }
#pragma unroll
        for (int f = 0; f < 2; ++f)
#pragma unroll
          for (int j = 0; j < HP; ++j) {
            const float2 t2 = cvf_tanh2(z[f][j]);
            const float2 o2 = ffma2(make_float2(-t2.x, -t2.y), t2, dup(1.0f));
            a[f][2 * j] = t2.x, a[f][2 * j + 1] = t2.y;
            om[0][f][2 * j] = o2.x, om[0][f][2 * j + 1] = o2.y;
          }
#pragma unroll
        for (int o = 0; o < H; ++o) *reinterpret_cast<float2*>(An + (size_t)o * P.Bp) = make_float2(a[0][o], a[1][o]);
      }
      // ---- hidden layers 2..NH
#pragma unroll
      for (int l = 2; l <= NH; ++l) {
        float2 z[2][HP];
#pragma unroll
        for (int j = 0; j < HP; ++j) z[0][j] = z[1][j] = lds2(W + I::bl(drp, l) + 2 * j);
        const float* wt = W + I::wt(drp, l);
#pragma unroll
        for (int kk = 0; kk < H; ++kk) {
          const float2 x0 = dup(a[0][kk]), x1 = dup(a[1][kk]);
#pragma unroll
          for (int q = 0; q < H / 4; ++q) {
            const float4 wv = ld4(wt + kk * H + 4 * q);
            z[0][2 * q] = ffma2(make_float2(wv.x, wv.y), x0, z[0][2 * q]);
            z[0][2 * q + 1] = ffma2(make_float2(wv.z, wv.w), x0, z[0][2 * q + 1]);
            z[1][2 * q] = ffma2(make_float2(wv.x, wv.y), x1, z[1][2 * q]);
            z[1][2 * q + 1] = ffma2(make_float2(wv.z, wv.w), x1, z[1][2 * q + 1]);
          }
        }
#pragma unroll
        for (int f = 0; f < 2; ++f)
#pragma unroll
          for (int j = 0; j < HP; ++j) {
            const float2 t2 = cvf_tanh2(z[f][j]);
            const float2 o2 = ffma2(make_float2(-t2.x, -t2.y), t2, dup(1.0f));
            a[f][2 * j] = t2.x, a[f][2 * j + 1] = t2.y;
            om[l - 1][f][2 * j] = o2.x, om[l - 1][f][2 * j + 1] = o2.y;
          }
#pragma unroll
        for (int o = 0; o < H; ++o) *reinterpret_cast<float2*>(An + (size_t)((l - 1) * H + o) * P.Bp) = make_float2(a[0][o], a[1][o]);
      }
      // ---- output y and the reverse sweep G_l = (1 - A_l^2) .* (W_{l+1}^T G_{l+1}),  G_{NH} seed = Wout
      float yv[2] = {W[I::bout(drp)], W[I::bout(drp)]};
      float g[2][H];
#pragma unroll
      for (int q = 0; q < H / 4; ++q) {
        const float4 wv = ld4(W + I::wout(drp) + 4 * q);
        const float wo[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
        for (int e = 0; e < 4; ++e)
#pragma unroll
          for (int f = 0; f < 2; ++f) {
            yv[f] = fmaf(wo[e], a[f][4 * q + e], yv[f]);
            g[f][4 * q + e] = wo[e] * om[NH - 1][f][4 * q + e];
          }
      }
#pragma unroll
      for (int l = NH; l >= 2; --l) {
        float2 h[2][HP];
#pragma unroll
        for (int j = 0; j < HP; ++j) h[0][j] = h[1][j] = make_float2(0.f, 0.f);
        const float* wn = W + I::wn(drp, l);
#pragma unroll
        for (int o = 0; o < H; ++o) {
          const float2 g0 = dup(g[0][o]), g1 = dup(g[1][o]);
#pragma unroll
          for (int q = 0; q < H / 4; ++q) {
            const float4 wv = ld4(wn + o * H + 4 * q);
            h[0][2 * q] = ffma2(make_float2(wv.x, wv.y), g0, h[0][2 * q]);
            h[0][2 * q + 1] = ffma2(make_float2(wv.z, wv.w), g0, h[0][2 * q + 1]);
            h[1][2 * q] = ffma2(make_float2(wv.x, wv.y), g1, h[1][2 * q]);
            h[1][2 * q + 1] = ffma2(make_float2(wv.z, wv.w), g1, h[1][2 * q + 1]);
          }
        }
#pragma unroll
        for (int f = 0; f < 2; ++f)
#pragma unroll
          for (int j = 0; j < HP; ++j) {
            g[f][2 * j] = h[f][j].x * om[l - 2][f][2 * j];
            g[f][2 * j + 1] = h[f][j].y * om[l - 2][f][2 * j + 1];
          }
      }
      // ---- u = W1^T G_1 in chunks of 12 coordinates (4 atoms), streamed to global memory and into the J sums
      float S2[2] = {0.f, 0.f};
      cvf_v3 gs[2], gsA[2], tau[2], kap[2];
#pragma unroll
      for (int f = 0; f < 2; ++f) gs[f] = gsA[f] = tau[f] = kap[f] = v3(0.f, 0.f, 0.f);
      float* Un = P.U + ((size_t)n * drp) * P.Bp + f0 + c0;
      const float* w1n = W + I::w1n(drp);
      float2 kiv[6];   // K^-1 of both frames, in flight while u is computed
      if (P.kind == 1) {
#pragma unroll
        for (int i = 0; i < 6; ++i) kiv[i] = __ldg(reinterpret_cast<const float2*>(P.Kinv + (size_t)i * P.Bp + f0 + c0));
      }
      for (int c = 0; c < drp / 12; ++c) {
        float2 acc[2][6];
#pragma unroll
        for (int p = 0; p < 6; ++p) acc[0][p] = acc[1][p] = make_float2(0.f, 0.f);
#pragma unroll
        for (int o = 0; o < H; ++o) {
          const float2 g0 = dup(g[0][o]), g1 = dup(g[1][o]);
          const float* wr = w1n + o * drp + 12 * c;
#pragma unroll
          for (int q = 0; q < 3; ++q) {
            const float4 wv = ld4(wr + 4 * q);
            acc[0][2 * q] = ffma2(make_float2(wv.x, wv.y), g0, acc[0][2 * q]);
            acc[0][2 * q + 1] = ffma2(make_float2(wv.z, wv.w), g0, acc[0][2 * q + 1]);
            acc[1][2 * q] = ffma2(make_float2(wv.x, wv.y), g1, acc[1][2 * q]);
            acc[1][2 * q + 1] = ffma2(make_float2(wv.z, wv.w), g1, acc[1][2 * q + 1]);
          }
        }
        float uu[2][12];
#pragma unroll
        for (int f = 0; f < 2; ++f)
#pragma unroll
          for (int p = 0; p < 6; ++p) uu[f][2 * p] = acc[f][p].x, uu[f][2 * p + 1] = acc[f][p].y;
#pragma unroll
        for (int j = 0; j < 12; ++j)
          *reinterpret_cast<float2*>(Un + (size_t)(12 * c + j) * P.Bp) = make_float2(uu[0][j], uu[1][j]);
        if (P.kind == 1) {
#pragma unroll
          for (int m = 0; m < 4; ++m) {
            const int r = 12 * c + 3 * m;
            const float2 yx = lds2(tile + r * F + c0), yy = lds2(tile + (r + 1) * F + c0), yz = lds2(tile + (r + 2) * F + c0);
            const cvf_v3 rf = v3(geo[r], geo[r + 1], geo[r + 2]);
            const float ina = geo[drp + r];
#pragma unroll
            for (int f = 0; f < 2; ++f) {
              const cvf_v3 gg = v3(uu[f][3 * m], uu[f][3 * m + 1], uu[f][3 * m + 2]);
              const cvf_v3 yv3 = f == 0 ? v3(yx.x, yy.x, yz.x) : v3(yx.y, yy.y, yz.y);
              S2[f] += dot(gg, gg);
              gs[f] = gs[f] + gg;
              gsA[f] = gsA[f] + ina * gg;
              tau[f] = tau[f] + cross(gg, yv3);
              kap[f] = kap[f] + cross(gg, rf);
            }
          }
        } else {
#pragma unroll
          for (int j = 0; j < 12; ++j) {
            const float aj = geo[12 * c + j];
#pragma unroll
            for (int f = 0; f < 2; ++f) S2[f] = fmaf(aj * uu[f][j], uu[f][j], S2[f]);
          }
        }
      }
      // ---- Dirichlet density and the alignment-Jacobian vectors (SURVEY 7.3-A; derivation in DESIGN.md)
      float Dv[2];
      if (P.kind == 1) {
        const float* ir = geo + 2 * drp;
        const float nA = ir[6], inA = ir[7];
        float* jq = P.JQ + ((size_t)n * 12) * P.Bp + f0 + c0;
        float out[2][12];
#pragma unroll
        for (int f = 0; f < 2; ++f) {
          float Ki[6];
#pragma unroll
          for (int i = 0; i < 6; ++i) Ki[i] = f == 0 ? kiv[i].x : kiv[i].y;
          const cvf_v3 gm = inA * gs[f];
          const cvf_v3 q = mul_sym(Ki, tau[f]);
          const cvf_v3 Iq = mul_sym(ir, q);
          Dv[f] = S2[f] - 2.0f * dot(gsA[f], gm) - 2.0f * dot(q, kap[f]) + nA * dot(gm, gm) + dot(q, Iq);
          const cvf_v3 dc = inA * gsA[f] - gm;
          const cvf_v3 omv = mul_sym(Ki, kap[f] - Iq);
          out[f][0] = gm.x, out[f][1] = gm.y, out[f][2] = gm.z, out[f][3] = q.x, out[f][4] = q.y, out[f][5] = q.z;
          out[f][6] = dc.x, out[f][7] = dc.y, out[f][8] = dc.z, out[f][9] = omv.x, out[f][10] = omv.y, out[f][11] = omv.z;
        }
#pragma unroll
        for (int i = 0; i < 12; ++i) *reinterpret_cast<float2*>(jq + (size_t)i * P.Bp) = make_float2(out[0][i], out[1][i]);
      } else {
        Dv[0] = S2[0], Dv[1] = S2[1];
      }
      *reinterpret_cast<float2*>(P.Dq + (size_t)n * P.Bp + f0 + c0) = make_float2(Dv[0], Dv[1]);
      *reinterpret_cast<float2*>(P.Ys + (size_t)n * P.Bp + f0 + c0) = make_float2(yv[0], yv[1]);
      if (y_out) {
#pragma unroll
        for (int f = 0; f < 2; ++f)
          if (f0 + c0 + f < P.B) y_out[(size_t)n * P.B + f0 + c0 + f] = yv[f];
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ stats
// fp64 batch sums S0, S1[i], S2[i][j], SD[i] (core.py:406-410,426) from w, y, D in ONE pass over the frames: a thread keeps all
// 1 + 2k + k^2 sums of its frames in registers (K networks: template), then a fixed-order block reduction; deterministic.
template <int K>
__global__ void __launch_bounds__(256) stats_kernel(const FastPlan P, const float* __restrict__ w, double* __restrict__ part) {
  constexpr int NS = 1 + 2 * K + K * K;
  __shared__ double red[8][NS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double acc[NS];
#pragma unroll
  for (int s = 0; s < NS; ++s) acc[s] = 0.0;
  for (long long f = (long long)blockIdx.x * blockDim.x + threadIdx.x; f < P.B; f += (long long)gridDim.x * blockDim.x) {
    const double wf = w[f];
    double y[K];
#pragma unroll
    for (int i = 0; i < K; ++i) y[i] = (double)P.Ys[(size_t)i * P.Bp + f];
    acc[0] += wf;
#pragma unroll
    for (int i = 0; i < K; ++i) {
      const double wy = wf * y[i];
      acc[1 + i] += wy;
#pragma unroll
      for (int j = 0; j < K; ++j) acc[1 + K + i * K + j] += wy * y[j];
      acc[1 + K + K * K + i] += wf * (double)P.Dq[(size_t)i * P.Bp + f];
    }
  }
#pragma unroll
  for (int s = 0; s < NS; ++s) {
    double v = acc[s];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) red[warp][s] = v;
  }
  __syncthreads();
  if (threadIdx.x < NS) {
    double t = 0.0;
    for (int q = 0; q < 8; ++q) t += red[q][threadIdx.x];
    part[(size_t)blockIdx.x * NS + threadIdx.x] = t;
  }
}

// ---- tensor memory as per-warp accumulator storage -----------------------------------------------------------------------
// Pass 2 adds ~2 200 weight-gradient partial sums per (32-frame tile, network) to running totals.  As fp64 atomics to a
// per-warp vector in global memory those additions were the kernel's largest consumer of load/store-pipe cycles (measured:
// ~1.3 cycles per lane).  Tensor memory (256 KB per SM, untouched by this SIMT kernel) holds them instead: a warp owns the 32
// lanes of its quadrant x 256 columns, every lane keeps the totals of the (output, input) pairs it computes anyway in columns
// of its own lane, and one tcgen05.ld / add / tcgen05.st round trip per group of 16 replaces the atomics (single owner, fixed
// order: deterministic).  The totals are fp32 over the ~10^2 tiles a warp processes and go to the fp64 vector once, at the end.
// tcgen05.ld / tcgen05.st of N consecutive 32-bit columns of the calling lane (32x32b shape: one TMEM lane per thread), N = 1, 2, 4, 8, 16
template <int N>
struct TmPiece;
template <>
struct TmPiece<1> {
  static __device__ __forceinline__ void ld(uint32_t a, uint32_t* r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(r[0]) : "r"(a) : "memory");
  }
  static __device__ __forceinline__ void st(uint32_t a, const uint32_t* r) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x1.b32 [%0], {%1};" ::"r"(a), "r"(r[0]) : "memory");
  }
};
template <>
struct TmPiece<2> {
  static __device__ __forceinline__ void ld(uint32_t a, uint32_t* r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(r[0]), "=r"(r[1]) : "r"(a) : "memory");
  }
  static __device__ __forceinline__ void st(uint32_t a, const uint32_t* r) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1, %2};" ::"r"(a), "r"(r[0]), "r"(r[1]) : "memory");
  }
};
template <>
struct TmPiece<4> {
  static __device__ __forceinline__ void ld(uint32_t a, uint32_t* r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a) : "memory");
  }
  static __device__ __forceinline__ void st(uint32_t a, const uint32_t* r) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]) : "memory");
  }
};
template <>
struct TmPiece<8> {
  static __device__ __forceinline__ void ld(uint32_t a, uint32_t* r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(a)
                 : "memory");
  }
  static __device__ __forceinline__ void st(uint32_t a, const uint32_t* r) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(a), "r"(r[0]), "r"(r[1]), "r"(r[2]),
                 "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
                 : "memory");
  }
};
template <>
struct TmPiece<16> {
  static __device__ __forceinline__ void ld(uint32_t a, uint32_t* r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(a)
        : "memory");
  }
  static __device__ __forceinline__ void st(uint32_t a, const uint32_t* r) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(a),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]),
        "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
        : "memory");
  }
};
// N columns as power-of-two pieces (16s first, then 8, 4, 2, 1), one wait at the end
template <int N>
struct TmIo {
  template <int OFF, int REM>
  static __device__ __forceinline__ void ld_pieces(uint32_t a, uint32_t* r) {
    if constexpr (REM > 0) {
      constexpr int P = REM >= 16 ? 16 : REM >= 8 ? 8 : REM >= 4 ? 4 : REM >= 2 ? 2 : 1;
      TmPiece<P>::ld(a + OFF, r + OFF);
      ld_pieces<OFF + P, REM - P>(a, r);
    }
  }
  template <int OFF, int REM>
  static __device__ __forceinline__ void st_pieces(uint32_t a, const uint32_t* r) {
    if constexpr (REM > 0) {
      constexpr int P = REM >= 16 ? 16 : REM >= 8 ? 8 : REM >= 4 ? 4 : REM >= 2 ? 2 : 1;
      TmPiece<P>::st(a + OFF, r + OFF);
      st_pieces<OFF + P, REM - P>(a, r);
    }
  }
  static __device__ __forceinline__ void ld(uint32_t a, float (&v)[N]) {
    uint32_t r[N];
    ld_pieces<0, N>(a, r);
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < N; ++i) v[i] = __uint_as_float(r[i]);
  }
  static __device__ __forceinline__ void st(uint32_t a, const float (&v)[N]) {
    uint32_t r[N];
#pragma unroll
    for (int i = 0; i < N; ++i) r[i] = __float_as_uint(v[i]);
    st_pieces<0, N>(a, r);
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
  }
};
// totals[a .. a+N) += v
template <int N>
__device__ __forceinline__ void tm_add(uint32_t a, const float (&v)[N]) {
  float t[N];
  TmIo<N>::ld(a, t);
#pragma unroll
  for (int i = 0; i < N; ++i) t[i] += v[i];
  TmIo<N>::st(a, t);
}
// Lane (half, og, ig) of a warp holds, after the cross-half shuffle, the full sum of every entry r[j][i] of its TO x TI tile; entry
// e = j * TI + i is kept by the half-warp e & 1, in slot e >> 1 of the group.
template <int TO, int TI, int GS>
__device__ __forceinline__ void tm_add_tile(uint32_t a, const float (&r)[TO][TI], int half) {
  static_assert((TO * TI + 1) / 2 == GS, "group size = ceil(entries / 2)");
  float v[GS];
#pragma unroll
  for (int p = 0; p < GS; ++p) {
    const int e0 = 2 * p, e1 = 2 * p + 1;
    const float v0 = e0 < TO * TI ? r[e0 / TI][e0 % TI] : 0.0f;
    const float v1 = e1 < TO * TI ? r[e1 / TI][e1 % TI] : 0.0f;
    v[p] = half ? v1 : v0;
  }
  tm_add<GS>(a, v);
}
constexpr int kTmColsPerWarp = 256;

// ------------------------------------------------------------------------------------------------ pass 2
// lane L ends with sum over lanes of v[L] (v[i >= N] treated as 0); 31 shuffles for up to 32 values.
template <int N>
__device__ __forceinline__ float warp_reduce_scatter(float (&v)[32], int lane) {
#pragma unroll
  for (int i = N; i < 32; ++i) v[i] = 0.0f;
#pragma unroll
  for (int m = 16; m >= 1; m >>= 1) {
    const bool hi = (lane & m) != 0;
#pragma unroll
    for (int i = 0; i < m; ++i) {
      const float send = hi ? v[i] : v[i + m];
      const float keep = hi ? v[i + m] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, m);
    }
  }
  return v[0];
}

// Warp-level outer product over the warp's 32 frames:  acc[j][i] += sum_f X[rowX(j)][f] * Z[rowZ(i)][f] for two operand
// pairs (Xa,Za) and (Xb,Zb).  Rows are kRowPad floats; a lane reads 4 frames per 128-bit load and keeps the even/odd
// frame partial sums packed in one FFMA2 accumulator.
template <int TO, int TI>
__device__ __forceinline__ void outer_tile(float2 (&acc)[TO][TI], const float* __restrict__ Xa, const float* __restrict__ Za,
                                           const float* __restrict__ Xb, const float* __restrict__ Zb, int strideX, int strideZ,
                                           int fbeg, int fend) {
#pragma unroll 1
  for (int f = fbeg; f < fend; f += 4) {
    float4 x[TO], z[TI];
#pragma unroll
    for (int j = 0; j < TO; ++j) x[j] = ld4(Xa + j * strideX + f);
#pragma unroll
    for (int i = 0; i < TI; ++i) z[i] = ld4(Za + i * strideZ + f);
    // every accumulator is touched once per sweep: dependent FFMA2s are TO * TI instructions apart
#pragma unroll
    for (int j = 0; j < TO; ++j)
#pragma unroll
      for (int i = 0; i < TI; ++i) acc[j][i] = ffma2(make_float2(x[j].x, x[j].y), make_float2(z[i].x, z[i].y), acc[j][i]);
#pragma unroll
    for (int j = 0; j < TO; ++j)
#pragma unroll
      for (int i = 0; i < TI; ++i) acc[j][i] = ffma2(make_float2(x[j].z, x[j].w), make_float2(z[i].z, z[i].w), acc[j][i]);
#pragma unroll
    for (int j = 0; j < TO; ++j) x[j] = ld4(Xb + j * strideX + f);
#pragma unroll
    for (int i = 0; i < TI; ++i) z[i] = ld4(Zb + i * strideZ + f);
    // every accumulator is touched once per sweep: dependent FFMA2s are TO * TI instructions apart
#pragma unroll
    for (int j = 0; j < TO; ++j)
#pragma unroll
      for (int i = 0; i < TI; ++i) acc[j][i] = ffma2(make_float2(x[j].x, x[j].y), make_float2(z[i].x, z[i].y), acc[j][i]);
#pragma unroll
    for (int j = 0; j < TO; ++j)
#pragma unroll
      for (int i = 0; i < TI; ++i) acc[j][i] = ffma2(make_float2(x[j].z, x[j].w), make_float2(z[i].z, z[i].w), acc[j][i]);
  }
}

// Pass 2.  One CTA per SM, up to 8 independent warps; a warp owns tiles of 32 frames (lane = frame) and a private set of
// operand rows: Z rows (A_l | T_l of every hidden layer -- A_l read back from pass 1's P.A, T_l propagated here; during layer 1
// they stage r and u) and X rows (s_l | G_l of the layer being reduced, then the flush buffer).  The first layer's weight
// gradient needs r and vhat of every frame as operand rows once (s_1, G_1) exist, when the Z rows are free again: they are
// re-staged from global memory (L2: the warp read r and wrote vhat a few microseconds earlier) in double-buffered column chunks,
// and the vhat lines are dropped from L2 once staged (discard.global.L2), so no intermediate of pass 2 goes through HBM.
template <int H, int NH, int CW>
__global__ void __launch_bounds__(256, 1)
pass2_kernel(const FastPlan P, const float* __restrict__ w, const double* __restrict__ combine, int rows_per_warp,
             const float* __restrict__ seed_extra, int net_split) {
  extern __shared__ __align__(16) float sm[];
  typedef Img<H, NH> I;
  constexpr int HP = H / 2, RP = kRowPad, TQ = H / 4;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nt = blockDim.x, nw = nt >> 5;
  const int drp = P.d_rp, d_r = P.d_r, k = P.k;
  float* wsm = sm;                                   // k * img2 (pass-2 prefix of every image)
  float* geo = wsm + k * P.img2_floats;
  double* comb = reinterpret_cast<double*>(geo + P.geo_floats);   // mean[k], cD[k], C2[k*k], a0[k]
  const int n_comb = 3 * k + k * k;
  float* rows0 = reinterpret_cast<float*>(comb + n_comb + (n_comb & 1));
  const bool inline_dw1 = drp == 12;                       // pass2_inline_dw1(): r and vhat keep rows of their own
  const int base_rows = rows_per_warp - (inline_dw1 ? 2 * drp : 0);
  float* Zr = rows0 + (size_t)warp * rows_per_warp * RP;   // [NH][2H] A_l | T_l; at the end, two chunk buffers of r | vhat rows
  float* Xr = Zr + (size_t)(base_rows - 2 * H) * RP;       // [2H]     s_l | G_l; flush buffer (the last rows of the block)
  float* Sr = inline_dw1 ? Zr + (size_t)base_rows * RP : Zr;   // [drp]    r staged for layer 1
  float* Su = Sr + drp * RP;                               // [drp]    u staged for layer 1
  float* Sj = Zr + 2 * drp * RP;                           // [12]     alignment-Jacobian vectors staged for layer 1
  for (int n = 0; n < k; ++n)
    for (int i = tid; i < P.img2_floats; i += nt) wsm[n * P.img2_floats + i] = P.img[(size_t)n * P.img_floats + i];
  for (int i = tid; i < P.geo_floats; i += nt) geo[i] = P.img[(size_t)k * P.img_floats + i];
  for (int i = tid; i < n_comb; i += nt) comb[i] = combine[3 + 2 * k + i];
  for (int i = tid; i < nw * rows_per_warp * RP; i += nt) rows0[i] = 0.0f;
  const int n_part = k * P.n_params;
  double* part = P.part + ((size_t)blockIdx.x * nw + warp) * n_part;
  // tensor-memory accumulators (see above): per network n_chunks groups for dW_1, NH - 1 groups for the hidden layers' dW,
  // four single slots (dWout | dbout by lane, db_NH .. db_1 by lane)
  constexpr int CI1 = CW / 4;
  constexpr int GS1 = (TQ * CI1 + 1) / 2, GSH = (TQ * TQ + 1) / 2, GSI = (TQ * 3 + 1) / 2;   // dW_1 chunk, hidden dW, 12-column dW_1
  const int n_chunks1 = inline_dw1 ? 1 : (d_r + CW - 1) / CW;
  const int tm_hid = n_chunks1 * GS1, tm_sing = tm_hid + (NH - 1) * GSH, tm_per_net = tm_sing + 4;
  const int tm_nets = kTmColsPerWarp / tm_per_net < k ? kTmColsPerWarp / tm_per_net : k;   // further networks: fp64 atomics
  for (int i = tm_nets * P.n_params + lane; i < n_part; i += 32) part[i] = 0.0;            // ... to this warp's vector in global memory
  __shared__ uint32_t tmem_slot;
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(&tmem_slot)),
                 "r"(512u)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmw = tmem_slot + ((uint32_t)(32 * (warp & 3)) << 16) + (uint32_t)(kTmColsPerWarp * (warp >> 2));
  {
    float z16[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) z16[i] = 0.0f;
    for (int c = 0; c < kTmColsPerWarp; c += 16) TmIo<16>::st(tmw + c, z16);
  }
  const double* c_mean = comb;
  const double* c_cD = comb + k;
  const double* c_C2 = comb + 2 * k;
  const double* c_a0 = comb + 2 * k + k * k;

  const long long n_tiles = P.Bp / 32;
  // work items: a 32-frame tile with all its networks, or -- small batches, net_split -- one (tile, network) pair per item
  const long long n_items = net_split ? n_tiles * k : n_tiles;
  for (long long q = (long long)blockIdx.x * nw + warp; q < n_items; q += (long long)gridDim.x * nw) {
    const long long t = net_split ? q / k : q;
    const int n_begin = net_split ? (int)(q - t * k) : 0, n_end = net_split ? n_begin + 1 : k;
    const long long f = t * 32 + lane;
    const float wf = f < P.B ? __ldg(w + f) : 0.0f;
    const long long t_next = net_split ? n_tiles : t + (long long)gridDim.x * nw;   // no look-ahead across work items when split
    float ysv[kMaxK];
#pragma unroll
    for (int j = 0; j < kMaxK; ++j) ysv[j] = j < k ? __ldg(P.Ys + (size_t)j * P.Bp + f) : 0.0f;
    for (int n = n_begin; n < n_end; ++n) {
      const float* W = wsm + n * P.img2_floats;
      double* pn = part + (size_t)n * P.n_params;
      const bool tm = n < tm_nets;                          // this network's totals live in tensor memory
      const uint32_t tmn = tmw + (uint32_t)(n * tm_per_net);
      float* Ut = P.U + ((size_t)n * drp) * P.Bp + t * 32;
      __syncwarp();   // the previous network's flush has finished reading the X rows
      if (P.kind == 1 || inline_dw1) stage_rows(Sr, P.Y + t * 32, d_r, P.Bp, lane);   // r: the alignment Jacobian / the in-row dW_1 read it
      stage_rows(Su, Ut, d_r, P.Bp, lane);
      if (P.kind == 1) stage_rows(Sj, P.JQ + ((size_t)n * 12) * P.Bp + t * 32, 12, P.Bp, lane);
      // L2 prefetch of what is read next: the next network's u rows, or the next tile's r rows and first u rows
      if (n + 1 < n_end) {
        prefetch_rows(P.U + ((size_t)(n + 1) * drp) * P.Bp + t * 32, d_r, P.Bp, lane);
        prefetch_rows(P.A + ((size_t)(n + 1) * NH * H) * P.Bp + t * 32, NH * H, P.Bp, lane);
        if (P.kind == 1) prefetch_rows(P.JQ + ((size_t)(n + 1) * 12) * P.Bp + t * 32, 12, P.Bp, lane);
      } else if (t_next < n_tiles) {
        prefetch_rows(P.Y + t_next * 32, d_r, P.Bp, lane);
        prefetch_rows(P.U + t_next * 32, d_r, P.Bp, lane);
        prefetch_rows(P.A + t_next * 32, NH * H, P.Bp, lane);
        if (P.kind == 1) prefetch_rows(P.JQ + t_next * 32, 12, P.Bp, lane);
        prefetch_rows(P.Ys + t_next * 32, k, P.Bp, lane);
        if (lane == 0) prefetch_l2_line(w + t_next * 32);
      }
      float seed;
      {
        double s = c_a0[n];
#pragma unroll
        for (int j = 0; j < kMaxK; ++j)
          if (j < k) s += c_C2[n * k + j] * ((double)ysv[j] - c_mean[j]);
        seed = (float)((double)wf * s);
        if (seed_extra != nullptr && f < P.B) seed += __ldg(seed_extra + (size_t)n * P.B + f);   // transfer-operator term
      }
      const float scale = (float)(2.0 * (double)wf * c_cD[n]);
      // ---- tangent forward, layer 1: zdot = W1 v; v = scale * J_r J_r^T u built on the fly.  The primal activations A_l are
      // not recomputed: pass 1 left them in P.A (same arithmetic, so the same values) and each lane reads its frame's column
      const float* An = P.A + ((size_t)n * NH * H) * P.Bp + f;
      float2 zd[HP];
#pragma unroll
      for (int j = 0; j < HP; ++j) zd[j] = make_float2(0.f, 0.f);
      if (P.kind == 1) {
        cp_async_wait_all();
        __syncwarp();
        const float* jq = Sj + lane;
        const cvf_v3 gm = v3(jq[0], jq[RP], jq[2 * RP]);
        const cvf_v3 q = v3(jq[3 * RP], jq[4 * RP], jq[5 * RP]);
        const cvf_v3 dc = v3(jq[6 * RP], jq[7 * RP], jq[8 * RP]);
        const cvf_v3 omv = v3(jq[9 * RP], jq[10 * RP], jq[11 * RP]);
#pragma unroll 2
        for (int a = 0; a < P.n_atoms; ++a) {
          const int r = 3 * a;
          const cvf_v3 uu = v3(Su[r * RP + lane], Su[(r + 1) * RP + lane], Su[(r + 2) * RP + lane]);
          const cvf_v3 yv3 = v3(Sr[r * RP + lane], Sr[(r + 1) * RP + lane], Sr[(r + 2) * RP + lane]);
          const cvf_v3 rf = v3(geo[r], geo[r + 1], geo[r + 2]);
          const float ina = geo[drp + r];
          const cvf_v3 gp = uu - ina * (gm + cross(rf, q));
          const cvf_v3 vh = (gp - dc) + cross(omv, yv3);   // vhat = J_r J_r^T u, kept for pass 2b in place of u
          Su[r * RP + lane] = vh.x, Su[(r + 1) * RP + lane] = vh.y, Su[(r + 2) * RP + lane] = vh.z;
          const cvf_v3 vv = scale * vh;
          const float vin[3] = {vv.x, vv.y, vv.z};
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            const float2 x1 = dup(vin[c]);
            const float* wr = W + (r + c) * H;
#pragma unroll
            for (int qq = 0; qq < TQ; ++qq) {
              const float4 wv = ld4(wr + 4 * qq);
              zd[2 * qq] = ffma2(make_float2(wv.x, wv.y), x1, zd[2 * qq]);
              zd[2 * qq + 1] = ffma2(make_float2(wv.z, wv.w), x1, zd[2 * qq + 1]);
            }
          }
        }
      } else {
        cp_async_wait_all();
        __syncwarp();
#pragma unroll 2
        for (int r = 0; r < d_r; ++r) {
          const float vh = geo[r] * Su[r * RP + lane];
          Su[r * RP + lane] = vh;
          const float vin = scale * vh;
          const float2 x1 = dup(vin);
          const float* wr = W + r * H;
#pragma unroll
          for (int qq = 0; qq < TQ; ++qq) {
            const float4 wv = ld4(wr + 4 * qq);
            zd[2 * qq] = ffma2(make_float2(wv.x, wv.y), x1, zd[2 * qq]);
            zd[2 * qq + 1] = ffma2(make_float2(wv.z, wv.w), x1, zd[2 * qq + 1]);
          }
        }
      }
      float a[H], tg[H];   // A_l, T_l = (1 - A_l^2) zdot_l of the current layer
#pragma unroll
      for (int o = 0; o < H; ++o) a[o] = __ldg(An + (size_t)o * P.Bp);
      // vhat rows -> global memory (in place of u), 16 bytes per lane, before the Z rows take over the staging area
      __syncwarp();
      if (!inline_dw1) store_rows(Ut, Su, d_r, P.Bp, lane);
#pragma unroll
      for (int j = 0; j < HP; ++j) {
        const float2 t2 = make_float2(a[2 * j], a[2 * j + 1]);
        const float2 g2 = cvf_fmul2(ffma2(make_float2(-t2.x, -t2.y), t2, dup(1.0f)), zd[j]);
        tg[2 * j] = g2.x, tg[2 * j + 1] = g2.y;
      }
      __syncwarp();
#pragma unroll
      for (int o = 0; o < H; ++o) Zr[o * RP + lane] = a[o], Zr[(H + o) * RP + lane] = tg[o];
#pragma unroll 1   // one copy of the layer code for every hidden layer: the kernel has to stay inside the instruction cache
      for (int l = 2; l <= NH; ++l) {
#pragma unroll
        for (int o = 0; o < H; ++o) a[o] = __ldg(An + (size_t)((l - 1) * H + o) * P.Bp);   // in flight under the products
#pragma unroll
        for (int j = 0; j < HP; ++j) zd[j] = make_float2(0.f, 0.f);
        const float* wt = W + I::wt(drp, l);
#pragma unroll
        for (int kk = 0; kk < H; ++kk) {
          const float2 x1 = dup(tg[kk]);
#pragma unroll
          for (int qq = 0; qq < TQ; ++qq) {
            const float4 wv = ld4(wt + kk * H + 4 * qq);
            zd[2 * qq] = ffma2(make_float2(wv.x, wv.y), x1, zd[2 * qq]);
            zd[2 * qq + 1] = ffma2(make_float2(wv.z, wv.w), x1, zd[2 * qq + 1]);
          }
        }
#pragma unroll
        for (int j = 0; j < HP; ++j) {
          const float2 t2 = make_float2(a[2 * j], a[2 * j + 1]);
          const float2 g2 = cvf_fmul2(ffma2(make_float2(-t2.x, -t2.y), t2, dup(1.0f)), zd[j]);
          tg[2 * j] = g2.x, tg[2 * j + 1] = g2.y;
        }
#pragma unroll
        for (int o = 0; o < H; ++o) Zr[((l - 1) * 2 * H + o) * RP + lane] = a[o], Zr[((l - 1) * 2 * H + H + o) * RP + lane] = tg[o];
      }
      // ---- output layer: dWout = sum_f seed A_NH + T_NH, dbout = sum_f seed;  G_NH, s_NH
      float gl[H], sl[H];
      {
        float red[32];
#pragma unroll
        for (int o = 0; o < H; ++o) red[o] = fmaf(seed, a[o], tg[o]);
        red[H] = seed;
        const float tot = warp_reduce_scatter<H + 1>(red, lane);
        if (tm) {
          const float t1[1] = {tot};
          tm_add<1>(tmn + tm_sing, t1);
        } else if (lane < H) atomicAdd(pn + P.gw_off[NH] + lane, (double)tot);
        else if (lane == H) atomicAdd(pn + P.gb_off[NH], (double)tot);
#pragma unroll
        for (int qq = 0; qq < TQ; ++qq) {
          const float4 wv = ld4(W + I::wout(drp) + 4 * qq);
          const float wo[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int o = 4 * qq + e;
            const float omo = fmaf(-a[o], a[o], 1.0f);
            gl[o] = omo * wo[e];
            sl[o] = fmaf(-2.0f * a[o] * wo[e], tg[o], omo * seed * wo[e]);
          }
        }
      }
      // ---- reverse sweep over the hidden layers with the outer products of each layer as soon as (s_l, G_l) exist
#pragma unroll 1
      for (int l = NH; l >= 1; --l) {
        // db_l = sum_f s_l
        {
          float red[32];
#pragma unroll
          for (int o = 0; o < H; ++o) red[o] = sl[o];
          const float tot = warp_reduce_scatter<H>(red, lane);
          if (tm) {
            const float t1[1] = {tot};
            tm_add<1>(tmn + tm_sing + 1 + (NH - l), t1);
          } else if (lane < H) atomicAdd(pn + P.gb_off[l - 1] + lane, (double)tot);
        }
        if (l >= 2) {
          __syncwarp();
#pragma unroll
          for (int o = 0; o < H; ++o) Xr[o * RP + lane] = sl[o], Xr[(H + o) * RP + lane] = gl[o];
          __syncwarp();
          // dW_l [H][H] += s_l (x) A_{l-1} + G_l (x) T_{l-1}: half-warps split the frames, 16 lanes x (TQ x TQ) entries
          const int half = lane >> 4, l16 = lane & 15, og = l16 >> 2, ig = l16 & 3;
          float2 acc[TQ][TQ];
#pragma unroll
          for (int j = 0; j < TQ; ++j)
#pragma unroll
            for (int i = 0; i < TQ; ++i) acc[j][i] = make_float2(0.f, 0.f);
          const float* Zl = Zr + (size_t)(l - 2) * 2 * H * RP;
          outer_tile<TQ, TQ>(acc, Xr + og * RP, Zl + ig * RP, Xr + (H + og) * RP, Zl + (H + ig) * RP, 4 * RP, 4 * RP, 16 * half,
                             16 * half + 16);
          float r2[TQ][TQ];
#pragma unroll
          for (int j = 0; j < TQ; ++j)
#pragma unroll
            for (int i = 0; i < TQ; ++i) {
              r2[j][i] = acc[j][i].x + acc[j][i].y;
              r2[j][i] += __shfl_xor_sync(0xffffffffu, r2[j][i], 16);
            }
          __syncwarp();
          if (tm) {
            tm_add_tile<TQ, TQ, GSH>(tmn + tm_hid + (l - 2) * GSH, r2, half);
          } else {
            if (half == 0) {
#pragma unroll
              for (int j = 0; j < TQ; ++j)
#pragma unroll
                for (int i = 0; i < TQ; ++i) Xr[(4 * j + og) * H + 4 * i + ig] = r2[j][i];
            }
            __syncwarp();
            for (int e = lane; e < H * H; e += 32) atomicAdd(pn + P.gw_off[l - 1] + e, (double)Xr[e]);
          }
          // next (G, s): h = W_l^T (G_l, s_l);  G_{l-1} = om h_G,  s_{l-1} = -2 A h_G T + om h_s
          float2 hg[HP], hs[HP];
#pragma unroll
          for (int j = 0; j < HP; ++j) hg[j] = hs[j] = make_float2(0.f, 0.f);
          const float* wn = W + I::wn(drp, l);
#pragma unroll
          for (int o = 0; o < H; ++o) {
            const float2 g0 = dup(gl[o]), s0 = dup(sl[o]);
#pragma unroll
            for (int qq = 0; qq < TQ; ++qq) {
              const float4 wv = ld4(wn + o * H + 4 * qq);
              hg[2 * qq] = ffma2(make_float2(wv.x, wv.y), g0, hg[2 * qq]);
              hg[2 * qq + 1] = ffma2(make_float2(wv.z, wv.w), g0, hg[2 * qq + 1]);
              hs[2 * qq] = ffma2(make_float2(wv.x, wv.y), s0, hs[2 * qq]);
              hs[2 * qq + 1] = ffma2(make_float2(wv.z, wv.w), s0, hs[2 * qq + 1]);
            }
          }
#pragma unroll
          for (int j = 0; j < HP; ++j) {
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              const int o = 2 * j + e;
              const float ao = Zl[o * RP + lane], to = Zl[(H + o) * RP + lane];
              const float omo = fmaf(-ao, ao, 1.0f);
              const float hgo = e == 0 ? hg[j].x : hg[j].y, hso = e == 0 ? hs[j].x : hs[j].y;
              gl[o] = omo * hgo;
              sl[o] = fmaf(-2.0f * ao * hgo, to, omo * hso);
            }
          }
        } else {
          // dW_1 = sum_f s_1 (x) r + (scale G_1) (x) vhat:  (s_1 | scale G_1) become X rows; r and vhat (the latter was written to
          // global memory in place of u during layer 1) come back in column chunks of CW rows each, double-buffered in the
          // Z rows that the reverse sweep no longer needs
          __syncwarp();
#pragma unroll
          for (int o = 0; o < H; ++o) Xr[o * RP + lane] = sl[o], Xr[(H + o) * RP + lane] = scale * gl[o];
          __syncwarp();
          if (!inline_dw1) {
            constexpr int CI = CW / 4;      // columns per lane (4 column groups) of a chunk of CW columns
            const int half = lane >> 4, l16 = lane & 15, og = l16 >> 2, ig = l16 & 3;
            const int n_chunks = (d_r + CW - 1) / CW;
            const float* Yt = P.Y + t * 32;
            auto stage_chunk = [&](int c) {
              float* R = Zr + (size_t)(c & 1) * 2 * CW * RP;
              const int c0 = c * CW, nr = d_r - c0 < CW ? d_r - c0 : CW;
              stage_rows(R, Yt + (size_t)c0 * P.Bp, nr, P.Bp, lane);
              stage_rows(R + CW * RP, Ut + (size_t)c0 * P.Bp, nr, P.Bp, lane);
              cp_async_commit();
            };
            stage_chunk(0);
            for (int c = 0; c < n_chunks; ++c) {
              if (c + 1 < n_chunks) {
                stage_chunk(c + 1);
                cp_async_wait_group<1>();
              } else {
                cp_async_wait_all();
              }
              __syncwarp();
              const float* R = Zr + (size_t)(c & 1) * 2 * CW * RP;
              const int c0 = c * CW;
              // the chunk's vhat rows were written by this warp only to come back from L2 here; nothing reads them again
              // (pass 2 consumes the scratch), so their lines need not reach HBM
              for (int r = c0 + lane; r < d_r && r < c0 + CW; r += 32) discard_l2_line(Ut + (size_t)r * P.Bp);
              float2 acc[TQ][CI];
#pragma unroll
              for (int j = 0; j < TQ; ++j)
#pragma unroll
                for (int i = 0; i < CI; ++i) acc[j][i] = make_float2(0.f, 0.f);
              // rows beyond d_r in the last chunk hold stale (finite) values of earlier tiles: their columns are not flushed
              outer_tile<TQ, CI>(acc, Xr + og * RP, R + (CI * ig) * RP, Xr + (H + og) * RP, R + (CW + CI * ig) * RP, 4 * RP, RP,
                                 16 * half, 16 * half + 16);
              // both half-warps end with the sums over all 32 frames; each keeps / flushes half of the entries
              float r1[TQ][CI];
#pragma unroll
              for (int j = 0; j < TQ; ++j)
#pragma unroll
                for (int i = 0; i < CI; ++i) {
                  r1[j][i] = acc[j][i].x + acc[j][i].y;
                  r1[j][i] += __shfl_xor_sync(0xffffffffu, r1[j][i], 16);
                }
              if (tm) {
                tm_add_tile<TQ, CI, GS1>(tmn + c * GS1, r1, half);
              } else {
#pragma unroll
                for (int j = 0; j < TQ; ++j)
#pragma unroll
                  for (int i = 0; i < CI; ++i) {
                    const int col = c0 + CI * ig + i;
                    if (((j * CI + i) & 1) == half && col < d_r) atomicAdd(pn + P.gw_off[0] + (4 * j + og) * d_r + col, (double)r1[j][i]);
                  }
              }
              __syncwarp();   // the chunk's buffer is restaged two iterations later; all lanes are done reading it
            }
          } else {
            // dW_1 [H][d_r <= 12] here: the same half-warp product as the hidden layers, 12 columns
            const int half = lane >> 4, l16 = lane & 15, og = l16 >> 2, ig = l16 & 3;
            float2 acc[TQ][3];
#pragma unroll
            for (int j = 0; j < TQ; ++j)
#pragma unroll
              for (int i = 0; i < 3; ++i) acc[j][i] = make_float2(0.f, 0.f);
            outer_tile<TQ, 3>(acc, Xr + og * RP, Sr + ig * RP, Xr + (H + og) * RP, Su + ig * RP, 4 * RP, 4 * RP, 16 * half,
                              16 * half + 16);
            float r1[TQ][3];
#pragma unroll
            for (int j = 0; j < TQ; ++j)
#pragma unroll
              for (int i = 0; i < 3; ++i) {
                r1[j][i] = acc[j][i].x + acc[j][i].y;
                r1[j][i] += __shfl_xor_sync(0xffffffffu, r1[j][i], 16);
              }
            __syncwarp();   // every lane has finished reading the X rows
            if (tm) {
              tm_add_tile<TQ, 3, GSI>(tmn, r1, half);
            } else {
              if (half == 0) {
#pragma unroll
                for (int j = 0; j < TQ; ++j)
#pragma unroll
                  for (int i = 0; i < 3; ++i) {
                    const int col = 4 * i + ig;
                    if (col < d_r) Xr[(4 * j + og) * d_r + col] = r1[j][i];
                  }
              }
              __syncwarp();
              for (int e = lane; e < H * d_r; e += 32) atomicAdd(pn + P.gw_off[0] + e, (double)Xr[e]);
            }
          }
        }
      }
    }
  }
  // ---- the CTA's gradient vector: the warps add their tensor-memory totals, one warp after the other (fixed order:
  // deterministic), into an fp64 vector in the shared memory the operand rows no longer need; networks whose totals went to
  // per-warp vectors in global memory by atomics (beyond tm_nets) are folded in after them; one vector per CTA leaves the SM
  __syncthreads();
  // [tm_nets * n_params]: up to kMaxK networks keep totals in tensor memory (e.g. [12,20,20,1] with k = 8); for every shape the
  // host accepts, their vectors take at most 43% of the operand rows (worst case [48,20,20,20,1], k = 7: 4 networks, 6 warps)
  double* acc = reinterpret_cast<double*>(rows0);
  const int n_acc = tm_nets * P.n_params;
  for (int i = tid; i < n_acc; i += nt) acc[i] = 0.0;
  __syncthreads();
  {
    const int half = lane >> 4, l16 = lane & 15, og = l16 >> 2, ig = l16 & 3;
    for (int qw = 0; qw < nw; ++qw) {
      if (warp == qw) {
        for (int n = 0; n < tm_nets; ++n) {
          double* pn = acc + (size_t)n * P.n_params;
          const uint32_t tmn = tmw + (uint32_t)(n * tm_per_net);
          if (inline_dw1) {
            float v[GSI];
            TmIo<GSI>::ld(tmn, v);
#pragma unroll
            for (int p = 0; p < GSI; ++p) {
              const int e = 2 * p + half;
              if (e >= TQ * 3) continue;
              const int j = e / 3, i = e - j * 3, col = 4 * i + ig;
              if (col < d_r) pn[P.gw_off[0] + (4 * j + og) * d_r + col] += (double)v[p];
            }
          } else {
            for (int c = 0; c < n_chunks1; ++c) {
              float v[GS1];
              TmIo<GS1>::ld(tmn + c * GS1, v);
#pragma unroll
              for (int p = 0; p < GS1; ++p) {
                const int e = 2 * p + half;
                if (e >= TQ * CI1) continue;
                const int j = e / CI1, i = e - j * CI1, col = c * CW + CI1 * ig + i;
                if (col < d_r) pn[P.gw_off[0] + (4 * j + og) * d_r + col] += (double)v[p];
              }
            }
          }
          for (int l = 2; l <= NH; ++l) {
            float v[GSH];
            TmIo<GSH>::ld(tmn + tm_hid + (l - 2) * GSH, v);
#pragma unroll
            for (int p = 0; p < GSH; ++p) {
              const int e = 2 * p + half;
              if (e >= TQ * TQ) continue;
              const int j = e / TQ, i = e - j * TQ;
              pn[P.gw_off[l - 1] + (4 * j + og) * H + 4 * i + ig] += (double)v[p];
            }
          }
          {
            float v[1];
            TmIo<1>::ld(tmn + tm_sing, v);
            if (lane < H) pn[P.gw_off[NH] + lane] += (double)v[0];
            else if (lane == H) pn[P.gb_off[NH]] += (double)v[0];
            for (int l = NH; l >= 1; --l) {
              TmIo<1>::ld(tmn + tm_sing + 1 + (NH - l), v);
              if (lane < H) pn[P.gb_off[l - 1] + lane] += (double)v[0];
            }
          }
        }
      }
      __syncthreads();
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_slot), "r"(512u) : "memory");
  double* cta_part = P.part + (size_t)blockIdx.x * nw * n_part;
  for (int i = tid; i < n_part; i += nt) {
    double sacc = 0.0;
    if (i < n_acc) sacc = acc[i];
    else
      for (int q = 0; q < nw; ++q) sacc += __ldcg(cta_part + (size_t)q * n_part + i);
    cta_part[i] = sacc;
  }
}

// ------------------------------------------------------------------------------------------------ host side
struct Shape {
  int H, NH;
};

static size_t pass1_smem_bytes(int k, int img_floats, int geo_floats, int tile_rows) {
  return ((size_t)k * img_floats + geo_floats + (size_t)tile_rows * kP1Frames) * sizeof(float);
}
// Pass 2a forms the first layer's weight gradient itself when the input is at most 12 wide (2-d / 3-d model systems): r and
// vhat then stay in 24 rows of their own behind the X rows, and pass 2b (one 12-column group for 5 of 32 lanes) is not launched.
static bool pass2_inline_dw1(int drp) { return drp == 12; }
static int pass2_rows_per_warp(int drp, int H, int NH) {
  // Z rows (A_l | T_l of every layer; later two double-buffered chunks of r | vhat rows for dW_1) followed by the X rows;
  // the staging of layer 1 (r, u, Jacobian vectors) may overlap the X rows, which are not in use yet
  const int z = 2 * NH * H > 4 * dw1_chunk_of(drp) ? 2 * NH * H : 4 * dw1_chunk_of(drp);
  const int need = z + 2 * H, stage = 2 * drp + 12;
  return (need > stage ? need : stage) + (pass2_inline_dw1(drp) ? 2 * drp : 0);
}
static size_t pass2_smem_bytes(int k, int img2_floats, int geo_floats, int drp, int H, int NH, int warps) {
  const int n_comb = 3 * k + k * k;
  return ((size_t)k * img2_floats + geo_floats) * sizeof(float) + (size_t)(n_comb + (n_comb & 1)) * sizeof(double) +
         (size_t)warps * pass2_rows_per_warp(drp, H, NH) * kRowPad * sizeof(float);
}
// most warps (<= 8) whose operand rows fit next to the weights; 0 if fewer than kP2MinWarps fit
static int pass2_warps(int k, int img2_floats, int geo_floats, int drp, int H, int NH) {
  for (int wv = kP2MaxWarps; wv >= kP2MinWarps; --wv)
    if (pass2_smem_bytes(k, img2_floats, geo_floats, drp, H, NH, wv) <= (size_t)max_smem_optin()) return wv;
  return 0;
}
// image sizes without the template (same arithmetic as Img<H, NH>)
static int img2_floats_of(int H, int NH, int drp) { return drp * H + H + (NH - 1) * (H * H + H) + H + 4 + (NH - 1) * H * H; }
static int img_floats_of(int H, int NH, int drp) { return img2_floats_of(H, NH, drp) + H * drp; }

// kind 2
static int n_adj_of(const int* c) { return 3 * c[0] + 2 * c[1] + 3 * c[2] + 4 * c[3]; }
static int n_st_of(const int* c, int n_self) {
  const int cap = c[1] + c[2] + c[3];
  return kStBond * c[1] + kStAngle * c[2] + kStDihedral * c[3] + (n_self < 0 ? 0 : n_self > cap ? cap : n_self);
}
static bool prep_feat_bulk_ok(int n_atoms, const void* x) {
  const int fl = 3 * n_atoms;
  int g = fl, b = 32;
  while (b) {
    const int r = g % b;
    g = b, b = r;
  }
  return g <= 2 && ((uintptr_t)x & 15) == 0;   // gcd(fl, 32): lanes reading the same coordinate are at most 2 deep in a bank
}
static size_t prep_feat_smem_bytes(int groups, int n_atoms, int n_feat) {
  const int S = (3 * n_atoms) | 1;   // the larger of the two row strides
  return (size_t)(32 + kFinfoInts * n_feat + (size_t)groups * ((32 * S + 3) & ~3)) * sizeof(float);
}
static int prep_feat_groups(int n_atoms, int n_feat) {
  for (int g = 4; g >= 1; --g)
    if (prep_feat_smem_bytes(g, n_atoms, n_feat) <= (size_t)max_smem_optin()) return g;
  return 0;
}
static int n_shared_of(const cvf_preproc* pp) {
  const int v = pp->n_shared_atoms;
  return v < 0 ? 0 : v > pp->n_used ? pp->n_used : v;
}
static int jjt_warps_per_net(int k) { return k <= 3 ? 4 : k <= 6 ? 2 : 1; }   // at most 12 warps per CTA
static size_t jjt_smem_bytes(int k, int d_r, int n_shared, int n_feat, int n_adj, int n_st) {
  const int W = jjt_warps_per_net(k), cap = n_adj > 0 ? n_adj : 1;
  return (size_t)(((n_shared + 1 + 3) & ~3) + ((n_shared + 3) & ~3) + ((n_feat + 1 + 3) & ~3)) * 4 + (size_t)(2 * cap + n_feat) * 16 +
         (size_t)((3 * n_shared + 3) & ~3) * 4 + (size_t)(n_st + kStConstRows) * 32 * 4 + (size_t)k * (d_r + 3 * n_shared + W) * 32 * 4;
}

static bool supported_shape(const NetPlan& np, Shape* s) {
  s->H = s->NH = 0;
  if (np.L < 2) return false;
  const int H = np.dims[1];
  for (int l = 1; l < np.L; ++l)
    if (np.dims[l] != H) return false;
  if (np.dims[np.L] != 1) return false;
  for (int l = 0; l < np.L - 1; ++l)
    if (np.act[l] != CVF_ACT_TANH) return false;   // the thread-private kernels are tanh-only
  s->H = H, s->NH = np.L - 1;
  return (H == 20 && (s->NH == 3 || s->NH == 2)) || (H == 32 && s->NH == 3) || (H == 16 && s->NH == 3);
}

}  // namespace fast

// Whether the fast path covers this task; fills the byte count of its scratch (0 otherwise).
bool fast_eigen_supported(const cvf_preproc* pp, const NetPlan& np, int k) {
  fast::Shape s;
  if (!fast::supported_shape(np, &s)) return false;
  if (k < 1 || k > kMaxK) return false;
  int d_r, tile_rows;
  const size_t cap = (size_t)max_smem_optin();
  if (pp->kind == 0) {
    d_r = tile_rows = pp->dim;
  } else if (pp->kind == 1 && pp->n_align == 0) {
    // feature map on the raw frame (kind 2 of the plan): the host-side record counts must be filled in
    const int* c = pp->n_feat_by_type;
    if (pp->n_feat < 1 || c[0] + c[1] + c[2] + c[3] != pp->n_feat || !pp->feat || !pp->used_atoms || pp->n_used < 1) return false;
    if (c[0] * 3 + c[1] + c[2] + c[3] * 2 != pp->d_r) return false;
    d_r = tile_rows = pp->d_r;
    if (fast::prep_feat_groups(pp->n_atoms, pp->n_feat) == 0) return false;
    if (fast::jjt_smem_bytes(k, d_r, fast::n_shared_of(pp), pp->n_feat, fast::n_adj_of(c), fast::n_st_of(c, pp->n_self_records)) > cap) return false;
  } else if (pp->kind == 1) {
    if (!pp->positions_only || !pp->used_identity || pp->n_align < 3 || pp->diag != nullptr || pp->n_used != pp->n_atoms) return false;
    d_r = 3 * pp->n_atoms;
    tile_rows = (d_r + 11) / 12 * 12;
  } else {
    return false;
  }
  if (d_r < 1) return false;
  const int drp = (d_r + 11) / 12 * 12, geo = fast::geo_floats_of(drp);
  return fast::pass1_smem_bytes(k, fast::img_floats_of(s.H, s.NH, drp), geo, tile_rows) <= cap &&
         fast::pass2_warps(k, fast::img2_floats_of(s.H, s.NH, drp), geo, drp, s.H, s.NH) > 0;
}

namespace fast {

static inline long long round_up(long long v, long long m) { return (v + m - 1) / m * m; }

template <int H, int NH>
static size_t plan_scratch(FastPlan* P, const cvf_preproc* pp, const NetPlan& np, int k, long long B, void* workspace) {
  typedef Img<H, NH> I;
  P->k = k;
  P->kind = pp->kind == 1 && pp->n_align == 0 ? 2 : pp->kind;
  P->d_r = P->kind == 0 ? pp->dim : P->kind == 2 ? pp->d_r : 3 * pp->n_atoms;
  P->d_rp = (int)round_up(P->d_r, 12);
  P->tile_rows = P->kind == 1 ? P->d_rp : P->d_r;
  P->n_atoms = pp->kind == 1 ? pp->n_atoms : 0;
  P->n_align = pp->kind == 1 ? pp->n_align : 0;
  P->n_used = P->n_feat = P->n_st = P->n_adj = P->n_self = P->n_shared = 0;
  P->used_atoms = P->feat = nullptr;
  if (P->kind == 2) {
    P->n_used = pp->n_used, P->n_feat = pp->n_feat;
    P->n_self = pp->n_self_records < 0 ? 0 : pp->n_self_records;
    P->n_shared = n_shared_of(pp);
    P->n_st = n_st_of(pp->n_feat_by_type, pp->n_self_records), P->n_adj = n_adj_of(pp->n_feat_by_type);
    P->used_atoms = pp->used_atoms, P->feat = pp->feat;
  }
  P->img_floats = I::floats(P->d_rp);
  P->img2_floats = I::p2_floats(P->d_rp);
  P->geo_floats = geo_floats_of(P->d_rp);
  P->n_params = np.n_params;
  for (int l = 0; l < np.L; ++l) P->gw_off[l] = np.gw_off[l], P->gb_off[l] = np.gb_off[l];
  P->B = B;
  P->Bp = round_up(B, kP1Frames);
  P->align_idx = pp->kind == 1 ? pp->align_used : nullptr;   // used_identity: positions in used_atoms are atom indices
  P->ref = pp->ref;
  P->diag = pp->diag;
  char* base = (char*)workspace;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    char* p = base ? base + off : nullptr;
    off += (bytes + 255) & ~(size_t)255;
    return p;
  };
  const int n_part = k * np.n_params > 1 + 2 * k + k * k ? k * np.n_params : 1 + 2 * k + k * k;
  P->part = (double*)take((size_t)sm_count() * kP2MaxWarps * n_part * sizeof(double));
  P->img = (float*)take(((size_t)k * P->img_floats + P->geo_floats) * sizeof(float));
  P->Y = (float*)take((size_t)P->d_rp * P->Bp * sizeof(float));
  P->Kinv = (float*)take((size_t)6 * P->Bp * sizeof(float));
  P->U = (float*)take((size_t)k * P->d_rp * P->Bp * sizeof(float));
  P->A = (float*)take((size_t)k * NH * H * P->Bp * sizeof(float));
  P->JQ = (float*)take((size_t)k * 12 * P->Bp * sizeof(float));
  P->Dq = (float*)take((size_t)k * P->Bp * sizeof(float));
  P->Ys = (float*)take((size_t)k * P->Bp * sizeof(float));
  P->tab = nullptr, P->ST = nullptr;
  if (P->kind == 2) {
    P->tab = (int*)take((size_t)tab_ints(P->n_feat, P->n_used, P->n_adj) * sizeof(int));
    P->ST = (float*)take((size_t)(P->n_st > 0 ? P->n_st : 1) * P->Bp * sizeof(float));
  }
  return off;
}

template <int H, int NH>
static int run_forward(const FastPlan& P, const float* x, const float* params, float* y_out, cudaStream_t stream) {
  CVF_LAUNCH(K_FAST_PACK, stream, pack_kernel<H, NH><<<P.k + 1 + (P.kind == 2 ? 1 : 0), 256, 0, stream>>>(P, params));
  CVF_CUDA(cudaGetLastError());
  if (P.kind == 2) {
    const int ng = prep_feat_groups(P.n_atoms, P.n_feat);
    const size_t smem = prep_feat_smem_bytes(ng, P.n_atoms, P.n_feat);
    CVF_CUDA(cudaFuncSetAttribute(prep_feat_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const long long n_tiles = P.Bp / 32;
    long long grid = sm_count();
    if ((n_tiles + ng - 1) / ng < grid) grid = (n_tiles + ng - 1) / ng;
    CVF_LAUNCH(K_FAST_PREP, stream,
               prep_feat_kernel<<<(int)grid, 128 * ng, smem, stream>>>(P, x, prep_feat_bulk_ok(P.n_atoms, x) ? 1 : 0));
  } else if (P.kind == 1) {
    const size_t smem = (size_t)(128 * ((3 * P.n_atoms) | 1) + 6 * 128) * sizeof(float) + (size_t)P.n_align * (3 * sizeof(double) + sizeof(int)) + 3 * sizeof(double);
    CVF_CUDA(cudaFuncSetAttribute(prep_align_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    long long per_sm = (long long)(228 * 1024) / (long long)(smem + 1024);
    per_sm = per_sm < 1 ? 1 : per_sm > 6 ? 6 : per_sm;
    long long grid = (long long)sm_count() * per_sm;
    if (P.Bp / 128 < grid) grid = P.Bp / 128;
    const int bulk = ((uintptr_t)x & 15) == 0 ? 1 : 0;   // 128 frames are 128 * 12 N bytes: always a multiple of 16
    CVF_LAUNCH(K_FAST_PREP, stream, prep_align_kernel<<<(int)grid, 128, smem, stream>>>(P, x, bulk));
  } else {
    long long grid = (long long)sm_count() * 8;
    if ((P.Bp + 255) / 256 < grid) grid = (P.Bp + 255) / 256;
    CVF_LAUNCH(K_FAST_PREP, stream, prep_transpose_kernel<<<(int)grid, 256, 0, stream>>>(P, x));
  }
  CVF_CUDA(cudaGetLastError());
  const size_t smem1 = pass1_smem_bytes(P.k, P.img_floats, P.geo_floats, P.tile_rows);
  if (smem1 > (size_t)max_smem_optin()) {
    set_error("fast eigen path: pass 1 needs %zu B of shared memory", smem1);
    return CVF_E_UNSUPPORTED;
  }
  CVF_CUDA(cudaFuncSetAttribute(pass1_kernel<H, NH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem1));
  long long grid = sm_count();
  const long long n_tiles1 = P.Bp / kP1Frames;
  const int split1 = n_tiles1 * P.k <= grid ? 1 : 0;      // fewer (tile, network) pairs than SMs: one pair per CTA
  if ((split1 ? n_tiles1 * P.k : n_tiles1) < grid) grid = split1 ? n_tiles1 * P.k : n_tiles1;
  CVF_LAUNCH(K_FAST_PASS1, stream, pass1_kernel<H, NH><<<(int)grid, kP1Threads, smem1, stream>>>(P, y_out, split1));
  CVF_CUDA(cudaGetLastError());
  if (P.kind == 2) {
    const int W = jjt_warps_per_net(P.k);
    const size_t smemj = jjt_smem_bytes(P.k, P.d_r, P.n_shared, P.n_feat, P.n_adj, P.n_st);
    CVF_CUDA(cudaFuncSetAttribute(jjt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemj));
    long long per_sm = (long long)(228 * 1024) / (long long)(smemj + 1024);
    if (per_sm < 1) per_sm = 1;
    if (per_sm > 64 / (P.k * W)) per_sm = 64 / (P.k * W);
    if (per_sm < 1) per_sm = 1;
    long long gj = (long long)sm_count() * per_sm;
    if (P.Bp / 32 < gj) gj = P.Bp / 32;
    CVF_LAUNCH(K_FAST_JJT, stream, jjt_kernel<<<(int)gj, 32 * P.k * W, smemj, stream>>>(P, W));
    CVF_CUDA(cudaGetLastError());
  }
  return 0;
}

template <int H, int NH>
static int run_stats(const cvf_preproc* pp, const NetPlan& np, int k, const float* x, const float* w, long long B,
                     const float* params, float* y_out, double* stats_out, void* workspace, size_t ws_bytes, cudaStream_t stream) {
  FastPlan P;
  const size_t need = plan_scratch<H, NH>(&P, pp, np, k, B, workspace);
  if (need > ws_bytes) {
    set_error("workspace too small: %zu < %zu", ws_bytes, need);
    return CVF_E_WORKSPACE;
  }
  int e = run_forward<H, NH>(P, x, params, y_out, stream);
  if (e) return e;
  const int ns = 1 + 2 * k + k * k;
  long long grid = (long long)sm_count() * 2;
  if ((B + 255) / 256 < grid) grid = (B + 255) / 256;
  switch (k) {
#define CVF_STATS_CASE(K_) \
  case K_:                 \
    CVF_LAUNCH(K_FAST_STATS, stream, stats_kernel<K_><<<(int)grid, 256, 0, stream>>>(P, w, P.part)); \
    break;
    CVF_STATS_CASE(1)
    CVF_STATS_CASE(2)
    CVF_STATS_CASE(3)
    CVF_STATS_CASE(4)
    CVF_STATS_CASE(5)
    CVF_STATS_CASE(6)
    CVF_STATS_CASE(7)
    CVF_STATS_CASE(8)
#undef CVF_STATS_CASE
    default:
      set_error("fast eigen path: k = %d", k);
      return CVF_E_UNSUPPORTED;
  }
  CVF_CUDA(cudaGetLastError());
  CVF_LAUNCH(K_REDUCE, stream, reduce_partials_kernel<<<(ns + 127) / 128, 128, 0, stream>>>(P.part, (int)grid, ns, 0, ns, stats_out));
  CVF_CUDA(cudaGetLastError());
  return 0;
}

template <int H, int NH>
static int run_grad(const cvf_preproc* pp, const NetPlan& np, int k, const float* x, const float* w, long long B,
                    const float* params, const double* combine, const float* seed_extra, double* grad_out, void* workspace,
                    size_t ws_bytes, int scratch_valid, cudaStream_t stream) {
  FastPlan P;
  const size_t need = plan_scratch<H, NH>(&P, pp, np, k, B, workspace);
  if (need > ws_bytes) {
    set_error("workspace too small: %zu < %zu", ws_bytes, need);
    return CVF_E_WORKSPACE;
  }
  if (!scratch_valid) {
    int e = run_forward<H, NH>(P, x, params, nullptr, stream);
    if (e) return e;
  }
  const int nw = pass2_warps(k, P.img2_floats, P.geo_floats, P.d_rp, H, NH);
  if (nw == 0) {
    set_error("fast eigen path: pass 2 does not fit shared memory");
    return CVF_E_UNSUPPORTED;
  }
  const size_t smem2 = pass2_smem_bytes(k, P.img2_floats, P.geo_floats, P.d_rp, H, NH, nw);
  if ((size_t)3 * np.n_params * sizeof(double) > (size_t)nw * pass2_rows_per_warp(P.d_rp, H, NH) * kRowPad * sizeof(float)) {
    // a floor, not the exact fold size: up to kMaxK networks keep totals in TMEM, and the fold of pass2_kernel fits the rows of
    // every supported shape (its comment)
    set_error("fast eigen path: the operand rows cannot hold the CTA's gradient vector");
    return CVF_E_UNSUPPORTED;
  }
  const long long n_tiles = P.Bp / 32;
  long long grid = sm_count();
  // small batches: (tile, network) pairs as work items, so that every warp of the chip gets at most two of them
  const int split2 = n_tiles * k <= 2 * grid * nw ? 1 : 0;
  const long long n_items2 = split2 ? n_tiles * k : n_tiles;
  if ((n_items2 + nw - 1) / nw < grid) grid = (n_items2 + nw - 1) / nw;
  if (dw1_chunk_of(P.d_rp) == 28) {
    CVF_CUDA(cudaFuncSetAttribute(pass2_kernel<H, NH, 28>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2));
    CVF_LAUNCH(K_FAST_PASS2A, stream, pass2_kernel<H, NH, 28><<<(int)grid, 32 * nw, smem2, stream>>>(P, w, combine, pass2_rows_per_warp(P.d_rp, H, NH), seed_extra, split2));
  } else {
    CVF_CUDA(cudaFuncSetAttribute(pass2_kernel<H, NH, 24>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2));
    CVF_LAUNCH(K_FAST_PASS2A, stream, pass2_kernel<H, NH, 24><<<(int)grid, 32 * nw, smem2, stream>>>(P, w, combine, pass2_rows_per_warp(P.d_rp, H, NH), seed_extra, split2));
  }
  CVF_CUDA(cudaGetLastError());
  const int n_part = k * np.n_params;
  CVF_LAUNCH(K_REDUCE, stream, reduce_partials_kernel<<<(n_part + 127) / 128, 128, 0, stream>>>(P.part, (int)grid, nw * n_part, 0, n_part, grad_out));
  CVF_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace fast

#define CVF_FAST_DISPATCH(CALL, ...)                                   \
  do {                                                                 \
    fast::Shape s_;                                                    \
    fast::supported_shape(np, &s_);                                    \
    if (s_.H == 20 && s_.NH == 3) return fast::CALL<20, 3>(__VA_ARGS__); \
    if (s_.H == 20 && s_.NH == 2) return fast::CALL<20, 2>(__VA_ARGS__); \
    if (s_.H == 32 && s_.NH == 3) return fast::CALL<32, 3>(__VA_ARGS__); \
    if (s_.H == 16 && s_.NH == 3) return fast::CALL<16, 3>(__VA_ARGS__); \
  } while (0)

size_t fast_eigen_workspace_bytes(const cvf_preproc* pp, const NetPlan& np, int k, long long B) {
  fast::FastPlan P;
  fast::Shape s_;
  fast::supported_shape(np, &s_);
  if (s_.H == 20 && s_.NH == 3) return fast::plan_scratch<20, 3>(&P, pp, np, k, B, nullptr);
  if (s_.H == 20 && s_.NH == 2) return fast::plan_scratch<20, 2>(&P, pp, np, k, B, nullptr);
  if (s_.H == 32 && s_.NH == 3) return fast::plan_scratch<32, 3>(&P, pp, np, k, B, nullptr);
  if (s_.H == 16 && s_.NH == 3) return fast::plan_scratch<16, 3>(&P, pp, np, k, B, nullptr);
  return 0;
}

int fast_eigen_stats(const cvf_preproc* pp, const NetPlan& np, int k, const float* x, const float* w, long long B,
                     const float* params, float* y_out, double* stats_out, void* workspace, size_t ws_bytes, cudaStream_t stream) {
  CVF_FAST_DISPATCH(run_stats, pp, np, k, x, w, B, params, y_out, stats_out, workspace, ws_bytes, stream);
  set_error("fast eigen path: shape not instantiated");
  return CVF_E_UNSUPPORTED;
}

int fast_eigen_grad(const cvf_preproc* pp, const NetPlan& np, int k, const float* x, const float* w, long long B,
                    const float* params, const double* combine, const float* seed_extra, double* grad_out, void* workspace,
                    size_t ws_bytes, int scratch_valid, cudaStream_t stream) {
  CVF_FAST_DISPATCH(run_grad, pp, np, k, x, w, B, params, combine, seed_extra, grad_out, workspace, ws_bytes, scratch_valid, stream);
  set_error("fast eigen path: shape not instantiated");
  return CVF_E_UNSUPPORTED;
}

}  // namespace cvf
