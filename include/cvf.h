/*
 * cvf.h -- C ABI of libcvf_sm100.so: the colvars-finder training step on B200 (sm_100a).
 *
 * The reference (zwpku/colvars-finder) has no native layer and no FFI; its boundary for this path is
 * the Python class API (colvarsfinder/core.py, nn.py).  This header is the thin C boundary that the
 * Python drop-in (colvars-finder_b200/colvarsfinder) binds with ctypes.  Each entry point names the
 * reference code it replaces.  INTEGRATION.md shows the binding.
 *
 * Conventions
 *   - all data pointers are DEVICE pointers owned by the caller (PyTorch's caching allocator); the
 *     library allocates nothing on the device.  The compute entry points keep no state between calls; the only process-wide
 *     state is the three testing switches (cvf_eigen_set_path, cvf_ae_set_fast_path, cvf_ae_set_wide_path: atomic ints, read
 *     once per call) and the launch accounting of cvf_profile_* (mutex-protected; meant for one profiling thread);
 *   - the descriptor structs (cvf_preproc, cvf_mlp) are HOST structs passed by pointer; the index /
 *     coefficient arrays they point to live on the device;
 *   - every call only enqueues work on `stream` (a cudaStream_t passed as void*); no hidden sync;
 *   - return value: 0 = ok, >0 = cudaError_t, <0 = argument error (CVF_E_*); never throws.
 *     cvf_last_error_string() describes the last non-zero return of the calling thread;
 *   - fp32 frames / parameters; batch sums and gradient sums are accumulated and returned in fp64.
 */
#ifndef CVF_H
#define CVF_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CVF_VERSION 100
#define CVF_MAX_LAYERS 8   /* linear layers per network chain (AutoEncoder: encoder + decoder) */
#define CVF_MAX_K 8        /* eigenfunctions per model */

#define CVF_E_ARG (-1)        /* null pointer / negative size / inconsistent descriptor */
#define CVF_E_UNSUPPORTED (-2) /* outside the supported envelope (depth, width, shared memory) */
#define CVF_E_WORKSPACE (-3)  /* workspace too small */

/* feature record types (molann-style features used by examples/dipeptide/main.ipynb:335-337) */
#define CVF_FEAT_POSITION 0   /* 1 atom  -> 3 outputs (aligned x,y,z) */
#define CVF_FEAT_BOND 1       /* 2 atoms -> |y_b - y_a| */
#define CVF_FEAT_ANGLE 2      /* 3 atoms -> cos of the angle at the middle atom */
#define CVF_FEAT_DIHEDRAL 3   /* 4 atoms -> (cos phi, sin phi) */

/* Pre-processing layer r(x): the caller-supplied `pp_layer` of core.py:65,122,403,635
 * (torch.nn.Identity in examples/2d/2d.ipynb:485; alignment + features in examples/dipeptide/main.ipynb:335-348). */
typedef struct cvf_preproc {
  int32_t kind;               /* 0: identity on a flat [B,dim] input; 1: molecular [B,n_atoms,3] input */
  int32_t dim;                /* kind 0: input dimension d (= d_r) */
  int32_t n_atoms;            /* kind 1: atoms per frame */
  int32_t n_used;             /* kind 1: atoms read by alignment or features */
  const int32_t* used_atoms;  /* [n_used] atom index inside the frame */
  int32_t n_align;            /* 0 = no alignment */
  const int32_t* align_used;  /* [n_align] positions in used_atoms of the alignment atoms */
  const float* ref;           /* [n_align,3] reference positions, centred */
  int32_t n_feat;             /* feature records */
  const int32_t* feat;        /* [n_feat,5]: type, then up to 4 positions in used_atoms */
  int32_t d_r;                /* output dimension of r */
  int32_t positions_only;     /* 1: feat is exactly POSITION of used atom 0,1,..,n_used-1 (d_r = 3 n_used), so
                                 r is the aligned frame itself and the kernels skip the feature copy */
  int32_t used_identity;      /* 1: used_atoms is 0,1,..,n_atoms-1 (every atom is read, in order) */
  const float* diag;          /* diag_coeff (core.py:348-354) gathered to [n_used*3] (kind 1) or [dim] (kind 0); NULL = ones */
  int32_t n_feat_by_type[4];  /* records of each CVF_FEAT_* type in feat (host-side counts: they size the scratch of the
                                 feature-Jacobian kernel, whose per-frame gradient stencils take 3 / 6 / 14 floats per
                                 bond / angle / dihedral) */
  int32_t n_self_records;     /* bond / angle / dihedral records with at least one atom that no other record reads (an atom
                                 read by a POSITION record never counts): their contribution through those atoms is a per-frame
                                 scalar ("self term") that the feature-Jacobian kernel keeps as one more stencil row.  Sizing
                                 hint only: a smaller value costs speed, not correctness; a larger one costs scratch */
  int32_t n_shared_atoms;     /* used atoms read by more than one record or by a POSITION record: the atoms whose gradient the
                                 feature-Jacobian kernel accumulates across records (sizes its shared memory; the kernel checks
                                 the value against the record list and poisons its output with NaN if it is too small) */
} cvf_preproc;

/* Linear+activation chain built by nn.create_sequential_nn (nn.py:29-59).  For nn.AutoEncoder the
 * chain is encoder followed by decoder (nn.py:114). */
/* activation after a layer (nn.py:29-59 takes any torch.nn.Module; these are the ones whose first and second derivatives are
 * functions of the activation's output, which is all the kernels keep).  One kind per chain, as in the reference (the same module
 * instance follows every layer but the last).  The thread-private / tensor-core kernels are tanh-only; other kinds run on the
 * general kernels. */
#define CVF_ACT_NONE 0
#define CVF_ACT_TANH 1
#define CVF_ACT_SIGMOID 2
#define CVF_ACT_SOFTPLUS 3   /* beta = 1 */
#define CVF_ACT_ELU 4        /* alpha = 1 */
#define CVF_ACT_RELU 5
typedef struct cvf_mlp {
  int32_t n_layers;
  int32_t dims[CVF_MAX_LAYERS + 1];
  int32_t act[CVF_MAX_LAYERS];   /* CVF_ACT_* after this layer */
} cvf_mlp;

int cvf_version(void);
/* hash of the sources this binary was compiled from (csrc/, include/cvf.h, compile flags), stamped by __graft_entry__.build();
 * "unstamped" for a build made by hand */
const char* cvf_source_hash(void);
const char* cvf_last_error_string(void);
/* sizeof(cvf_preproc) / sizeof(cvf_mlp) as this library was compiled: lets a binding check its own struct layout */
size_t cvf_sizeof_preproc(void);
size_t cvf_sizeof_mlp(void);

/* number of float parameters of one chain, in torch's parameters() order: W1[out,in], b1[out], W2, b2, ... */
int64_t cvf_mlp_param_count(const cvf_mlp* net);

/* Kabsch alignment of every frame onto the reference (the alignment half of pp_layer; no reference
 * source -- molann.ann.AlignmentLayer, examples/dipeptide/main.ipynb:345).
 * x [B,n_atoms,3] -> y [B,n_atoms,3];  optional R_out [B,9] (row-major, y=(x-c)R) and c_out [B,3]. */
int cvf_align_fwd(const float* x, int64_t B, int32_t n_atoms, const int32_t* align_idx, int32_t n_align,
                  const float* ref_centred, float* y_out, float* R_out, float* c_out, void* stream);

/* Whole-trajectory pre-pass of AutoEncoderTask.__init__ (core.py:635): r_out[B,d_r] = pp(x). */
int cvf_features_fwd(const float* x, int64_t B, const cvf_preproc* pp, float* r_out, void* stream);

/* Vector-Jacobian products of the two calls above: the autograd backward of utils.Align / FeatureMap / Preprocessing, which
 * replaces the backward of molann's alignment and feature layers that torch.autograd.grad(y, X) runs at core.py:424.
 * First order only.  The rotation is recomputed from x (the forward keeps nothing).
 * cvf_align_vjp:    g_y [B,n_atoms,3] = dg/dy  ->  g_x [B,n_atoms,3] = dg/dx; same arguments and checks as cvf_align_fwd.
 * cvf_features_vjp: g_r [B,d_r] = dg/dr  ->  g_x [B,n_atoms,3] = dg/dx for a kind-1 descriptor, with or without alignment;
 *                   atoms that no record reads get exact zeros. */
int cvf_align_vjp(const float* x, int64_t B, int32_t n_atoms, const int32_t* align_idx, int32_t n_align,
                  const float* ref_centred, const float* g_y, float* g_x, void* stream);
int cvf_features_vjp(const float* x, int64_t B, const cvf_preproc* pp, const float* g_r, float* g_x, void* stream);

/* ---- EigenFunctionTask.loss_func, generator branch (core.py:387-457) split at its batch sums ---- */

/* doubles in the stats vector: S0, S1[k], S2[k*k], SD[k] */
int32_t cvf_eigen_num_stats(int32_t k);
/* doubles in the combine vector: loss, obj, pen, eig[k] (sorted), cvec[k], mean[k], cD[k], C2[k*k], a0[k].
 * The last four blocks are the coefficients of pass 2: for frame f and network i the seed d loss / d y_i is
 * w_f (a0_i + sum_j C2_ij (y_j - mean_j)) and the Dirichlet term enters with weight 2 w_f cD_i.  cvf_eigen_combine writes
 * a0 = 0 (its loss depends on S1, S2 only through central moments); a caller that differentiates another function of the
 * batch sums fills the vector itself (colvarsfinder/_ops.py: cvf::eigen_stats backward). */
int32_t cvf_eigen_num_combine(int32_t k);
/* bytes of scratch needed by cvf_eigen_stats / cvf_eigen_grad on a batch of B frames: per-CTA partial sums and, on the
 * fast path, the frame-minor intermediates pass 1 leaves for pass 2 (aligned frames, grad_r y, Jacobian vectors, hidden
 * activations: about 2 KB per frame for three [66,20,20,20,1] networks). */
size_t cvf_eigen_workspace_bytes(const cvf_preproc* pp, const cvf_mlp* net, int32_t k, int64_t B);
/* 1 if (pp, net, k) runs on the thread-private FFMA2 kernels (cvf_eigen_fast.cu), 0 if on the general row-engine kernels */
int cvf_eigen_path(const cvf_preproc* pp, const cvf_mlp* net, int32_t k);
/* testing / profiling switch: 0 = choose automatically (default), 1 = always the general kernels */
int cvf_eigen_set_path(int32_t mode);

/* Pass 1: y = model(pp(X)), grad_x y_i, Dirichlet densities; batch sums (core.py:403-410,424-426).
 * params [k * cvf_mlp_param_count] fp32.  y_out [k,B] fp32 (kept for pass 2).  stats_out fp64. */
int cvf_eigen_stats(const float* x, const float* w, int64_t B, const cvf_preproc* pp, const cvf_mlp* net,
                    int32_t k, const float* params, float* y_out, double* stats_out,
                    void* workspace, size_t workspace_bytes, void* stream);

/* After the cross-GPU sum of stats: loss, eigenvalues, cvec, objective, penalty (core.py:426-455) and
 * the per-frame seed coefficients of pass 2.  eig_w: HOST array [k]. */
int cvf_eigen_combine(const double* stats, int32_t k, double alpha, const double* eig_w, double beta,
                      int32_t sort, double* combine_out, void* stream);

/* Pass 2: d loss / d params (replaces loss.backward(), core.py:517).  grad_out [k * param_count] fp64,
 * summed over this rank's frames.  scratch_valid = 1 promises that `workspace` still holds what the cvf_eigen_stats
 * call on the SAME x, w, params left there (the normal loss -> backward sequence); 0 recomputes it. */
int cvf_eigen_grad(const float* x, const float* w, int64_t B, const cvf_preproc* pp, const cvf_mlp* net,
                   int32_t k, const float* params, const float* y_in, const double* combine, const float* seed_extra,
                   double* grad_out, void* workspace, size_t workspace_bytes, int32_t scratch_valid, void* stream);
/* seed_extra (NULL for the generator loss): [k,B] per-frame additions to d loss / d y_i, see the transfer-operator calls below */

/* ---- EigenFunctionTask.loss_func, transfer-operator branch (lag_tau > 0: core.py:412-416,428,440) ----
 * y = model(pp(X)) and y' = model(pp(X_lagged)) come from two cvf_eigen_stats calls (their SD entries are not used).
 * cvf_eigen_tlag_terms, extra_out == NULL: sx_out[i] = sum_f w_f (y'_i - y_i)^2 (workspace: >= 4 * SMs * k doubles);
 *                       extra_out != NULL: extra_out[i][f] = coef[i] w_f (y_i - y'_i), the seed_extra of the backward pass on X
 *                       (its negative is the seed_extra of the backward pass on X_lagged).
 * cvf_eigen_tlag_combine: loss, eigenvalues, cvec, objective, penalty (core.py:428-455, including the reference's pairing of
 *   numerator idx with denominator cvec[idx] at core.py:440) and the coefficient vectors of the two backward passes, both in the
 *   cvf_eigen_combine layout; combine_out carries k more doubles at its end, the coef[] of cvf_eigen_tlag_terms.
 *   tau = traj_dt * lag_idx;  eig_w: HOST array [k]. */
int cvf_eigen_tlag_terms(const float* y, const float* y_lag, const float* w, int64_t B, int32_t k, const double* coef,
                         double* sx_out, float* extra_out, void* workspace, size_t workspace_bytes, void* stream);
int cvf_eigen_tlag_combine(const double* stats, const double* stats_lag, const double* sx, int32_t k, double alpha,
                           const double* eig_w, double tau, int32_t sort, double* combine_out, double* combine_lag_out,
                           void* stream);

/* ---- AutoEncoderTask.weighted_MSE_loss + backward (core.py:652-666,708) ---- */
/* bytes of scratch for a batch of B frames.  Chains whose weights fit shared memory run in one fused kernel (per-CTA partial
 * sums only); wider ones run layer by layer as dense fp32 products over chunks of frames and keep the chunk's activations here. */
size_t cvf_ae_workspace_bytes(const cvf_mlp* net, int64_t B);
/* sums_out[2] = { sum_f w_f |dec(enc(F_f)) - F_f|^2 , sum_f w_f };  grad_out [param_count] fp64 holds the
 * gradient of the FIRST sum (not yet divided by sum w).  grad_out may be NULL (evaluation only). */
int cvf_ae_step(const float* feat, const float* w, int64_t B, const cvf_mlp* net, const float* params,
                double* sums_out, double* grad_out, void* workspace, size_t workspace_bytes, void* stream);

/* The same with a separate reconstruction target: sum_f w_f |dec(enc(F_f)) - T_f|^2 with T [B, d] (the time-lagged
 * autoencoder loss of RegAutoEncoderTask.weighted_MSE_loss, core.py:876-887, where T = pp(X_lagged)).  target == NULL or
 * target == feat is cvf_ae_step; otherwise the chain must fit shared memory (general kernel). */
int cvf_ae_step_target(const float* feat, const float* target, const float* w, int64_t B, const cvf_mlp* net,
                       const float* params, double* sums_out, double* grad_out, void* workspace, size_t workspace_bytes,
                       void* stream);

/* testing / profiling switch for chains that fit shared memory: 0 = the thread-private kernels (cvf_ae_fast.cu) when the chain
 * is encoder [d,20,20,20,e] + decoder [e,10,10,d], e = 1..3, d <= 72 (default); 1 = always the general row-engine kernel */
int cvf_ae_set_fast_path(int32_t mode);

/* Products of the layer-wise autoencoder path: 0 = tcgen05 tensor cores, fp32 operands split into two TF32 terms and three
 * products per block (hi*hi + lo*hi + hi*lo) accumulated in fp32 in tensor memory; 1 = fp32 SIMT (FFMA2). */
int cvf_ae_set_wide_path(int32_t mode);

/* ---- WeightedTrajectory's weight handling on the device (utils.py:140-169) ----
 * w [n] fp64 raw weights.  w is normalised to mean 1; states with min_w < w < max_w are kept; the kept weights are renormalised
 * to mean 1.  idx_out [n] receives the ascending indices of the kept states, w_out [n] their weights, *n_keep_out (device) their
 * number.  workspace: cvf_weights_filter_workspace_bytes(n). */
size_t cvf_weights_filter_workspace_bytes(int64_t n);
int cvf_weights_filter(const double* w, int64_t n, double min_w, double max_w, int64_t* idx_out, double* w_out,
                       int64_t* n_keep_out, void* workspace, size_t workspace_bytes, void* stream);

/* Launch accounting for bench.py (no reference counterpart).  The library counts every kernel it launches; with
 * cvf_profile_enable(1) each launch is also bracketed by CUDA events on the stream it was enqueued on.
 * cvf_profile_read fills, per kernel id < cvf_profile_num_kernels(): summed milliseconds of the timed launches, how many were
 * timed, and the launch count since the last reset; it synchronises on the recorded events. */
int cvf_profile_enable(int32_t on);
int32_t cvf_profile_num_kernels(void);
const char* cvf_profile_kernel_name(int32_t id);
int cvf_profile_read(double* ms_out, int64_t* timed_out, int64_t* launches_out, int32_t reset);

/* Measurement helper for bench.py (no reference counterpart): enqueue a kernel that issues exactly
 * *flops_out = 2 * fmas fp32 FMA flops on independent register chains, so that the fp32 SIMT peak used as the
 * compute-roofline denominator is measured on the same GPU, same clocks, as the step kernels. */
int cvf_fma_probe(float* sink, int32_t iters, double* flops_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CVF_H */
