/*
 * gpode.h -- C ABI of libgpode.so: the sparse-GP latent vector field of VAE-GP-ODE and its
 * fixed-step rollout, forward and backward, as hand-written CUDA for sm_100a (NVIDIA B200).
 *
 * The reference (IlzeAmandaA/VAE-GP-ODE) has no FFI: the path sits behind Python nn.Modules.  Each
 * entry point names the reference interface it replaces (paths relative to
 * experiments/model/ in the reference tree).  INTEGRATION.md shows the ctypes binding.
 *
 * Conventions
 *   - all tensors are fp32, row-major, contiguous DEVICE pointers owned by the caller; the library
 *     never allocates, frees or retains a pointer after the call returns;
 *   - every call only ENQUEUES work on `stream` (a cudaStream_t passed as void*; NULL = legacy default
 *     stream); no host synchronisation, no global mutable state, re-entrant;
 *   - return value: 0 ok; <0 argument/shape error (GPODE_E_*), never a silent fallback;
 *     >0 a cudaError_t raised by a launch.  No C++ exception crosses the ABI.
 */
#ifndef GPODE_H_
#define GPODE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GPODE_VERSION 211 /* major*100 + minor */

/* kernel variants (core/kernels.py: RBF dimwise=False / dimwise=True :29-195, DivergenceFreeKernel :201-393) */
enum { GPODE_RBF_SHARED = 0, GPODE_RBF_DIMWISE = 1, GPODE_DF = 2 };
/* torchdiffeq fixed-grid methods reachable through Flow(solver=...) (core/flow.py:49,78-85) */
enum { GPODE_EULER = 0, GPODE_MIDPOINT = 1, GPODE_RK4 = 2 /* 3/8 rule */ };

enum {
  GPODE_OK = 0,
  GPODE_E_NULL = -1,        /* a required pointer is NULL */
  GPODE_E_SHAPE = -2,       /* a size is non-positive or inconsistent (e.g. DF with D_in != D_out) */
  GPODE_E_UNSUPPORTED = -3, /* shape outside the compiled range (D_in > 16, DF D > 8, L > 65535, parameter tile > 227 KB ...) */
  GPODE_E_WORKSPACE = -4,   /* workspace / save buffer too small or misaligned */
  GPODE_E_ENUM = -5         /* unknown variant / method / order */
};

/*
 * One function sample of the GP per MC sample l = 0..L-1 -- what SVGP_Layer.build_cache() leaves
 * behind (core/svpy.py:103-121): Z, lengthscales and variance are shared by all samples, the
 * random-feature draws and nu are per sample.  Layouts are the reference's own, with a leading L.
 *
 *   variant            ell            var        eps / omega         phase           w               nu
 *   RBF_SHARED         (D_in)         (1)        (L,D_in,S)          (L,1,S)         (L,S,D_out)     (L,M,D_out)
 *   RBF_DIMWISE        (D_out,D_in)   (D_out)    (L,D_in,S,D_out)    (L,1,S,D_out)   (L,S,D_out)     (L,D_out,M,1)
 *   DF (D_in==D_out=D) (D,D)          (D)        (L,D,S,D)           (L,1,S,D)       (L,2S,D)        (L,M*D,1)
 *
 * `eps` are the standard-normal frequency draws; the kernels use omega = eps / ell exactly like
 * RBF.sample_freq (core/kernels.py:112-124), which is what carries the lengthscale gradient through
 * the random features.  `B` (DF only) is the state-independent operator B(omega) (L,S,D,D) of
 * DivergenceFreeKernel.rff_forward (core/kernels.py:327-336), hoisted to once per rollout.
 */
typedef struct GpodeProblem {
  int32_t variant;
  int32_t L;      /* MC samples (independent function samples), at most 65535: the launches put L on grid y / z */
  int32_t N;      /* states (trajectories) per sample */
  int32_t D_in;   /* GP input dim = ODE state dim (order 1: q, order 2: 2q) */
  int32_t D_out;  /* GP output dim */
  int32_t M;      /* inducing points */
  int32_t S;      /* random Fourier features */
  int32_t flags;  /* GPODE_FLAG_* (0 = defaults); replaces the environment switches of ABI 1.x */
  const float* Z;     /* (M,D_in) */
  const float* ell;
  const float* var;
  const float* eps;
  const float* phase;
  const float* w;
  const float* nu;
  const float* B;     /* DF only, else NULL */
} GpodeProblem;

/* Gradients w.r.t. the GpodeProblem tensors (same layouts).  Written (not accumulated).  Any pointer
 * may be NULL to skip that output.  No gradient exists for eps / phase / w: they are plain draws
 * in the reference (requires_grad=False).  d_ell holds the DIRECT dependence only (through K(x,Z)
 * and through omega = eps/ell); the dependence through nu and B is carried by d_nu / d_B. */
typedef struct GpodeParamGrads {
  float* d_Z;    /* (M,D_in), summed over samples */
  float* d_ell;  /* like ell, summed over samples */
  float* d_var;  /* like var, summed over samples */
  float* d_nu;   /* like nu (per sample) */
  float* d_B;    /* DF only: like B (per sample) */
} GpodeParamGrads;

int gpode_version(void);
const char* gpode_error_string(int code);
/* Kernel-selection flags (GpodeProblem.flags).  Shapes alone pick the kernels (each shape has exactly one default); these
 * flags exist for the parity tests and for A/B measurements and never change results beyond rounding:
 *   RBF variants at D_in > 8 and >= 32,768 states: */
#define GPODE_FLAG_FWD_MMA 1      /* forward sweep on the warp-level tensor path (mma.sync) instead of tcgen05 */
#define GPODE_FLAG_FWD_TCGEN05 2  /* forward sweep on tcgen05 even when its 256-unit operand tiles are > 15 % padding */
#define GPODE_FLAG_BWD_MMA 4      /* reverse sweep + separate parameter-gradient pass on the warp-level tensor path (mma.sync) */
#define GPODE_FLAG_BWD_TCGEN05 16 /* fused reverse sweep + parameter gradients on tcgen05 / tensor memory (rbf_bwd_tc.cuh): the default, the flag pins it */
/* (bit 8 is reserved.)  Parameter gradients are sums over all state evaluations accumulated with floating-point atomics, so their
 * last bits differ from run to run; tests/test_gpu_rbf.py::test_run_to_run_spread bounds the spread (<= 2e-6 of the gradient norm,
 * below the parity error against the fp64 oracle).  Trajectories, f and dL/dz0 involve no atomics and are bit-reproducible. */
/* Which forward-sweep kernel family gpode_field_fwd / gpode_rollout_fwd will launch for this problem (shapes and the flags
 * above decide; no CUDA call is made): */
#define GPODE_FWD_FFMA 0   /* FP32 / MUFU pipes (every D_in <= 8, small batches, the divergence-free kernel) */
#define GPODE_FWD_MMA 1    /* warp-level tensor path (mma.sync) */
#define GPODE_FWD_TCGEN05 2 /* tcgen05.mma with the accumulators in tensor memory */
int gpode_forward_kernel(const GpodeProblem* p);
/* Small batches (N * L <= 148 x 32 states -- the shapes the reference trains at): the sweep kernels give 32 states to a CTA of several
 * warps and split the work of an evaluation over a thread-block cluster (RBF: the output dimensions; divergence-free kernel: the rows
 * of every streamed chunk), all-gathering the results through distributed shared memory.  Returns the cluster size such a problem is
 * launched with (1 ... 8; 1 also for batches that fill the chip, where every state already has its own thread), < 0 on error.
 * Shapes decide; no CUDA call is made. */
int gpode_cluster_size(const GpodeProblem* p);

/* bytes of scratch the calls below need for this problem (T, method only matter for the rollout).
 * `workspace` must be 256-byte aligned and is clobbered by every call. */
size_t gpode_workspace_bytes(const GpodeProblem* p, int T, int method);
/* floats of the forward->backward save buffer of a rollout (stage inputs, stage derivatives, prior part) */
size_t gpode_rollout_save_floats(const GpodeProblem* p, int T, int method);

/* SVGP_Layer.forward (core/svpy.py:123-142) = kern.rff_forward + kern.f_update
 * (core/kernels.py:140-153,174-181 / 319-351,390-393) for every state of every sample.
 *   x (L,N,D_in) -> f (L,N,D_out); f_prior (L,N,D_out) receives the rff part (needed by the backward; may be NULL). */
int gpode_field_fwd(const GpodeProblem* p, const float* x, float* f, float* f_prior,
                    void* workspace, size_t workspace_bytes, void* stream);

/* autograd backward of SVGP_Layer.forward (implicit in the reference: loss.backward(), main.py:210).
 *   g = dL/df (L,N,D_out), f / f_prior as returned by gpode_field_fwd -> dx (L,N,D_in) and the parameter gradients. */
int gpode_field_bwd(const GpodeProblem* p, const float* x, const float* g, const float* f,
                    const float* f_prior, float* dx, const GpodeParamGrads* grads,
                    void* workspace, size_t workspace_bytes, void* stream);

/* Flow.forward = torchdiffeq.odeint(ODEfunc, z0, ts, method) on the fixed grid ts, for all L samples
 * in one launch (core/flow.py:30-45,68-86; core/odegpvae.py:37-45).
 *   z0 (N,D_in) if z0_per_sample == 0 (the reference feeds every sample the same z0), else (L,N,D_in);
 *   ts (T) fp32 on the device; order 1: dz = f(z); order 2: dz = [z[q:], f(z)] with q = D_out, D_in = 2q;
 *   traj (L,N,T,D_in) row-major, traj[:,:,0] = z0.
 *   save: gpode_rollout_save_floats() floats if a backward will follow, else NULL. */
int gpode_rollout_fwd(const GpodeProblem* p, const float* z0, int z0_per_sample, const float* ts, int T,
                      int method, int order, float* traj, float* save,
                      void* workspace, size_t workspace_bytes, void* stream);

/* reverse-mode sweep through the unrolled solver (what autograd does for use_adjoint=False, core/flow.py:76):
 *   dtraj = dL/dtraj (L,N,T,D_in) -> dz0 (L,N,D_in) (per sample; sum over L if z0 was shared) and parameter gradients. */
int gpode_rollout_bwd(const GpodeProblem* p, const float* ts, int T, int method, int order,
                      const float* traj, const float* save, const float* dtraj, float* dz0,
                      const GpodeParamGrads* grads, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Per-rollout setup at the M inducing points (what sits in the autograd graph of SVGP_Layer.build_cache),
 * batched over output dimensions and MC samples.  RBF variants: one (M x M) system per output dimension (or one shared);
 * divergence-free kernel: ONE (M D x M D) system shared by the L samples (D <= 8, M D <= 4096), factored by a blocked
 * Cholesky spread over the chip.  All of it in double precision inside, fp32 at the ABI.
 * ------------------------------------------------------------------------------------------- */

/* scratch bytes / forward->backward save floats of gpode_compute_nu_* (p: variant, L, M, D_in, D_out, Z, ell, var are read) */
size_t gpode_nu_workspace_bytes(const GpodeProblem* p);
size_t gpode_nu_save_floats(const GpodeProblem* p);

/* RBF.compute_nu (core/kernels.py:155-172) fused with K(Z,Z) (core/kernels.py:98-110, called at svpy.py:118), and
 * DivergenceFreeKernel.compute_nu (core/kernels.py:376-387) fused with its block Gram matrix (core/kernels.py:289-303):
 *   Lc = chol(K(Z,Z) + 1e-5 I) (lower triangle read, like torch.linalg.cholesky), nu = Lc^-T (u - Lc^-1 u_prior);
 *   one system per output dim (dimwise), one shared (shared), or one of order M D (DF: rows m D + component).
 *   u_prior = rff_forward(Z) and u = sample_inducing() are (L,M,D_out); nu comes out in the GpodeProblem layout.
 *   save: gpode_nu_save_floats() floats (Cholesky factors + Lc^-1 u_prior) for the backward.
 *   info (optional, Kc int32; DF: 1): 0, or 1 + index of the first non-positive pivot (torch.linalg.cholesky raises there). */
int gpode_compute_nu_fwd(const GpodeProblem* p, const float* u_prior, const float* u, float* nu, float* save, int32_t* info,
                         void* workspace, size_t workspace_bytes, void* stream);
/* autograd backward of the above: d_nu (nu layout) -> d_u_prior, d_u (L,M,D_out) and the direct dependence of K(Z,Z) on
 * Z (M,D_in), ell, var (layouts of GpodeProblem; written, not accumulated).  Any output may be NULL. */
int gpode_compute_nu_bwd(const GpodeProblem* p, const float* u, const float* save, const float* d_nu, float* d_u_prior, float* d_u,
                         float* d_Z, float* d_ell, float* d_var, void* workspace, size_t workspace_bytes, void* stream);

/* SVGP_Layer.sample_inducing (core/svpy.py:88-101, q_diag=False) for L samples on the PACKED lower-triangular parameter
 * (Us_sqrt.optvar, (D_out, M(M+1)/2) row-major tril order, misc/transforms.py:71-77):
 *   u[l,n,d] = sum_{m<=n} Lq_d[n,m] eps_u[l,m,d] + Um[n,d];   eps_u, u (L,M,D_out), Um (M,D_out). */
int gpode_inducing_sample_fwd(int L, int M, int D_out, const float* Lq_packed, const float* Um, const float* eps_u, float* u, void* stream);
int gpode_inducing_sample_bwd(int L, int M, int D_out, const float* eps_u, const float* d_u, float* d_Lq_packed, float* d_Um, void* stream);

/* SVGP_Layer.kl (core/svpy.py:144-175, q_diag=False) on the packed parameter: kl (1 float on the device)
 *   = 1/2 sum_d ( -sum_i log Lq_d[i,i]^2 + |Um[:,d]|^2 + |Lq_d|_F^2 - M );  d_kl is a device scalar. */
int gpode_kl_fwd(int M, int D_out, const float* Lq_packed, const float* Um, float* kl, void* stream);
int gpode_kl_bwd(int M, int D_out, const float* Lq_packed, const float* Um, const float* d_kl, float* d_Lq_packed, float* d_Um, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Either side of the flow (SURVEY.md section 8f rank 3).
 * ------------------------------------------------------------------------------------------- */

/* Function-sample draws on the device instead of host numpy + H2D (core/kernels.py:13-26 sample_normal / sample_uniform as used by
 * build_cache :126-137 / :305-316, and svpy.py:12-18,94): counter-based Philox4x32-10, up to four output segments in one launch
 * (w, eps, phase01, eps_u).  Element i of segment s = lane i % 4 of philox(counter = (i / 4 + offset [64 bit], s, 0), key = seed);
 * GPODE_DRAW_UNIFORM: (r >> 8) 2^-24 in [0, 1); GPODE_DRAW_NORMAL: Box-Muller on the lane pairs (0, 1) and (2, 3):
 * sqrt(-2 ln u1) (cos, sin)(2 pi u2), u1 = ((r >> 8) + 1) 2^-24.  Same distribution as the reference's draws, not the same numbers
 * (the reference's own are unseeded, kernels.py:17).  Advance `offset` by ceil(max count / 4) between calls. */
enum { GPODE_DRAW_NORMAL = 0, GPODE_DRAW_UNIFORM = 1 };
int gpode_philox_fill(int nseg, float* const* outs, const uint64_t* counts, const int32_t* kinds, uint64_t seed, uint64_t offset, void* stream);
/* the bare generator, for known-answer tests: out[4 i .. 4 i + 3] = philox4x32_10(counters[4 i ..], keys[2 i ..]) (device pointers) */
int gpode_philox_raw(const uint32_t* counters, const uint32_t* keys, uint32_t* out, int n, void* stream);

/* Decoder.log_prob (core/vae.py:136-153, bernoulli) fused with the reduction of elbo() (create_model.py:51-53:
 * lhood.sum([2,3,4,5]).mean(0)):  z (L,N,P) reconstructions, x (N,P) targets (P = T * pixels; x is NOT repeated L times),
 *   lhood[n] = 1/L sum_{l,p} log(z) x + log(1 - z)(1 - x);      d_z = d_lhood[n] / L (x / z - (1 - x) / (1 - z)). */
size_t gpode_bernoulli_workspace_bytes(int N);
int gpode_bernoulli_lhood_fwd(int L, int N, int64_t P, const float* z, const float* x, float* lhood, void* workspace, size_t workspace_bytes, void* stream);
int gpode_bernoulli_lhood_bwd(int L, int N, int64_t P, const float* z, const float* x, const float* d_lhood, float* d_z, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GPODE_H_ */
