// C ABI of libgpode.so (include/gpode.h): argument checking, workspace carving, kernel sequencing.
// Nothing here allocates, synchronises or keeps state: every call enqueues on the caller's stream.
#include <cstdio>
#include <cstdlib>

#include "common.cuh"
#include "df.h"
#include "rbf.h"
#include "setup.h"
#include "elbo.h"

using namespace gpode;

namespace {

struct Ws {  // byte offsets inside the workspace (256-B aligned), see gpode_workspace_bytes
  size_t packed, xs, ks, fps, ybar, ystage, kbar, gsave, acc, acc_bytes, total;
  size_t a_dnu, a_pg, a_dell_x, a_dvar, a_dell_z;  // offsets inside acc
};

int check_problem(const GpodeProblem* p) {
  if (!p) return GPODE_E_NULL;
  if (p->variant != GPODE_RBF_SHARED && p->variant != GPODE_RBF_DIMWISE && p->variant != GPODE_DF) return GPODE_E_ENUM;
  if (p->L < 1 || p->N < 1 || p->D_in < 1 || p->D_out < 1 || p->M < 1 || p->S < 1) return GPODE_E_SHAPE;
  if (!p->Z || !p->ell || !p->var || !p->eps || !p->phase || !p->w || !p->nu) return GPODE_E_NULL;
  if (p->D_in > kMaxD || p->D_out > kMaxD || p->M > 512) return GPODE_E_UNSUPPORTED;
  if (static_cast<long>(p->L) * p->N > (1L << 30)) return GPODE_E_UNSUPPORTED;
  if (p->L > kMaxSamples) return GPODE_E_UNSUPPORTED;   // every sweep, pack and parameter-gradient launch puts L on grid y or z
  if (p->variant == GPODE_DF) {
    if (p->D_in != p->D_out) return GPODE_E_SHAPE;
    if (!p->B) return GPODE_E_NULL;
    if (p->D_in > kDfMaxD) return GPODE_E_UNSUPPORTED;
  }
  return GPODE_OK;
}

RbfGeom rbf_geom(const GpodeProblem* p, int order) {
  RbfGeom g;
  g.L = p->L;
  g.N = p->N;
  g.NL = p->L * p->N;
  g.D_in = p->D_in;
  g.D_out = p->D_out;
  g.DP = (p->D_in + 1) / 2 * 2;
  g.M = p->M;
  g.S = p->S;
  g.MP2 = (p->M + 1) / 2;
  g.SP2 = (p->S + 1) / 2;
  g.hdr_floats = rbf_hdr_floats(g.DP);
  g.row_floats = rbf_row_floats(g.DP);
  const int rc_max = kChunkBytes / (g.row_floats * 4);   // rows per chunk, balanced inside each section
  g.NCs = (g.SP2 + rc_max - 1) / rc_max;
  g.RCs = (g.SP2 + g.NCs - 1) / g.NCs;
  g.NCm = (g.MP2 + rc_max - 1) / rc_max;
  g.RCm = (g.MP2 + g.NCm - 1) / g.NCm;
  g.stage_floats = (g.RCs > g.RCm ? g.RCs : g.RCm) * g.row_floats;
  g.order = order;
  g.off = p->D_in - p->D_out;
  g.flags = p->flags;
  g.cg.stage_floats = g.stage_floats;
  g.cg.rowf_s = g.cg.rowf_m = g.row_floats;
  g.cg.SP2 = g.SP2; g.cg.MP2 = g.MP2; g.cg.NCs = g.NCs; g.cg.NCm = g.NCm; g.cg.RCs = g.RCs; g.cg.RCm = g.RCm;
  g.cg.K = g.D_out;
  g.cg.blk_floats = (g.SP2 + g.MP2) * g.row_floats;
  g.cg.tail = 0;
  return g;
}

size_t packed_floats(const GpodeProblem* p) {
  if (p->variant == GPODE_DF) return df_packed_floats(df_geom(p));
  return rbf_packed_floats(rbf_geom(p, 1));
}

size_t acc_floats(const GpodeProblem* p, Ws* w) {
  if (p->variant == GPODE_DF) return df_acc_floats(df_geom(p));
  const RbfGeom g = rbf_geom(p, 1);
  size_t o = 0;
  auto take = [&](size_t n) { const size_t at = o; o += (n + 63) / 64 * 64; return at; };
  const size_t a_dnu = take(static_cast<size_t>(g.L) * g.D_out * 2 * g.MP2);
  const size_t a_pg = take(static_cast<size_t>(g.L) * g.D_out * 2 * g.MP2 * g.DP);
  const size_t a_dell_x = take(static_cast<size_t>(g.D_out) * g.DP);
  const size_t a_dvar = take(g.D_out);
  const size_t a_dell_z = take(static_cast<size_t>(g.D_out) * g.DP);
  if (w) {
    w->a_dnu = a_dnu;
    w->a_pg = a_pg;
    w->a_dell_x = a_dell_x;
    w->a_dvar = a_dvar;
    w->a_dell_z = a_dell_z;
  }
  return o;
}

Ws layout(const GpodeProblem* p, int T, int method) {
  Ws w = {};
  const size_t NL = static_cast<size_t>(p->L) * p->N;
  const int stages = method_stages(method);
  const size_t steps = T > 1 ? static_cast<size_t>(T - 1) : 1;
  size_t o = 0;
  auto take = [&](size_t floats) { const size_t at = o; o += align_up(floats * 4, 256); return at; };
  w.packed = take(packed_floats(p));
  w.xs = take(stages * p->D_in * NL);   // one step of stage inputs / derivatives / prior parts (forward without saves)
  w.ks = take(stages * p->D_in * NL);
  w.fps = take(stages * p->D_out * NL);
  w.ybar = take(p->D_in * NL);
  w.ystage = take(stages * p->D_in * NL);
  w.kbar = take(p->D_in * NL);
  w.gsave = take(steps * stages * p->D_out * NL);
  w.acc_bytes = acc_floats(p, &w) * 4;
  w.acc = take(w.acc_bytes / 4);
  w.total = o;
  return w;
}

RbfAccum rbf_acc(char* ws, const Ws& w) {
  RbfAccum a;
  float* base = reinterpret_cast<float*>(ws + w.acc);
  a.dnu = base + w.a_dnu;
  a.pg = base + w.a_pg;
  a.dell_x = base + w.a_dell_x;
  a.dvar = base + w.a_dvar;
  a.dell_z = base + w.a_dell_z;
  return a;
}

int check_ws(const void* ws, size_t bytes, size_t need) {
  if (!ws) return GPODE_E_NULL;
  if ((reinterpret_cast<uintptr_t>(ws) & 255) != 0 || bytes < need) return GPODE_E_WORKSPACE;
  return GPODE_OK;
}

int rbf_check_smem(const RbfGeom& g) { return rbf_smem_bytes(g, 32, 1, true) <= kSmemLimit ? GPODE_OK : GPODE_E_UNSUPPORTED; }

cudaError_t rbf_pack(const GpodeProblem* p, const RbfGeom& g, float* packed, cudaStream_t st, bool fwd) {
  RbfPackArgs a;
  a.g = g;
  a.with_tc = fwd ? 1 : 2;
  a.variant = p->variant;
  a.Z = p->Z; a.ell = p->ell; a.var = p->var; a.eps = p->eps; a.phase = p->phase; a.w = p->w; a.nu = p->nu;
  a.packed = packed;
  return rbf_launch_pack(a, st);
}

// CTAs along the state-evaluation axis of a parameter-gradient kernel: the grid (chunks x ctas_per_chunk) should fill
// the chip's resident-CTA slots a whole number of times (the CTAs do equal work: no tail wave)
int pgrad_chunks(long evals_per_sample, int ctas_per_chunk, int ctas_per_sm) {
  const long slots = 148L * ctas_per_sm;
  long maxc = (evals_per_sample + 255) / 256;
  if (maxc < 1) maxc = 1;
  long best = 1;
  double best_eff = -1.0;
  for (int w = 2; w <= 8; ++w) {
    long c = slots * w / ctas_per_chunk;
    if (c > maxc) c = maxc;
    if (c < 1) c = 1;
    const long total = c * ctas_per_chunk, waves = (total + slots - 1) / slots;
    const double eff = static_cast<double>(total) / static_cast<double>(waves * slots);
    if (eff > best_eff + 1e-9) {
      best_eff = eff;
      best = c;
    }
  }
  return static_cast<int>(best);
}

cudaError_t rbf_param_grads(const GpodeProblem* p, const RbfGeom& g, const float* packed, const float* xsave, const float* gsave,
                            long n_te, const RbfAccum& acc, const GpodeParamGrads* grads, cudaStream_t st) {
  RbfPgradArgs pa;
  pa.g = g;
  pa.packed = packed;
  pa.xsave = xsave;
  pa.gsave = gsave;
  pa.n_te = n_te;
  if (rbf_pgrad_use_mma(g)) {
    int pg_mt, pg_mblk;
    rbf_pgrad_mma_shape(g, pg_mt, pg_mblk);
    pa.chunks = pgrad_chunks(n_te * g.N, g.D_out * g.L * pg_mblk, pg_mt == 1 ? 3 : 2);
  } else {
    int pg_threads, pg_pp, pg_mblk;
    rbf_pgrad_shape(g, pg_threads, pg_pp, pg_mblk);
    pa.chunks = pgrad_chunks(n_te * g.N, g.D_out * g.L * pg_mblk, 6 * kPgThreads / pg_threads);
  }
  pa.acc = acc;
  cudaError_t e = cudaSuccess;
  // the fused tcgen05 reverse sweep has already filled dnu / pg (rbf_bwd_tc.cuh): no separate pass over the exponentials
  if (!rbf_bwd_use_tc(g) && (e = rbf_launch_pgrad(pa, st)) != cudaSuccess) return e;
  RbfFinalizeArgs fa;
  fa.g = g;
  fa.variant = p->variant;
  fa.Z = p->Z; fa.ell = p->ell; fa.var = p->var; fa.nu = p->nu;
  fa.acc = acc;
  fa.d_Z = grads ? grads->d_Z : nullptr;
  fa.d_ell = grads ? grads->d_ell : nullptr;
  fa.d_var = grads ? grads->d_var : nullptr;
  fa.d_nu = grads ? grads->d_nu : nullptr;
  return rbf_launch_finalize(fa, st);
}

int df_check_smem(const DfGeom& g) { return df_smem_bytes(g, 128, 2, true, false) + 48 * 1024 <= kSmemLimit ? GPODE_OK : GPODE_E_UNSUPPORTED; }

cudaError_t df_pack(const GpodeProblem* p, const DfGeom& g, float* packed, cudaStream_t st) {
  DfPackArgs a;
  a.g = g;
  a.Z = p->Z; a.ell = p->ell; a.var = p->var; a.eps = p->eps; a.phase = p->phase; a.w = p->w; a.nu = p->nu; a.B = p->B;
  a.packed = packed;
  return df_launch_pack(a, st);
}

cudaError_t df_param_grads(const GpodeProblem* p, const DfGeom& g, const float* packed, const float* xsave, const float* gsave, long n_te,
                           const DfAccum& acc, const GpodeParamGrads* grads, cudaStream_t st) {
  DfPgradArgs pa;
  pa.g = g;
  pa.packed = packed;
  pa.xsave = xsave;
  pa.gsave = gsave;
  pa.n_te = n_te;
  pa.chunks_b = pgrad_chunks(n_te * g.N, g.L * ((g.D * g.SP2 + 127) / 128), 4);
  pa.acc = acc;
  cudaError_t e = df_launch_pgrad(pa, st);
  if (e != cudaSuccess) return e;
  DfFinalizeArgs fa;
  fa.g = g;
  fa.ell = p->ell; fa.var = p->var; fa.w = p->w;
  fa.acc = acc;
  fa.d_Z = grads ? grads->d_Z : nullptr;
  fa.d_ell = grads ? grads->d_ell : nullptr;
  fa.d_var = grads ? grads->d_var : nullptr;
  fa.d_nu = grads ? grads->d_nu : nullptr;
  fa.d_B = grads ? grads->d_B : nullptr;
  return df_launch_finalize(fa, st);
}

// T == 1: no step is taken, every parameter gradient is exactly zero (outputs are written, never left uninitialised)
cudaError_t zero_param_grads(const GpodeProblem* p, const GpodeParamGrads* grads, cudaStream_t st) {
  if (!grads) return cudaSuccess;
  const size_t D_in = p->D_in, D_out = p->D_out, M = p->M, L = p->L, S = p->S;
  const bool df = p->variant == GPODE_DF, dimwise = p->variant == GPODE_RBF_DIMWISE;
  const size_t n_ell = (df || dimwise) ? D_out * D_in : D_in, n_var = (df || dimwise) ? D_out : 1;
  const size_t n_nu = L * M * D_out;   // (L,D_out,M,1) / (L,M,D_out) / (L,M*D,1)
  struct { float* ptr; size_t n; } outs[5] = {{grads->d_Z, M * D_in}, {grads->d_ell, n_ell}, {grads->d_var, n_var}, {grads->d_nu, n_nu},
                                              {df ? grads->d_B : nullptr, L * S * D_in * D_in}};
  for (auto& o : outs)
    if (o.ptr) {
      cudaError_t e = cudaMemsetAsync(o.ptr, 0, o.n * sizeof(float), st);
      if (e != cudaSuccess) return e;
    }
  return cudaSuccess;
}

}  // namespace

extern "C" {

int gpode_version(void) { return GPODE_VERSION; }

int gpode_forward_kernel(const GpodeProblem* p) {
  if (!p) return GPODE_E_NULL;
  if (p->variant == GPODE_DF) return GPODE_FWD_FFMA;
  const RbfGeom g = rbf_geom(p, 1);
  if (rbf_fwd_use_tc(g)) return GPODE_FWD_TCGEN05;
  return (g.DP > 8 && rbf_fwd_use_mma(g)) ? GPODE_FWD_MMA : GPODE_FWD_FFMA;
}

int gpode_cluster_size(const GpodeProblem* p) {
  if (!p) return GPODE_E_NULL;
  if (p->N < 1 || p->L < 1 || p->D_out < 1) return GPODE_E_SHAPE;
  if (p->variant == GPODE_DF) {
    const DfGeom g = df_geom(p);
    return df_use_small(g) ? df_cluster(g, 32) : 1;
  }
  const RbfGeom g = rbf_geom(p, 1);
  return rbf_use_small(g) ? rbf_small_cluster(g) : 1;
}

const char* gpode_error_string(int code) {
  switch (code) {
    case GPODE_OK: return "ok";
    case GPODE_E_NULL: return "a required pointer is NULL";
    case GPODE_E_SHAPE: return "invalid or inconsistent shape";
    case GPODE_E_UNSUPPORTED: return "shape outside the compiled range (D_in/D_out <= 16, DF D <= 8, M <= 512, L <= 65535, L*N <= 2^30, parameter tile <= 227 KB)";
    case GPODE_E_WORKSPACE: return "workspace too small or not 256-byte aligned";
    case GPODE_E_ENUM: return "unknown variant / method / order";
    default: return code > 0 ? cudaGetErrorString(static_cast<cudaError_t>(code)) : "unknown error";
  }
}

size_t gpode_workspace_bytes(const GpodeProblem* p, int T, int method) {
  if (check_problem(p) != GPODE_OK) return 0;
  if (method < GPODE_EULER || method > GPODE_RK4) return 0;
  return layout(p, T, method).total;
}

size_t gpode_rollout_save_floats(const GpodeProblem* p, int T, int method) {
  if (check_problem(p) != GPODE_OK || T < 1) return 0;
  if (method < GPODE_EULER || method > GPODE_RK4) return 0;
  const size_t NL = static_cast<size_t>(p->L) * p->N;
  const size_t steps = T > 1 ? T - 1 : 1;
  return steps * method_stages(method) * (2 * static_cast<size_t>(p->D_in) + p->D_out) * NL;
}

int gpode_field_fwd(const GpodeProblem* p, const float* x, float* f, float* f_prior, void* workspace, size_t workspace_bytes,
                    void* stream) {
  int rc = check_problem(p);
  if (rc) return rc;
  if (!x || !f) return GPODE_E_NULL;
  const Ws w = layout(p, 2, GPODE_EULER);
  if ((rc = check_ws(workspace, workspace_bytes, w.total))) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  char* ws = static_cast<char*>(workspace);
  float* packed = reinterpret_cast<float*>(ws + w.packed);
  if (p->variant == GPODE_DF) {
    const DfGeom g = df_geom(p);
    if ((rc = df_check_smem(g))) return rc;
    cudaError_t e = df_pack(p, g, packed, st);
    if (e != cudaSuccess) return static_cast<int>(e);
    DfFieldFwdArgs a;
    a.g = g;
    a.packed = packed;
    a.x = x;
    a.f = f;
    a.f_prior = f_prior;
    return static_cast<int>(df_launch_field_fwd(a, st));
  }
  const RbfGeom g = rbf_geom(p, 1);
  if ((rc = rbf_check_smem(g))) return rc;
  cudaError_t e = rbf_pack(p, g, packed, st, true);
  if (e != cudaSuccess) return static_cast<int>(e);
  RbfFieldFwdArgs a;
  a.g = g;
  a.packed = packed;
  a.x = x;
  a.f = f;
  a.f_prior = f_prior;
  return static_cast<int>(rbf_launch_field_fwd(a, st));
}

int gpode_field_bwd(const GpodeProblem* p, const float* x, const float* g_out, const float* f, const float* f_prior, float* dx,
                    const GpodeParamGrads* grads, void* workspace, size_t workspace_bytes, void* stream) {
  int rc = check_problem(p);
  if (rc) return rc;
  if (!x || !g_out || !f || !f_prior || !dx) return GPODE_E_NULL;
  const Ws w = layout(p, 2, GPODE_EULER);
  if ((rc = check_ws(workspace, workspace_bytes, w.total))) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  char* ws = static_cast<char*>(workspace);
  float* packed = reinterpret_cast<float*>(ws + w.packed);
  cudaError_t e = cudaMemsetAsync(ws + w.acc, 0, w.acc_bytes, st);
  if (e != cudaSuccess) return static_cast<int>(e);
  if (p->variant == GPODE_DF) {
    const DfGeom g = df_geom(p);
    if ((rc = df_check_smem(g))) return rc;
    if ((e = df_pack(p, g, packed, st)) != cudaSuccess) return static_cast<int>(e);
    DfFieldBwdArgs a;
    a.g = g;
    a.packed = packed;
    a.x = x;
    a.gout = g_out;
    a.f = f;
    a.f_prior = f_prior;
    a.dx = dx;
    a.xsave = reinterpret_cast<float*>(ws + w.xs);
    a.gsave = reinterpret_cast<float*>(ws + w.gsave);
    a.acc = df_acc(reinterpret_cast<float*>(ws + w.acc), g);
    if ((e = df_launch_field_bwd(a, st)) != cudaSuccess) return static_cast<int>(e);
    return static_cast<int>(df_param_grads(p, g, packed, a.xsave, a.gsave, 1, a.acc, grads, st));
  }
  const RbfGeom g = rbf_geom(p, 1);
  if ((rc = rbf_check_smem(g))) return rc;
  if ((e = rbf_pack(p, g, packed, st, false)) != cudaSuccess) return static_cast<int>(e);
  RbfFieldBwdArgs a;
  a.g = g;
  a.packed = packed;
  a.x = x;
  a.gout = g_out;
  a.f = f;
  a.f_prior = f_prior;
  a.dx = dx;
  a.xsave = reinterpret_cast<float*>(ws + w.xs);
  a.gsave = reinterpret_cast<float*>(ws + w.gsave);
  a.acc = rbf_acc(ws, w);
  if ((e = rbf_launch_field_bwd(a, st)) != cudaSuccess) return static_cast<int>(e);
  return static_cast<int>(rbf_param_grads(p, g, packed, a.xsave, a.gsave, 1, a.acc, grads, st));
}

int gpode_rollout_fwd(const GpodeProblem* p, const float* z0, int z0_per_sample, const float* ts, int T, int method, int order,
                      float* traj, float* save, void* workspace, size_t workspace_bytes, void* stream) {
  int rc = check_problem(p);
  if (rc) return rc;
  if (!z0 || !ts || !traj) return GPODE_E_NULL;
  if (T < 1) return GPODE_E_SHAPE;
  if (method < GPODE_EULER || method > GPODE_RK4 || (order != 1 && order != 2)) return GPODE_E_ENUM;
  if ((order == 1 && p->D_in != p->D_out) || (order == 2 && p->D_in != 2 * p->D_out)) return GPODE_E_SHAPE;
  if (order == 2 && p->variant == GPODE_DF) return GPODE_E_SHAPE;  // the reference DF kernel needs D_in == D_out
  const Ws w = layout(p, T, method);
  if ((rc = check_ws(workspace, workspace_bytes, w.total))) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  char* ws = static_cast<char*>(workspace);
  float* packed = reinterpret_cast<float*>(ws + w.packed);
  const int stages = method_stages(method);
  const size_t NL = static_cast<size_t>(p->L) * p->N;
  const size_t steps = T > 1 ? T - 1 : 1;
  float *xs, *ks, *fps;
  if (save) {
    xs = save;
    ks = xs + steps * stages * p->D_in * NL;
    fps = ks + steps * stages * p->D_in * NL;
  } else {
    xs = reinterpret_cast<float*>(ws + w.xs);
    ks = reinterpret_cast<float*>(ws + w.ks);
    fps = reinterpret_cast<float*>(ws + w.fps);
  }
  if (p->variant == GPODE_DF) {
    const DfGeom g = df_geom(p);
    if ((rc = df_check_smem(g))) return rc;
    cudaError_t e = df_pack(p, g, packed, st);
    if (e != cudaSuccess) return static_cast<int>(e);
    DfRolloutFwdArgs a;
    a.g = g;
    a.packed = packed;
    a.z0 = z0;
    a.z0_per_sample = z0_per_sample;
    a.ts = ts;
    a.T = T;
    a.method = method;
    a.keep = save ? 1 : 0;
    a.traj = traj;
    a.xsave = xs;
    a.ksave = ks;
    a.fpsave = fps;
    return static_cast<int>(df_launch_rollout_fwd(a, st));
  }
  const RbfGeom g = rbf_geom(p, order);
  if ((rc = rbf_check_smem(g))) return rc;
  cudaError_t e = rbf_pack(p, g, packed, st, true);
  if (e != cudaSuccess) return static_cast<int>(e);
  RbfRolloutFwdArgs a;
  a.g = g;
  a.packed = packed;
  a.z0 = z0;
  a.z0_per_sample = z0_per_sample;
  a.ts = ts;
  a.T = T;
  a.method = method;
  a.keep = save ? 1 : 0;
  a.traj = traj;
  a.xsave = xs;
  a.ksave = ks;
  a.fpsave = fps;
  return static_cast<int>(rbf_launch_rollout_fwd(a, st));
}

int gpode_rollout_bwd(const GpodeProblem* p, const float* ts, int T, int method, int order, const float* traj, const float* save,
                      const float* dtraj, float* dz0, const GpodeParamGrads* grads, void* workspace, size_t workspace_bytes,
                      void* stream) {
  int rc = check_problem(p);
  if (rc) return rc;
  if (!ts || !save || !dtraj || !dz0) return GPODE_E_NULL;
  (void)traj;
  if (T < 1) return GPODE_E_SHAPE;
  if (method < GPODE_EULER || method > GPODE_RK4 || (order != 1 && order != 2)) return GPODE_E_ENUM;
  if ((order == 1 && p->D_in != p->D_out) || (order == 2 && p->D_in != 2 * p->D_out)) return GPODE_E_SHAPE;
  if (order == 2 && p->variant == GPODE_DF) return GPODE_E_SHAPE;
  const Ws w = layout(p, T, method);
  if ((rc = check_ws(workspace, workspace_bytes, w.total))) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  char* ws = static_cast<char*>(workspace);
  float* packed = reinterpret_cast<float*>(ws + w.packed);
  const int stages = method_stages(method);
  const size_t NL = static_cast<size_t>(p->L) * p->N;
  const size_t steps = T > 1 ? T - 1 : 1;
  const float* xs = save;
  const float* ks = xs + steps * stages * p->D_in * NL;
  const float* fps = ks + steps * stages * p->D_in * NL;
  cudaError_t e = cudaMemsetAsync(ws + w.acc, 0, w.acc_bytes, st);
  if (e != cudaSuccess) return static_cast<int>(e);
  if (p->variant == GPODE_DF) {
    const DfGeom g = df_geom(p);
    if ((rc = df_check_smem(g))) return rc;
    if ((e = df_pack(p, g, packed, st)) != cudaSuccess) return static_cast<int>(e);
    DfRolloutBwdArgs a;
    a.g = g;
    a.packed = packed;
    a.ts = ts;
    a.T = T;
    a.method = method;
    a.xsave = xs;
    a.ksave = ks;
    a.fpsave = fps;
    a.dtraj = dtraj;
    a.dz0 = dz0;
    a.gsave = reinterpret_cast<float*>(ws + w.gsave);
    a.ybar = reinterpret_cast<float*>(ws + w.ybar);
    a.ystage = reinterpret_cast<float*>(ws + w.ystage);
    a.kbar = reinterpret_cast<float*>(ws + w.kbar);
    a.acc = df_acc(reinterpret_cast<float*>(ws + w.acc), g);
    if ((e = df_launch_rollout_bwd(a, st)) != cudaSuccess) return static_cast<int>(e);
    if (T < 2) return static_cast<int>(zero_param_grads(p, grads, st));
    return static_cast<int>(df_param_grads(p, g, packed, xs, a.gsave, static_cast<long>(T - 1) * stages, a.acc, grads, st));
  }
  const RbfGeom g = rbf_geom(p, order);
  if ((rc = rbf_check_smem(g))) return rc;
  if ((e = rbf_pack(p, g, packed, st, false)) != cudaSuccess) return static_cast<int>(e);
  RbfRolloutBwdArgs a;
  a.g = g;
  a.packed = packed;
  a.ts = ts;
  a.T = T;
  a.method = method;
  a.xsave = xs;
  a.ksave = ks;
  a.fpsave = fps;
  a.dtraj = dtraj;
  a.dz0 = dz0;
  a.gsave = reinterpret_cast<float*>(ws + w.gsave);
  a.ybar = reinterpret_cast<float*>(ws + w.ybar);
  a.ystage = reinterpret_cast<float*>(ws + w.ystage);
  a.kbar = reinterpret_cast<float*>(ws + w.kbar);
  a.acc = rbf_acc(ws, w);
  if ((e = rbf_launch_rollout_bwd(a, st)) != cudaSuccess) return static_cast<int>(e);
  if (T < 2) return static_cast<int>(zero_param_grads(p, grads, st));
  return static_cast<int>(rbf_param_grads(p, g, packed, xs, a.gsave, static_cast<long>(T - 1) * stages, a.acc, grads, st));
}

/* ---- per-rollout setup: compute_nu, inducing sample, KL (setup_kernels.cu) ---- */
static int nu_geom(const GpodeProblem* p, NuGeom* g) {
  if (!p) return GPODE_E_NULL;
  if (p->variant != GPODE_RBF_SHARED && p->variant != GPODE_RBF_DIMWISE && p->variant != GPODE_DF) return GPODE_E_ENUM;
  if (p->L < 1 || p->D_in < 1 || p->D_out < 1 || p->M < 1) return GPODE_E_SHAPE;
  const bool df = p->variant == GPODE_DF;
  if (df && p->D_in != p->D_out) return GPODE_E_SHAPE;
  if (p->D_in > kMaxD || p->D_out > kMaxD || p->M > 512 || (df && (p->D_in > 8 || p->M * p->D_in > 4096))) return GPODE_E_UNSUPPORTED;
  if (!p->Z || !p->ell || !p->var) return GPODE_E_NULL;
  g->L = p->L; g->M = p->M; g->D_in = p->D_in; g->D_out = p->D_out;
  g->dimwise = p->variant == GPODE_RBF_DIMWISE ? 1 : 0;
  g->df = df ? 1 : 0;
  g->n = df ? p->M * p->D_in : p->M;
  g->Kc = g->dimwise ? p->D_out : 1;
  g->NR = (g->dimwise || df) ? p->L : p->L * p->D_out;
  g->jitter = 1e-5f;
  return GPODE_OK;
}

size_t gpode_nu_workspace_bytes(const GpodeProblem* p) {
  NuGeom g;
  if (nu_geom(p, &g) != GPODE_OK) return 0;
  return align_up(nu_ws_floats(g) * 4, 256);
}
size_t gpode_nu_save_floats(const GpodeProblem* p) {
  NuGeom g;
  if (nu_geom(p, &g) != GPODE_OK) return 0;
  return nu_save_floats(g);
}
int gpode_compute_nu_fwd(const GpodeProblem* p, const float* u_prior, const float* u, float* nu, float* save, int32_t* info,
                         void* workspace, size_t workspace_bytes, void* stream) {
  NuGeom g;
  int rc = nu_geom(p, &g);
  if (rc) return rc;
  if (!u_prior || !u || !nu || !save) return GPODE_E_NULL;
  if ((rc = check_ws(workspace, workspace_bytes, align_up(nu_ws_floats(g) * 4, 256)))) return rc;
  return static_cast<int>(nu_forward(g, p->Z, p->ell, p->var, u_prior, u, nu, save, info, static_cast<float*>(workspace),
                                     static_cast<cudaStream_t>(stream)));
}
int gpode_compute_nu_bwd(const GpodeProblem* p, const float* u, const float* save, const float* d_nu, float* d_u_prior, float* d_u,
                         float* d_Z, float* d_ell, float* d_var, void* workspace, size_t workspace_bytes, void* stream) {
  NuGeom g;
  int rc = nu_geom(p, &g);
  if (rc) return rc;
  if (!u || !save || !d_nu) return GPODE_E_NULL;
  if ((rc = check_ws(workspace, workspace_bytes, align_up(nu_ws_floats(g) * 4, 256)))) return rc;
  return static_cast<int>(nu_backward(g, p->Z, p->ell, p->var, u, save, d_nu, d_u_prior, d_u, d_Z, d_ell, d_var,
                                      static_cast<float*>(workspace), static_cast<cudaStream_t>(stream)));
}
static int check_lq(int L, int M, int D_out, const void* a, const void* b, const void* c, const void* d) {
  if (L < 1 || M < 1 || D_out < 1) return GPODE_E_SHAPE;
  if (M > 4096 || D_out > 64) return GPODE_E_UNSUPPORTED;
  if (!a || !b || !c || !d) return GPODE_E_NULL;
  return GPODE_OK;
}
int gpode_inducing_sample_fwd(int L, int M, int D_out, const float* Lq_packed, const float* Um, const float* eps_u, float* u, void* stream) {
  int rc = check_lq(L, M, D_out, Lq_packed, Um, eps_u, u);
  if (rc) return rc;
  return static_cast<int>(inducing_forward(L, M, D_out, Lq_packed, Um, eps_u, u, static_cast<cudaStream_t>(stream)));
}
int gpode_inducing_sample_bwd(int L, int M, int D_out, const float* eps_u, const float* d_u, float* d_Lq_packed, float* d_Um, void* stream) {
  int rc = check_lq(L, M, D_out, eps_u, d_u, d_Lq_packed, d_Um);
  if (rc) return rc;
  return static_cast<int>(inducing_backward(L, M, D_out, eps_u, d_u, d_Lq_packed, d_Um, 0, static_cast<cudaStream_t>(stream)));
}
int gpode_kl_fwd(int M, int D_out, const float* Lq_packed, const float* Um, float* kl, void* stream) {
  int rc = check_lq(1, M, D_out, Lq_packed, Um, kl, kl);
  if (rc) return rc;
  return static_cast<int>(kl_forward(M, D_out, Lq_packed, Um, kl, static_cast<cudaStream_t>(stream)));
}
int gpode_kl_bwd(int M, int D_out, const float* Lq_packed, const float* Um, const float* d_kl, float* d_Lq_packed, float* d_Um, void* stream) {
  int rc = check_lq(1, M, D_out, Lq_packed, Um, d_kl, d_Lq_packed);
  if (rc) return rc;
  if (!d_Um) return GPODE_E_NULL;
  return static_cast<int>(kl_backward(M, D_out, Lq_packed, Um, d_kl, d_Lq_packed, d_Um, static_cast<cudaStream_t>(stream)));
}


/* ---- either side of the flow: device draws, fused Bernoulli log-likelihood (elbo_kernels.cu) ---- */
int gpode_philox_fill(int nseg, float* const* outs, const uint64_t* counts, const int32_t* kinds, uint64_t seed, uint64_t offset, void* stream) {
  if (nseg < 1 || nseg > 4) return GPODE_E_SHAPE;
  if (!outs || !counts || !kinds) return GPODE_E_NULL;
  unsigned long long ns[4];
  int ks[4];
  for (int i = 0; i < nseg; ++i) {
    if (!outs[i] && counts[i]) return GPODE_E_NULL;
    if (kinds[i] != GPODE_DRAW_NORMAL && kinds[i] != GPODE_DRAW_UNIFORM) return GPODE_E_ENUM;
    ns[i] = counts[i];
    ks[i] = kinds[i];
  }
  return static_cast<int>(philox_fill(nseg, outs, ns, ks, seed, offset, static_cast<cudaStream_t>(stream)));
}
int gpode_philox_raw(const uint32_t* counters, const uint32_t* keys, uint32_t* out, int n, void* stream) {
  if (n < 1) return GPODE_E_SHAPE;
  if (!counters || !keys || !out) return GPODE_E_NULL;
  return static_cast<int>(philox_raw(counters, keys, out, n, static_cast<cudaStream_t>(stream)));
}
size_t gpode_bernoulli_workspace_bytes(int N) { return N > 0 ? align_up(static_cast<size_t>(N) * 8, 256) : 0; }
int gpode_bernoulli_lhood_fwd(int L, int N, int64_t P, const float* z, const float* x, float* lhood, void* workspace, size_t workspace_bytes, void* stream) {
  if (L < 1 || N < 1 || P < 1) return GPODE_E_SHAPE;
  if (!z || !x || !lhood) return GPODE_E_NULL;
  int rc = check_ws(workspace, workspace_bytes, gpode_bernoulli_workspace_bytes(N));
  if (rc) return rc;
  return static_cast<int>(bernoulli_forward(L, N, static_cast<long>(P), z, x, lhood, static_cast<double*>(workspace), static_cast<cudaStream_t>(stream)));
}
int gpode_bernoulli_lhood_bwd(int L, int N, int64_t P, const float* z, const float* x, const float* d_lhood, float* d_z, void* stream) {
  if (L < 1 || N < 1 || P < 1) return GPODE_E_SHAPE;
  if (!z || !x || !d_lhood || !d_z) return GPODE_E_NULL;
  return static_cast<int>(bernoulli_backward(L, N, static_cast<long>(P), z, x, d_lhood, d_z, static_cast<cudaStream_t>(stream)));
}

}  // extern "C"
