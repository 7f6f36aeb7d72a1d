"""GPU: every kernel instantiation the launch heuristics can pick, against autograd through the fp64 oracle (oracle/field.py).

The rows (tests/dispatch_cases.py) each reach one family: the RBF small-batch policy with clusters of 1, 2, 7 and 8 CTAs, the RBF FFMA
policy with R = 1, 2, 4 at D <= 8 and D > 8 (with the mma.sync parameter-gradient pass), the mma.sync and tcgen05 tensor path (order 2,
shared lengthscales, the 15 % padding threshold), the DF warp-split policy with clusters of 2, 3, 5, 6, 7, 8 CTAs and the DF thread <->
state policy at 32, 64, 128 threads and R = 2.  For each row: field and prior part, field VJP with every leaf gradient, rollout
trajectories and rollout backward (dz0 and every leaf gradient), per method.  Bars as in the rest of the suite, norm-wise: field 1e-5,
trajectories and gradients 1e-4.

Rows with more states than the fp64 oracle can follow use the masked-subset scheme of test_gpu_baseline_shapes.py: the upstream gradient
is non-zero on a subset only -- states 0 and N - 1, both sides of the first and the last boundary of every CTA size a family uses, the
ragged tail, and a random draw -- plus linearity of the backward over the whole batch, and replication: the second half of the batch is
a copy of the first, so trajectories and dz0 of the copies must be bit-identical (DESIGN.md section 2), which catches index errors in
far CTAs a subset can miss.

test_launch_witness records with torch.profiler which kernels a row launches (instantiation in the name, grid of the launch), kept apart
from the parity checks so that a profiler problem cannot hide a parity result.
"""
import json
import math
import os
import re
import tempfile

import numpy as np
import pytest
import torch

from oracle import field as OF
from dispatch_cases import FLAG_BITS, ROWS, row_id
from helpers import DF_CASES, gpu_sample, load_golden, oracle_cache, rel, t
from test_gpu_baseline_shapes import make_cache

pytestmark = pytest.mark.gpu

FIELD_TOL, TRAJ_TOL, GRAD_TOL = 1e-5, 1e-4, 1e-4
ORACLE_ALL = 600          # rows up to this many states are checked on every state
CTA_SIZES = (32, 64, 96, 128, 192, 256, 384, 512)       # states per CTA of every family (threads x R)
GRIDS = {"uniform": lambda T: 0.1 * np.arange(T), "nonuniform": lambda T: np.cumsum([0.0, 0.07, 0.16, 0.05][:T]),
         "decreasing": lambda T: 0.3 - 0.1 * np.arange(T), "T1": lambda T: np.zeros(1), "T2": lambda T: np.array([0.0, 0.15])}


def _gp():
    import gpode_b200
    return gpode_b200


def subset(N, seed):
    """the states the oracle follows on a large row"""
    if N <= ORACLE_ALL:
        return np.arange(N)
    idx = {0, 1, N - 3, N - 2, N - 1}
    for b in CTA_SIZES:
        last = (N - 1) // b * b
        idx.update(i for i in (b - 1, b, last - 1, last, last + 1) if 0 <= i < N)
    idx.update(np.random.RandomState(seed).choice(N, size=32, replace=False).tolist())
    return np.array(sorted(idx))


def shared_cache(variant, D_in, D_out, M, S, seed, perturb, nu_scale, shared=None):
    """make_cache for RBF with one lengthscale vector and one variance for all outputs (the reference's dimwise=False): omega (D_in, S),
    phase (1, S), w (S, D_out), nu (M, D_out)"""
    rs = np.random.RandomState(seed)
    f64 = lambda a: torch.tensor(a, dtype=torch.float64)
    c = dict(variant=variant, Z=f64(rs.normal(size=(M, D_in))), ell=f64(2.0 + perturb * rs.uniform(size=D_in)),
             var=f64(1.0 + perturb * rs.uniform(size=1)), eps=f64(rs.normal(size=(D_in, S))), phase=f64(rs.uniform(size=(1, S)) * 2 * math.pi),
             w=f64(rs.normal(size=(S, D_out))), nu=f64(nu_scale * rs.normal(size=(M, D_out))))
    for k in ("Z", "ell", "var", "nu"):
        c[k] = shared[k] if (shared is not None and k != "nu") else c[k].requires_grad_(True)
    c["omega"] = OF.make_omega(c["eps"], c["ell"], variant)
    return c, ("Z", "ell", "var", "nu")


class Problem:
    """one row: L function samples sharing Z / ell / var (fp64 caches with leaf tensors) and their fp32 copies on the GPU"""

    def __init__(self, row, seed=0):
        self.row = row
        make = shared_cache if row.variant == "rbf_shared" else make_cache
        args = dict(perturb=0.5, nu_scale=0.05)
        self.caches = [make(row.variant, row.D_in, row.D_out, row.M, row.S, seed=seed, **args)[0]]
        for l in range(1, row.L):
            self.caches.append(make(row.variant, row.D_in, row.D_out, row.M, row.S, seed=seed + l, shared=self.caches[0], **args)[0])
        self.df = row.variant == "df"
        self.shared = ("Z", "ell", "var")
        self.per_sample = ("nu", "B") if self.df else ("nu",)

    def gpu(self):
        ss = [gpu_sample(c) for c in self.caches]
        s = {k: ss[0][k] for k in self.shared}
        for k in ("eps", "phase", "w") + self.per_sample:
            s[k] = torch.cat([q[k] for q in ss], 0)
        for k in self.shared + self.per_sample:
            s[k].requires_grad_(True)
        return s

    def leaves(self, s):
        return [s[k] for k in self.shared + self.per_sample]

    def oracle_leaves(self):
        return [self.caches[0][k] for k in self.shared] + [c[k] for k in self.per_sample for c in self.caches]

    def oracle_grads(self, want):
        """oracle gradients in the layout of the GPU leaves: per-sample leaves stacked over l"""
        n, L = len(self.shared), self.row.L
        out = list(want[:n])
        for j in range(len(self.per_sample)):
            out.append(torch.stack(list(want[n + j * L:n + (j + 1) * L])))
        return out

    def names(self):
        return ["d" + k for k in self.shared + self.per_sample]

    def field(self, s, x):
        return _gp().gp_field(x, s["Z"], s["nu"], s["eps"], s["phase"], s["w"], s["ell"], s["var"], self.row.variant, s.get("B"))

    def rollout(self, s, z0, ts, method):
        return _gp().gp_rollout(z0, ts, s["Z"], s["nu"], s["eps"], s["phase"], s["w"], s["ell"], s["var"], self.row.variant, self.row.order,
                                method, s.get("B"))


def replicated(rs, L, N, D, scale):
    """(L, N, D) float32 states whose second half [h, 2h) is a copy of the first (h = N // 2)"""
    a = (scale * rs.normal(size=(L, N, D))).astype(np.float32)
    h = N // 2
    a[:, h:2 * h] = a[:, :h]
    return a


def assert_copies_identical(a, N, what):
    h = N // 2
    assert torch.equal(a[..., :h, :, :] if a.dim() == 4 else a[..., :h, :], a[..., h:2 * h, :, :] if a.dim() == 4 else a[..., h:2 * h, :]), \
        "%s: the copies in the second half of the batch differ from the first half" % what


def check_backward(label, run, mask_np, G_np, want, names, idx, dim_x):
    """run(G) -> (dx, leaf grads) on the GPU.  G_np (L, N, ...) is the dense upstream gradient, mask_np selects the subset the oracle
    follows (want = oracle gradients of the masked loss: [dx on the subset] + leaves).  Large rows also check linearity over the whole
    batch and return the dense dx for the replication check."""
    dx_m, pg_m = run(G_np * mask_np)
    e = rel(dx_m[..., idx, :] if dim_x else dx_m[idx], want[0])
    print("  %s d%s vs fp64 %.2e" % (label, "x" if dim_x else "z0", e))
    assert e < GRAD_TOL, (label, "dx", e)
    for nm, a, b in zip(names, pg_m, want[1:]):
        e = rel(a, b)
        print("  %s %s vs fp64 %.2e" % (label, nm, e))
        assert e < GRAD_TOL, (label, nm, e)
    if mask_np.all():
        return None
    dx_f, pg_f = run(G_np)
    dx_c, pg_c = run(G_np * (1.0 - mask_np))
    assert rel(dx_f, dx_m + dx_c) < 1e-6, label
    for nm, a, b1, b2 in zip(names, pg_f, pg_m, pg_c):
        e = rel(a, b1 + b2)
        print("  %s %s linearity over all states %.2e" % (label, nm, e))
        assert e < GRAD_TOL, (label, nm, e)
    return dx_f


def variance_cancellation(g, f, fp):
    """how many times the terms of the variance-gradient sum sum_n,k g (f - f_p / 2) cancel (fp64).  With one variance for all outputs
    (rbf_shared) that gradient is a single number: relative to it, the per-state error of any fp32 evaluation of f is amplified by this
    factor, so a draw where it is large measures the draw rather than the kernel"""
    t = g * (f - 0.5 * fp)
    return float(t.abs().sum() / t.sum().abs())


def run_row(row, grid="uniform"):
    seed = row.seed
    P = Problem(row, seed)
    L, N, D, Do = row.L, row.N, row.D_in, row.D_out
    rs = np.random.RandomState(seed + 7)
    idx = subset(N, seed)
    big = len(idx) < N
    mask = np.zeros((1, N, 1), dtype=np.float32)
    mask[:, idx] = 1.0
    print("%s [%s] N=%d L=%d: oracle on %d states" % (row.family, grid, N, L, len(idx)))
    with _gp().kernel_flags(FLAG_BITS[row.flags]):
        if grid == "uniform":
            # ---- field, prior part, field VJP ----
            x_np = replicated(rs, L, N, D, 1.2)
            s = P.gpu()
            f, fp = P.field(s, torch.tensor(x_np, device="cuda"))
            if big:
                assert_copies_identical(f, N, row.family + " field")
            for l, c in enumerate(P.caches):
                xs = torch.tensor(x_np[l, idx], dtype=torch.float64)
                e_f, e_p = rel(f[l, idx], OF.field(xs, c)), rel(fp[l, idx], OF.prior(xs, c))
                print("  field l=%d vs fp64 %.2e  prior part %.2e" % (l, e_f, e_p))
                assert e_f < FIELD_TOL and e_p < FIELD_TOL, (l, e_f, e_p)
            g_np = rs.normal(size=(L, N, Do)).astype(np.float32)
            g_np[:, N // 2:2 * (N // 2)] = g_np[:, :N // 2]
            xs = [torch.tensor(x_np[l, idx], dtype=torch.float64).requires_grad_(True) for l in range(L)]
            loss = sum((OF.field(xs[l], c) * torch.tensor(g_np[l, idx], dtype=torch.float64)).sum() for l, c in enumerate(P.caches))
            want = torch.autograd.grad(loss, xs + P.oracle_leaves(), retain_graph=True)      # (omega = eps / ell is built once per cache)
            if row.variant == "rbf_shared":
                kappa = max(variance_cancellation(torch.tensor(g_np[l, idx], dtype=torch.float64), OF.field(xs[l], c).detach(),
                                                  OF.prior(xs[l], c).detach()) for l, c in enumerate(P.caches))
                print("  shared variance gradient: terms cancel %.0f-fold" % kappa)
                assert kappa < 100, "ill-conditioned draw for the shared variance gradient (%.0f-fold cancellation): choose another seed" % kappa
            want = [torch.stack(list(want[:L]))] + P.oracle_grads(want[L:])

            def run_field(G):
                s = P.gpu()
                x = torch.tensor(x_np, device="cuda").requires_grad_(True)
                f, _ = P.field(s, x)
                gr = torch.autograd.grad(f, [x] + P.leaves(s), torch.tensor(G, device="cuda"))
                return gr[0], list(gr[1:])

            dx = check_backward("field-bwd", run_field, mask, g_np, want, P.names(), idx, True)
            if dx is not None:
                assert_copies_identical(dx, N, row.family + " dx")
        # ---- rollouts ----
        T = 3 if big else 4
        ts_np = GRIDS[grid](T)
        T = len(ts_np)
        ts = torch.tensor(ts_np, dtype=torch.float32, device="cuda")
        ts64 = torch.tensor(ts_np, dtype=torch.float32).double()
        z0_np = replicated(rs, 1, N, D, 0.8)[0]
        G_np = rs.normal(size=(L, N, T, D)).astype(np.float32)
        G_np[:, N // 2:2 * (N // 2)] = G_np[:, :N // 2]
        for method in row.methods:
            label = "%s rollout" % method
            s = P.gpu()
            z0 = torch.tensor(z0_np, device="cuda").requires_grad_(True)
            traj = P.rollout(s, z0, ts, method)
            assert traj.shape == (L, N, T, D)
            assert torch.equal(traj[:, :, 0], z0.detach()[None].expand(L, N, D))
            if big:
                assert_copies_identical(traj, N, row.family + " " + label)
            z64 = torch.tensor(z0_np[idx], dtype=torch.float64).requires_grad_(True)
            trajs = [OF.rollout(z64, ts64, c, row.order, method) for c in P.caches]
            e = rel(traj[:, idx], torch.stack([tr.detach() for tr in trajs]))
            print("  %s traj vs fp64 %.2e" % (label, e))
            assert e < TRAJ_TOL, (label, e)
            loss = sum((tr * torch.tensor(G_np[l][idx], dtype=torch.float64)).sum() for l, tr in enumerate(trajs))
            want = torch.autograd.grad(loss, [z64] + P.oracle_leaves(), allow_unused=True, retain_graph=True)
            want = [want[0]] + P.oracle_grads([w if w is not None else torch.zeros_like(v) for w, v in zip(want[1:], P.oracle_leaves())])

            def run_rollout(G, traj=traj, s=s, z0=z0):
                gr = torch.autograd.grad(traj, [z0] + P.leaves(s), torch.tensor(G, device="cuda"), retain_graph=True)
                return gr[0], list(gr[1:])

            dz = check_backward(label + "-bwd", run_rollout, mask[..., None], G_np, want, P.names(), idx, False)
            if dz is not None:
                assert_copies_identical(dz, N, row.family + " " + label + " dz0")
            if T == 1:        # no step taken: dz0 is the upstream gradient at t0 and no parameter has a gradient
                gm = torch.tensor(G_np * mask[..., None], device="cuda")
                dz1, pg = run_rollout(G_np * mask[..., None])
                assert torch.equal(dz1, gm[:, :, 0].sum(0))
                for nm, a in zip(P.names(), pg):
                    assert float(a.abs().max()) == 0.0, nm


PARAMS = [pytest.param(r, "uniform", id=row_id(r)) for r in ROWS]
PARAMS += [pytest.param(r, g, id="%s-%s" % (row_id(r), g)) for r in ROWS if r.grids for g in ("nonuniform", "decreasing", "T1", "T2")]


@pytest.mark.parametrize("row,grid", PARAMS)
def test_dispatch_row_vs_fp64(row, grid):
    run_row(row, grid)


@pytest.mark.parametrize("name,ts_scale", [(n, 1.0) for n in DF_CASES] + [("df_o1_pert", 2.0)])
def test_df_midpoint_rollout_backward_golden(name, ts_scale):
    """the DF reverse sweep with the midpoint tableau on the three DF goldens (euler and rk4 are in test_gpu_df.py).  ts_scale = 2: steps of
    0.2, where the stage coefficient a[1][0] carries weight in the gradients -- a change of it by 2e-4 moves them by 4e-4 .. 2e-3 while an
    fp32 evaluation of the same solve stays within 2e-5 of fp64"""
    g = load_golden(name)
    g["ts"] = g["ts"] * ts_scale
    c = oracle_cache(g, leaves=True)
    c["B"] = c["B"].detach().clone().requires_grad_(True)
    leaves = ("Z", "nu", "ell", "var", "B")
    z64 = t(g["z0"], torch.float64).requires_grad_(True)
    G = t(g["G"], torch.float64)
    want = torch.autograd.grad((OF.rollout(z64, t(g["ts"], torch.float64), c, 1, "midpoint") * G).sum(), [z64] + [c[k] for k in leaves])
    s = gpu_sample(c)
    for k in leaves:
        s[k].requires_grad_(True)
    z0 = t(g["z0"], device="cuda").requires_grad_(True)
    traj = _gp().gp_rollout(z0, t(g["ts"], device="cuda"), s["Z"], s["nu"], s["eps"], s["phase"], s["w"], s["ell"], s["var"], "df", 1,
                            "midpoint", s["B"])
    (traj[0] * t(g["G"], device="cuda")).sum().backward()
    got = [z0.grad, s["Z"].grad, s["nu"].grad[0], s["ell"].grad, s["var"].grad, s["B"].grad[0]]
    for nm, a, b in zip(("dz0", "dZ", "dnu", "dell", "dvar", "dB"), got, want):
        e = rel(a, b)
        print("%s midpoint rollout-bwd %s vs fp64 %.2e" % (name, nm, e))
        assert e < GRAD_TOL, (nm, e)


# ------------------------------------------------------------------------------------------------------------------------
# launch witness: which instantiation each row launches, from the kernel names and grids torch.profiler records
# ------------------------------------------------------------------------------------------------------------------------
SWEEPS = ("k_field_fwd", "k_rollout_fwd", "k_field_bwd", "k_rollout_bwd")


def launched_kernels(row):
    """(whitespace-free demangled name, grid) of every kernel one field fwd + bwd and one rollout fwd + bwd of the row launch"""
    from torch.profiler import ProfilerActivity, profile
    P = Problem(row, row.seed)
    rs = np.random.RandomState(1)
    s = P.gpu()
    x = torch.tensor(rs.normal(size=(row.L, row.N, row.D_in)), dtype=torch.float32, device="cuda").requires_grad_(True)
    z0 = torch.tensor(rs.normal(size=(row.N, row.D_in)), dtype=torch.float32, device="cuda").requires_grad_(True)
    ts = 0.1 * torch.arange(3, dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    with _gp().kernel_flags(FLAG_BITS[row.flags]), profile(activities=[ProfilerActivity.CUDA]) as prof:
        f, _ = P.field(s, x)
        f.sum().backward()
        if row.methods:
            P.rollout(s, z0, ts, row.methods[0]).sum().backward()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as fh:
            events = json.load(fh)["traceEvents"]
    out = []
    for ev in events:
        if ev.get("cat") == "kernel":
            out.append((re.sub(r"\s+", "", ev["name"]), tuple(ev.get("args", {}).get("grid", ()))))
    return out


@pytest.mark.parametrize("row", ROWS, ids=row_id)
def test_launch_witness(row):
    kernels = launched_kernels(row)
    assert kernels, "the profiler recorded no CUDA kernel"
    sweeps = [(n, g) for n, g in kernels if any(("::%s<" % k) in n for k in SWEEPS)]
    print("%s:" % row.family)
    for n, g in sorted(set(kernels)):
        print("   %s grid %s" % (n[:140], g))
    for k in SWEEPS if row.methods else SWEEPS[::2]:
        pol, per = (row.fwd, row.fwd_per) if k.endswith("fwd") else (row.bwd, row.bwd_per)
        pat = re.compile(r"::%s<gpode::%s>\(" % (k, pol))
        hits = [(n, g) for n, g in sweeps if ("::%s<" % k) in n]
        assert hits, "%s: %s never launched" % (row.family, k)
        for n, g in hits:       # every launch of this sweep kernel is the intended instantiation, with the intended grid
            assert pat.search(n), "%s: %s launched %s, expected %s" % (row.family, k, n, pol)
            if g:
                if per is not None:
                    assert g[0] == math.ceil(row.N / per), (row.family, k, g, per)
                assert g[1] == row.L and (len(g) < 3 or g[2] == row.cluster), (row.family, k, g)
    for e in row.extra:
        assert any(re.search(e, n) for n, _ in kernels), "%s: no launch of %s" % (row.family, e)
