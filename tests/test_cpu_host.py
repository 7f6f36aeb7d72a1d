"""CPU: the C-ABI library loads and exports every symbol include/gpode.h declares; host-side logic of
the drop-in modules (state_dict keys, draw order, transforms, errors) -- no compute calls."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from helpers import load_golden, rel, t

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from gpode_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "gpode.h")).read()
    declared = sorted(set(re.findall(r"\b(gpode_[a-z_0-9]+)\s*\(", hdr)))
    assert declared, "no declarations found"
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name
    assert sorted(_lib.EXPORTS) == declared
    L = _lib.load()
    assert L.gpode_version() == 211
    assert b"NULL" in L.gpode_error_string(-1)
    # argument checking happens before any CUDA call: NULL problem -> 0 bytes / error code
    assert L.gpode_workspace_bytes(None, 16, 2) == 0
    p = _lib.GpodeProblem()
    assert L.gpode_field_fwd(ctypes.byref(p), None, None, None, None, 0, None) < 0



@pytest.mark.parametrize("variant", ["rbf_dimwise", "df"])
def test_sample_count_limit(variant):
    """every sweep, pack and parameter-gradient launch puts the sample index L on grid y or z (at most 65,535): a larger L is refused
    with GPODE_E_UNSUPPORTED by the argument check, before any CUDA call, instead of failing at launch"""
    from gpode_b200 import _lib
    L = _lib.load()
    dummy = ctypes.c_void_p(256)          # never dereferenced: the shape check comes first
    p = _lib.GpodeProblem()
    p.variant, p.N, p.D_in, p.D_out, p.M, p.S = _lib.VARIANTS[variant], 2, 4, 4, 8, 8
    p.Z = p.ell = p.var = p.eps = p.phase = p.w = p.nu = p.B = dummy
    for Lm, ok in ((65535, True), (65536, False), (1 << 20, False)):
        p.L = Lm
        assert (L.gpode_workspace_bytes(ctypes.byref(p), 3, _lib.RK4) > 0) == ok, Lm
        assert (L.gpode_rollout_save_floats(ctypes.byref(p), 3, _lib.RK4) > 0) == ok, Lm
        if not ok:
            assert L.gpode_field_fwd(ctypes.byref(p), dummy, dummy, dummy, dummy, 0, None) == -3      # GPODE_E_UNSUPPORTED
    assert b"L <= 65535" in L.gpode_error_string(-3)

def test_forward_kernel_selection(monkeypatch):
    """which forward kernel family a problem gets depends on shapes only (plus GpodeProblem.flags): no CUDA call involved, and no
    environment variable is read"""
    from gpode_b200 import _lib
    L = _lib.load()

    def kind(variant, N, Lm, D, M, S, flags=0):
        p = _lib.GpodeProblem()
        p.variant, p.L, p.N, p.D_in, p.D_out, p.M, p.S, p.flags = _lib.VARIANTS[variant], Lm, N, D, D, M, S, flags
        return L.gpode_forward_kernel(ctypes.byref(p))

    monkeypatch.setenv("GPODE_FWD", "mma")      # ABI 1.x switch: must be ignored now
    assert L.gpode_forward_kernel(None) < 0
    assert kind("rbf_dimwise", 65536, 8, 16, 512, 256) == 2      # config 5: tensor memory
    assert kind("rbf_dimwise", 65536, 8, 16, 300, 100) == 1      # 400 units would pad to 768: mma.sync
    assert kind("rbf_dimwise", 1024, 8, 16, 512, 256) == 0       # small batch: FFMA
    assert kind("rbf_dimwise", 1048576, 1, 6, 256, 256) == 0     # D <= 8: FFMA
    assert kind("df", 1048576, 1, 6, 256, 256) == 0
    assert kind("rbf_dimwise", 65536, 8, 16, 512, 256, _lib.FLAG_FWD_MMA) == 1
    assert kind("rbf_dimwise", 65536, 8, 16, 300, 100, _lib.FLAG_FWD_TCGEN05) == 2


def test_small_batch_cluster_size():
    """small batches split an evaluation over a thread-block cluster (RBF: output dimensions, DF: rows of every chunk); the size depends
    on shapes only: as many CTAs per block of 32 states as fit the chip once, at most 8 (and at most D_out for RBF)"""
    from gpode_b200 import _lib
    L = _lib.load()

    def csize(variant, N, Lm, D_in, D_out, M, S):
        p = _lib.GpodeProblem()
        p.variant, p.L, p.N, p.D_in, p.D_out, p.M, p.S = _lib.VARIANTS[variant], Lm, N, D_in, D_out, M, S
        return L.gpode_cluster_size(ctypes.byref(p))

    assert L.gpode_cluster_size(None) < 0
    assert csize("rbf_dimwise", 25, 1, 6, 6, 100, 256) == 6        # config 1: one block of states, six outputs
    assert csize("rbf_dimwise", 50, 1, 6, 3, 100, 256) == 3        # config 3 (order 2): three outputs
    assert csize("rbf_dimwise", 25, 1, 6, 12, 20, 64) == 8         # capped at the portable cluster size
    assert csize("rbf_dimwise", 25, 1, 16, 16, 100, 256) == 1      # 410 KB of parameter rows do not fit a CTA: not the small-batch policy
    assert csize("rbf_dimwise", 1024, 4, 6, 6, 100, 256) == 1      # 128 blocks of 32 states: the chip is full already
    assert csize("rbf_dimwise", 65536, 8, 16, 16, 512, 256) == 1   # config 5: not a small batch
    assert csize("df", 256, 4, 6, 6, 100, 256) == 4                # config 2: 32 blocks of states x 4 fit 148 SMs
    assert csize("df", 25, 1, 6, 6, 100, 256) == 8
    assert csize("df", 1048576, 1, 6, 6, 256, 256) == 1


def test_state_dict_keys_match_reference():
    from gpode_b200.core.flow import Flow
    from gpode_b200.core.svpy import SVGP_Layer
    for kernel, d_out, order in (("RBF", 6, 1), ("DF", 6, 1), ("RBF", 3, 2)):
        gp = SVGP_Layer(D_in=6, D_out=d_out, M=10, S=8, dimwise=True, device="cpu", kernel=kernel)
        sd = Flow(gp, order=order, solver="euler").state_dict()
        assert list(sd.keys()) == ["odefunc._num_evals", "odefunc.diffeq.kern.unconstrained_lengthscales",
                                   "odefunc.diffeq.kern.unconstrained_variance", "odefunc.diffeq.inducing_loc.optvar",
                                   "odefunc.diffeq.Um.optvar", "odefunc.diffeq.Us_sqrt.optvar"]
        assert sd["odefunc.diffeq.Us_sqrt.optvar"].shape == (d_out, 55)
        assert sd["odefunc.diffeq.kern.unconstrained_lengthscales"].shape == (d_out, 6)
    gp = SVGP_Layer(D_in=6, D_out=6, M=10, S=8, dimwise=False, device="cpu", kernel="RBF")
    assert gp.kern.unconstrained_lengthscales.shape == (6,) and gp.kern.unconstrained_variance.shape == (1,)
    assert abs(gp.kern.lengthscales[0].item() - 0.2) < 1e-6 and abs(gp.kern.variance[0].item() - 0.1) < 1e-6


@pytest.mark.parametrize("name", ["rbf_dimwise_o1", "rbf_shared_o1", "df_d4"])
def test_build_cache_setup_matches_reference(name, monkeypatch):
    """per-rollout setup (torch ops) on CPU: same draw order, nu and kl agree with the reference."""
    from gpode_b200.core import kernels as K
    from gpode_b200.core import svpy as SV
    from oracle import field as OF
    from helpers import oracle_cache
    g = load_golden(name)
    m = g["meta"]
    gp = SV.SVGP_Layer(D_in=m["D_in"], D_out=m["D_out"], M=m["M"], S=m["S"], dimwise=m["dimwise"], device="cpu", kernel=m["kernel"])
    with torch.no_grad():
        gp.kern.unconstrained_lengthscales.copy_(t(g["p_raw_ell"]))
        gp.kern.unconstrained_variance.copy_(t(g["p_raw_var"]))
        gp.inducing_loc.optvar.copy_(t(g["p_Z"]))
        gp.Um.optvar.copy_(t(g["p_Um"]))
        gp.Us_sqrt.optvar.copy_(t(g["p_Us_sqrt"]))
    q = [g["draw_w"], g["draw_eps"], g["draw_phase01"], g["draw_eps_u"]]
    calls = []

    def feed(shape, seed=None):
        v = q[len(calls)]
        calls.append(tuple(shape))
        assert tuple(v.shape) == tuple(shape)
        return torch.tensor(v)

    monkeypatch.setattr(K, "sample_normal", feed)
    monkeypatch.setattr(K, "sample_uniform", feed)
    monkeypatch.setattr(SV, "sample_normal", feed)
    gp.build_cache()
    assert len(calls) == 4
    assert abs(gp.kl().item() - float(g["kl"])) < 1e-5 * abs(float(g["kl"]))
    # compare nu through the pathwise update it feeds (nu itself is ill-conditioned)
    c_ref = oracle_cache(g, torch.float64, shared_nu=True)
    c_new = dict(c_ref)
    c_new["nu"] = gp.kern.nu.detach().double()
    x = t(g["x"], torch.float64)
    assert rel(OF.update(x, c_new), OF.update(x, c_ref)) < 1e-3
    assert rel(gp.kern.rff_omega, c_ref["omega"]) < 1e-6
    s = gp.field_sample()
    assert s.eps.shape[0] == 1 and s.nu.shape[0] == 1


def test_transforms_roundtrip():
    from gpode_b200.misc import transforms
    from gpode_b200.misc.constraint_utils import invsoftplus, softplus
    lt = transforms.LowerTriangular(5, 3)
    packed = np.random.RandomState(0).normal(size=(3, 15)).astype(np.float32)
    full = lt.forward(packed)
    assert full.shape == (3, 5, 5) and np.allclose(np.triu(full[1], 1), 0)
    assert np.array_equal(lt.backward(full), packed)
    ft = lt.forward_tensor(torch.tensor(packed))
    assert np.array_equal(ft.numpy(), full)
    assert torch.equal(lt.backward_tensor(ft), torch.tensor(packed))
    # row-major tril order, like np.tril_indices
    assert full[0, 1, 0] == packed[0, 1] and full[0, 1, 1] == packed[0, 2]
    v = torch.tensor([0.2, 2.0, 1e-3])
    assert torch.allclose(softplus(invsoftplus(v)), v, rtol=1e-5)
    sp = transforms.SoftPlus()
    assert np.allclose(sp.forward(sp.backward(np.array([0.5, 3.0]))), [0.5, 3.0])


def test_no_cpu_path():
    """the product path has no CPU fallback: a CPU tensor raises instead of silently computing."""
    from gpode_b200.core.svpy import SVGP_Layer
    gp = SVGP_Layer(D_in=6, D_out=6, M=10, S=8, device="cpu")
    gp.build_cache()
    with pytest.raises(RuntimeError):
        gp(torch.zeros(4, 6))
    from gpode_b200.core.flow import Flow
    with pytest.raises(NotImplementedError):
        Flow(gp, order=1, solver="dopri5")(torch.zeros(4, 6), torch.arange(3.0))
    with pytest.raises(RuntimeError):                 # the adjoint mode runs on the same CUDA kernels: CPU tensors raise there too
        Flow(gp, order=1, solver="rk4", use_adjoint=True)(torch.zeros(4, 6), torch.arange(3.0))


def test_time_grid_helpers():
    """misc/torch_utils.py:49-61 mirrors: same values as the reference's helpers"""
    from gpode_b200.misc.torch_utils import compute_ts_dense, insert_zero_t0
    ts = 0.1 * torch.arange(5, dtype=torch.float)
    d = compute_ts_dense(ts, 4)
    want = torch.cat([torch.linspace(t1, t2, 4)[:-1] for (t1, t2) in zip(ts[:-1], ts[1:])] + [ts[-1:]])      # the reference's expression
    assert torch.equal(d, want) and d.shape[0] == 3 * 4 + 1 and torch.equal(d[::3], ts)
    assert compute_ts_dense(ts, 1) is ts
    z = insert_zero_t0(ts)
    assert torch.equal(z, torch.cat([torch.tensor([0.0]), ts + ts[1] - ts[0]]))


def test_oracle_adjoint_converges_to_the_discrete_gradient():
    """oracle/solvers.py odeint_adjoint (torchdiffeq's adjoint restated): on a small nonlinear ODE its gradients approach the
    exact gradients of the discrete solve as the grid is refined, at the order of the method -- and for euler on a LINEAR field
    with a symmetric matrix both coincide exactly."""
    from oracle import solvers
    torch.manual_seed(0)

    class Lin(torch.nn.Module):
        def __init__(self):
            super().__init__()
            A = torch.randn(3, 3, dtype=torch.float64)
            self.A = torch.nn.Parameter(0.3 * (A + A.t()))

        def forward(self, t, y):
            return torch.tanh(y @ self.A)
    f = Lin()
    y0 = torch.randn(5, 3, dtype=torch.float64)
    G = torch.randn(1, dtype=torch.float64)
    errs = []
    for T in (9, 17, 33):
        t = torch.linspace(0, 0.8, T, dtype=torch.float64)
        w = torch.randn(T, 5, 3, dtype=torch.float64, generator=torch.Generator().manual_seed(1))[: T] * 0 + 1.0
        ya = y0.clone().requires_grad_(True)
        f.zero_grad()
        (solvers.odeint_adjoint(f, ya, t, method="rk4") * w).sum().backward()
        ga, gA = ya.grad.clone(), f.A.grad.clone()
        yb = y0.clone().requires_grad_(True)
        f.zero_grad()
        (solvers.odeint(f, yb, t, method="rk4") * w).sum().backward()
        errs.append(max(float((ga - yb.grad).norm() / yb.grad.norm()), float((gA - f.A.grad).norm() / f.A.grad.norm())))
    assert errs[0] < 1e-3 and errs[2] < errs[1] < errs[0] and errs[2] < errs[0] / 20, errs
