"""CPU: the full-model golden vectors (tests/golden/elbo_*.npz) against the reference itself (where a copy of it is present, see
oracle/reference_harness.py), the restated model (oracle/model.py) against the reference's fp64 run stored in them, and the synthetic
rotating-digit generator."""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import elbo_harness as EH
from oracle import field as OF
from oracle import glyph
from oracle import model as RM
from oracle import reference_harness as rh

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_gpu_elbo import CASES, GOLDEN_DIR, load, rel  # noqa: E402


def test_rotating_glyph_generator_is_deterministic_and_normalised():
    x = glyph.rotating_sequences(5, 16, seed=121)
    assert x.shape == (5, 16, 1, 28, 28) and x.dtype == np.float32
    assert np.array_equal(x, glyph.rotating_sequences(5, 16, seed=121))
    raw = x * np.float32(glyph.MNIST_STD) + np.float32(glyph.MNIST_MEAN)          # data/utils.py:13-14 undone
    assert raw.min() > -1e-6 and raw.max() < 1 + 1e-6 and raw.max() > 0.9
    # frame t is frame 0 rotated by t * 360 / 15 degrees (data/mnist.py:174-175): a full turn brings the digit back
    assert rel(x[:, 15], x[:, 0]) < 0.05 and rel(x[:, 7], x[:, 0]) > 0.5
    for cfg in ("cfg1", "cfg3"):
        g = load(cfg, "rk4")
        assert abs(glyph.checksum(EH.inputs(cfg)) - float(g["x_checksum"])) <= 1e-9 * abs(float(g["x_checksum"]))


@pytest.mark.skipif(not rh.reference_available(), reason="reference tree not present")
@pytest.mark.parametrize("cfg,solver", [("cfg1", "rk4"), ("cfg3", "euler")])
def test_golden_elbo_reproduces_from_the_reference(cfg, solver):
    """replaying the stored draws through the reference's own classes gives the stored ELBO terms and gradients back"""
    ref = rh.load_reference()
    g = load(cfg, solver)
    args = EH.make_args(cfg, solver, "cpu")
    model = EH.init_model(ref["create_model"], ref["initialization"], args, g["meta"]["model_seed"])
    model.load_state_dict({k[3:]: torch.tensor(v) for k, v in g.items() if k.startswith("sd/")}, strict=True)
    draws = EH.Replay([g["gp_draw/%03d" % i] for i in range(int(g["n_gp_draws"]))])
    noise = EH.Replay([g["enc_noise/%03d" % i] for i in range(int(g["n_enc_noise"]))])
    saved = (ref["kernels"].sample_normal, ref["kernels"].sample_uniform, ref["svpy"].sample_normal, ref["vae"].Encoder.sample)
    try:
        ref["kernels"].sample_normal = ref["kernels"].sample_uniform = ref["svpy"].sample_normal = draws
        EH.patch_encoder_noise(ref["vae"], noise)
        scal, grads = EH.run_loss(ref["create_model"], model, torch.tensor(EH.inputs(cfg)), g["meta"]["L"])
    finally:
        ref["kernels"].sample_normal, ref["kernels"].sample_uniform, ref["svpy"].sample_normal, ref["vae"].Encoder.sample = saved
    for k in ("loss", "nlhood", "kl_reg", "kl_gp"):
        assert abs(scal[k] - float(g["ref32/" + k])) <= 2e-6 * abs(float(g["ref32/" + k])), k
    total = np.sqrt(sum(float(np.sum(v.astype(np.float64) ** 2)) for k, v in g.items() if k.startswith("ref32/grad/")))
    for k, v in grads.items():
        want = g["ref32/grad/" + k]
        if np.linalg.norm(want) > 1e-9 * total:
            assert rel(v, want) < 1e-4, k          # thread-count dependent fp32 summation order only


class _FixedFlow(torch.autograd.Function):
    """the flow boundary of the reference's fp64 run: z0 -> its latent trajectories; backward: its dL/dz0 through the rollouts"""

    @staticmethod
    def forward(ctx, z0, ztL, dz0):
        ctx.dz0 = dz0
        return ztL.clone()

    @staticmethod
    def backward(ctx, g):
        return ctx.dz0, None, None


class _StoredFlow(torch.nn.Module):
    def __init__(self, fb):
        super().__init__()
        self.ztL, self.dz0 = torch.tensor(fb["ztL"], dtype=torch.float64), torch.tensor(fb["dz0"], dtype=torch.float64)
        self.kl_gp, self.i = float(fb["kl_gp"]), 0

    def forward(self, z0, ts):
        dz0 = self.dz0 if self.i == 0 else torch.zeros_like(self.dz0)      # the rollouts' whole share of dL/dz0, counted once
        self.i += 1
        return _FixedFlow.apply(z0, self.ztL[self.i - 1], dz0)

    def kl(self):
        return torch.tensor(self.kl_gp, dtype=torch.float64)


@pytest.mark.parametrize("cfg,solver", CASES)
def test_restated_model_reproduces_the_reference_fp64_run(cfg, solver, monkeypatch):
    """oracle/model.py (the reference's VAE / ODEGPVAE / elbo / compute_loss, restated) in float64 with the stored state_dict and
    encoder noise, and the reference's own fp64 flow boundary (tests/golden/elbo_flow_*.npz) in place of the GP flow: the encoder
    sample z0, the four ELBO terms and the gradient of every encoder / decoder parameter are the reference's fp64 run's"""
    g = load(cfg, solver)
    fb = np.load(os.path.join(GOLDEN_DIR, "elbo_flow_%s_%s.npz" % (cfg, solver)))
    args = EH.make_args(cfg, solver, "cpu")
    vae = RM.VAE(frames=args.frames, n_filt=args.n_filt, latent_dim=args.latent_dim, order=args.ode).double()
    vae.load_state_dict({k[len("sd/vae."):]: torch.tensor(v) for k, v in g.items() if k.startswith("sd/vae.")}, strict=True)
    vae.prior = torch.distributions.Normal(vae.prior.loc.double(), vae.prior.scale.double())
    model = RM.ODEGPVAE(_StoredFlow(fb), vae, args.Ndata, args.ode, args.frames, args.dt).train()
    monkeypatch.setattr(RM.Encoder, "sample", RM.Encoder.sample)      # restored after the test
    noise = EH.Replay([g["enc_noise/%03d" % i] for i in range(int(g["n_enc_noise"]))], torch.float64)
    EH.patch_encoder_noise(RM, noise)
    z0 = {}
    sample_trajectories = model.sample_trajectories

    def spy(z, T, L=1):
        z0["z"] = z
        return sample_trajectories(z, T, L)
    model.sample_trajectories = spy
    X = torch.tensor(EH.inputs(cfg, g["meta"]["x_seed"]), dtype=torch.float64)
    scal = RM.compute_loss(model, X, g["meta"]["L"])
    scal[0].backward()
    assert noise.left() == 0 and model.flow.i == g["meta"]["L"]
    assert rel(z0["z"].detach().numpy(), fb["z0"]) < 1e-12
    for k, v in zip(("loss", "nlhood", "kl_reg", "kl_gp"), scal):
        assert abs(v.item() - float(g["ref64/" + k])) <= 1e-10 * abs(float(g["ref64/" + k])), k
    total = np.sqrt(sum(float(np.sum(g[k].astype(np.float64) ** 2)) for k in g if k.startswith("ref64/grad/")))
    for n, p in vae.named_parameters():
        want = g["ref64/grad/vae." + n]
        if np.linalg.norm(want) > 1e-9 * total:                       # (conv biases in front of a BatchNorm: exact zeros)
            assert rel(p.grad.numpy(), want) < 1e-6, n                 # fp32 storage of the stored gradients


@pytest.mark.parametrize("solver", ["euler", "rk4"])
def test_restated_model_forecast_reproduces_the_reference_fp64_run(solver, monkeypatch):
    """config 3's forward-only T = 64 forecast, ``model(X, 1, T_custom=64)`` as tests/test_gpu_elbo.py calls it, through
    oracle/model.py in float64 with the fp64 oracle flow (oracle/field.py) on the forecast's stored GP draws and encoder noise:
    the latent trajectories and the per-frame reconstruction sums are the reference's fp64 forecast's"""
    g = load("cfg3", solver)
    args = EH.make_args("cfg3", solver, "cpu")
    vae = RM.VAE(frames=args.frames, n_filt=args.n_filt, latent_dim=args.latent_dim, order=args.ode).double()
    vae.load_state_dict({k[len("sd/vae."):]: torch.tensor(v) for k, v in g.items() if k.startswith("sd/vae.")}, strict=True)
    sd = lambda k: torch.tensor(g["sd/flow.odefunc.diffeq." + k], dtype=torch.float64)
    n_gp, n_noise = int(g["n_gp_draws"]), int(g["n_enc_noise"])
    w, eps, phase01, eps_u = [torch.tensor(g["gp_draw/%03d" % (n_gp + i)], dtype=torch.float64) for i in range(4)]   # one sample
    c = OF.build_cache("rbf_dimwise", sd("inducing_loc.optvar"), sd("kern.unconstrained_lengthscales"), sd("kern.unconstrained_variance"),
                       sd("Um.optvar"), OF.tril_from_packed(sd("Us_sqrt.optvar"), args.num_inducing),
                       dict(w=w, eps=eps, phase01=phase01, eps_u=eps_u))

    class OracleFlow(torch.nn.Module):
        def forward(self, z0, ts):
            return OF.rollout(z0, ts.double(), c, args.ode, solver)

    model = RM.ODEGPVAE(OracleFlow(), vae, args.Ndata, args.ode, args.frames, args.dt).train()
    monkeypatch.setattr(RM.Encoder, "sample", RM.Encoder.sample)      # restored after the test
    n_all = len([k for k in g if k.startswith("enc_noise/")])
    EH.patch_encoder_noise(RM, EH.Replay([g["enc_noise/%03d" % i] for i in range(n_noise, n_all)], torch.float64))
    ztl = {}
    sample_trajectories = model.sample_trajectories

    def spy(z, T, L=1):
        ztl["z"] = sample_trajectories(z, T, L)
        return ztl["z"]
    model.sample_trajectories = spy
    X = torch.tensor(EH.inputs("cfg3", g["meta"]["x_seed"]), dtype=torch.float64)
    with torch.no_grad():
        Xrec, _, _ = model(X, 1, T_custom=64)
    assert ztl["z"].shape == (1, X.shape[0], 64, 6) and Xrec.shape[:3] == (1, X.shape[0], 64)
    assert rel(ztl["z"].numpy(), g["ref64/fc_ztL"]) < 1e-6                            # fp32 storage of the stored trajectories
    assert rel(Xrec.sum((3, 4, 5)).numpy(), g["ref64/fc_xrec_sums"]) < 1e-10
