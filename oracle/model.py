"""The reference's full model around the GP flow, restated: conv VAE (experiments/model/core/vae.py), ODEGPVAE
(core/odegpvae.py), build_model / elbo / compute_loss (create_model.py) and initialize_and_fix_kernel_parameters
(core/initialization.py).  TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

Same module names, parameter names (so the reference's state_dict loads strictly), operation order and random-draw order as the
reference; ``SVGP_Layer`` / ``Flow`` are the drop-in classes of gpode_b200 (INTEGRATION.md section 1).  Pinned against the
reference by tests/test_oracle_elbo.py: with the stored draws and the stored fp64 flow boundary, it reproduces the reference's fp64
ELBO terms and every encoder / decoder gradient stored in tests/golden/elbo_*.npz.
"""
import torch
import torch.nn as nn
from torch.distributions import Normal
from torch.distributions import kl_divergence as kl

from gpode_b200.core.flow import Flow
from gpode_b200.core.svpy import SVGP_Layer
from gpode_b200.misc.constraint_utils import invsoftplus


class Flatten(nn.Module):
    def forward(self, x):
        return x.view(x.size(0), -1)


class UnFlatten(nn.Module):
    def __init__(self, w):
        super().__init__()
        self.w = w

    def forward(self, x):
        return x.view(x.size(0), -1, self.w, self.w)


class Encoder(nn.Module):
    """3 x (5x5 conv, stride 2) on 28 x 28 frames -> (4 n_filt, 4, 4) -> mean and log-variance of the latent initial state"""

    def __init__(self, steps=1, n_filt=8, q=8):
        super().__init__()
        h_dim = n_filt * 4 ** 3
        self.cnn = nn.Sequential(
            nn.Conv2d(steps, n_filt, kernel_size=5, stride=2, padding=(2, 2)),
            nn.BatchNorm2d(n_filt),
            nn.ReLU(),
            nn.Conv2d(n_filt, n_filt * 2, kernel_size=5, stride=2, padding=(2, 2)),
            nn.BatchNorm2d(n_filt * 2),
            nn.ReLU(),
            nn.Conv2d(n_filt * 2, n_filt * 4, kernel_size=5, stride=2, padding=(2, 2)),
            nn.ReLU(),
            Flatten())
        self.fc = nn.Linear(h_dim, 2 * q)

    def forward(self, x):
        z = self.fc(self.cnn(x))
        q = z.shape[1] // 2
        return z[:, :q], z[:, q:]

    def sample(self, mu, logvar):
        std = torch.exp(0.5 * logvar)
        return mu + std * torch.randn_like(std)

    def q_dist(self, mu_s, logv_s, mu_v=None, logv_v=None):
        if mu_v is not None:
            mu_s, logv_s = torch.cat([mu_s, mu_v], 1), torch.cat([logv_s, logv_v], 1)
        return Normal(mu_s, torch.exp(0.5 * logv_s))


class Decoder(nn.Module):
    """latent positions -> fc -> (4 n_filt, 4, 4) -> 4 transposed convs -> 28 x 28 Bernoulli means"""

    def __init__(self, n_filt=8, q=8, distribution="bernoulli"):
        super().__init__()
        h_dim = n_filt * 4 ** 3
        self.distribution = distribution
        self.fc = nn.Linear(q, h_dim)
        self.decnn = nn.Sequential(
            UnFlatten(4),
            nn.ConvTranspose2d(h_dim // 16, n_filt * 8, kernel_size=3, stride=1, padding=(0, 0)),
            nn.BatchNorm2d(n_filt * 8),
            nn.ReLU(),
            nn.ConvTranspose2d(n_filt * 8, n_filt * 4, kernel_size=5, stride=2, padding=(1, 1)),
            nn.BatchNorm2d(n_filt * 4),
            nn.ReLU(),
            nn.ConvTranspose2d(n_filt * 4, n_filt * 2, kernel_size=5, stride=2, padding=(1, 1), output_padding=(1, 1)),
            nn.BatchNorm2d(n_filt * 2),
            nn.ReLU(),
            nn.ConvTranspose2d(n_filt * 2, 1, kernel_size=5, stride=1, padding=(2, 2)),
            nn.Sigmoid())

    def forward(self, z, dims):
        L, N, T, q = dims
        return self.decnn(self.fc(z.contiguous().view([L * N * T, q]))).view([L, N, T, 1, 28, 28])

    def log_prob(self, x, z, L=1):
        """log Bernoulli(x | z) per element, x repeated over the L samples: (L,N,T,1,28,28)"""
        XL = x.repeat([L] + [1] * x.ndim)
        return torch.log(z) * XL + torch.log(1 - z) * (1 - XL)


class VAE(nn.Module):
    def __init__(self, frames=5, n_filt=8, latent_dim=8, order=1, device="cpu", distribution="bernoulli"):
        super().__init__()
        self.encoder = Encoder(steps=1, n_filt=n_filt, q=latent_dim)
        if order == 2:
            self.encoder_v = Encoder(steps=frames, n_filt=n_filt, q=latent_dim)
        self.decoder = Decoder(n_filt=n_filt, q=latent_dim, distribution=distribution)
        self.prior = Normal(torch.zeros(latent_dim * order, device=device), torch.ones(latent_dim * order, device=device))


class ODEGPVAE(nn.Module):
    def __init__(self, flow, vae, num_observations, order, steps, dt):
        super().__init__()
        self.flow, self.vae = flow, vae
        self.num_observations, self.order, self.v_steps, self.dt = num_observations, order, steps, dt

    def build_decoding(self, ztL, dims):
        L, N, T, D = dims
        if self.order == 1:
            return self.vae.decoder(ztL, [L, N, T, D])
        q = D // 2
        return self.vae.decoder(ztL[:, :, :, :q], [L, N, T, q])

    def sample_trajectories(self, z0, T, L=1):
        ts = self.dt * torch.arange(T, dtype=torch.float).to(z0.device)
        return torch.cat([self.flow(z0, ts).unsqueeze(0) for _ in range(L)], 0)

    def forward(self, X, L=1, T_custom=None):
        N, T = X.shape[0], X.shape[1]
        s0_mu, s0_logv = self.vae.encoder(X[:, 0])
        z0 = self.vae.encoder.sample(s0_mu, s0_logv)
        v0_mu, v0_logv = None, None
        if self.order == 2:
            v0_mu, v0_logv = self.vae.encoder_v(torch.squeeze(X[:, 0:self.v_steps], 2))
            v0 = self.vae.encoder_v.sample(v0_mu, v0_logv)
            z0 = torch.cat([z0, v0], 1)
        if T_custom:
            T = T_custom
        ztL = self.sample_trajectories(z0, T, L)
        Xrec = self.build_decoding(ztL, [L, N, T, z0.shape[1]])
        return Xrec, (s0_mu, s0_logv), (v0_mu, v0_logv)


def build_model(args):
    gp = SVGP_Layer(D_in=args.D_in, D_out=args.D_out, M=args.num_inducing, S=args.num_features, dimwise=args.dimwise,
                    q_diag=args.q_diag, device=args.device, kernel=args.kernel)
    flow = Flow(diffeq=gp, order=args.ode, solver=args.solver, use_adjoint=args.use_adjoint)
    vae = VAE(frames=args.frames, n_filt=args.n_filt, latent_dim=args.latent_dim, order=args.ode, device=args.device)
    return ODEGPVAE(flow=flow, vae=vae, num_observations=args.Ndata, order=args.ode, steps=args.frames, dt=args.dt)


def elbo(model, X, Xrec, s0_mu, s0_logv, v0_mu, v0_logv, L):
    q = model.vae.encoder.q_dist(s0_mu, s0_logv, v0_mu, v0_logv)
    kl_reg = kl(q, model.vae.prior).sum(-1)
    if model.vae.decoder.distribution != "bernoulli":
        raise ValueError("Currently only bernoulli dist implemented")
    lhood = model.vae.decoder.log_prob(X, Xrec, L).sum([2, 3, 4, 5]).mean(0)
    kl_u = model.flow.kl()
    return lhood.mean(), kl_reg.mean(), kl_u


def compute_loss(model, data, L):
    Xrec, (s0_mu, s0_logv), (v0_mu, v0_logv) = model(data, L)
    lhood, kl_reg, kl_gp = elbo(model, data, Xrec, s0_mu, s0_logv, v0_mu, v0_logv, L)
    loss = -(lhood * model.num_observations - kl_reg * model.num_observations - kl_gp)
    return loss, -lhood, kl_reg, kl_gp


def initialize_and_fix_kernel_parameters(model, lengthscale_value=1.25, variance_value=0.5, fix=False):
    k = model.flow.odefunc.diffeq.kern
    with torch.no_grad():
        k.unconstrained_lengthscales.copy_(invsoftplus(lengthscale_value * torch.ones_like(k.unconstrained_lengthscales)))
        k.unconstrained_variance.copy_(invsoftplus(variance_value * torch.ones_like(k.unconstrained_variance)))
    k.unconstrained_lengthscales.requires_grad_(not fix)
    k.unconstrained_variance.requires_grad_(not fix)
    return model
