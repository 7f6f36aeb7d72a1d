#!/usr/bin/env python
"""bench.py -- GP-ODE RK4 latent trajectory-steps/s, forward + backward, on N B200s of one node.

    python bench.py --gpus 1 --steps 3 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the reference's CPU path (oracle port) on the host cores

One "step" = one pass of the hot path over one batch: fixed-grid RK4 (3/8 rule) rollout of every
(trajectory, MC-sample) latent state over the T-point grid and its reverse sweep with all parameter
gradients.  Default workload = BASELINE.json configs[4] ("scaled data-parallel rollout": 65,536
trajectories x 8 MC samples, latent_dim 16, M=512 inducing, S=256 features, T=64, RK4).  At N GPUs the
SAME total problem is sharded by trajectory (SURVEY.md section 8d row 5: 65,536 / N trajectories x 8 samples
per GPU; `--scaling weak` keeps the full problem on every GPU instead): ranks hold independent trajectory
shards of one seeded z0, parameters and function samples are replicated, one NCCL all-reduce of the
kernel-level gradients per step (timed separately).  Unit of work: trajectory-step = one state advanced
over one grid interval, all 4 stages, forward and backward (SURVEY.md section 8d).

Prints ONE JSON line (rank 0).  `value` = kernel path with inputs resident in HBM; `e2e` = the same
metric through the public drop-in API (Flow.forward_samples -> build_cache -> rollout -> backward) with
z0 and the random draws coming from host memory every step and the loss / gradients read back.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "vae-gp-ode_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

# dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel (the reverse sweep), per launch, from the ncu capture named here
# (one B200; the stage saves make it ~9x the algorithmic 192 B per trajectory-step, and still < 1 % of the HBM peak)
TRAFFIC = {
    # dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel (fused tcgen05 reverse sweep), one launch of the full workload
    "cfg5_rbf_d16_m512_t64_rk4": (27873726464 + 9134574592, "k_rollout_bwd<RbfTcBwdPolicy<16>>, profiles/traffic_r02_cfg5_default.csv"),
}

WORKLOADS = {
    # BASELINE.json configs[4]; per GPU
    "cfg5_rbf_d16_m512_t64_rk4": dict(variant="rbf_dimwise", kernel="RBF", N=65536, L=8, D_in=16, D_out=16, M=512, S=256, T=64,
                                      order=1, method="rk4", ell=2.0, var=1.0),
    # smaller shapes for quick looks (not the headline)
    "cfg5_eighth": dict(variant="rbf_dimwise", kernel="RBF", N=8192, L=8, D_in=16, D_out=16, M=512, S=256, T=64, order=1,
                        method="rk4", ell=2.0, var=1.0),
    "cfg5_t3": dict(variant="rbf_dimwise", kernel="RBF", N=65536, L=8, D_in=16, D_out=16, M=512, S=256, T=3, order=1,
                    method="rk4", ell=2.0, var=1.0),   # config-5 shapes, 2 grid intervals: short enough for ncu --set full
    "cfg4_rbf_d6_m256_t2_euler": dict(variant="rbf_dimwise", kernel="RBF", N=1048576, L=1, D_in=6, D_out=6, M=256, S=256, T=2,
                                      order=1, method="euler", ell=2.0, var=1.0),
    "cfg4_df_d6_m256_t2_euler": dict(variant="df", kernel="DF", N=1048576, L=1, D_in=6, D_out=6, M=256, S=256, T=2,
                                     order=1, method="euler", ell=2.0, var=1.0),
    "cfg2_df_d6_m100_t16_rk4": dict(variant="df", kernel="DF", N=256, L=4, D_in=6, D_out=6, M=100, S=256, T=16, order=1,
                                    method="rk4", ell=2.0, var=1.0),
    "cfg2x_df_d6_m100_t16_rk4": dict(variant="df", kernel="DF", N=65536, L=4, D_in=6, D_out=6, M=100, S=256, T=16, order=1,
                                     method="rk4", ell=2.0, var=1.0),   # config-2 shapes with 256x the batch: fills the chip
    "cfg1_rbf_d6_m100_t16_rk4": dict(variant="rbf_dimwise", kernel="RBF", N=25, L=1, D_in=6, D_out=6, M=100, S=256, T=16, order=1,
                                     method="rk4", ell=2.0, var=1.0),
}
DEFAULT_WORKLOAD = "cfg5_rbf_d16_m512_t64_rk4"
STAGES = {"euler": 1, "midpoint": 2, "rk4": 4}


def algorithmic_work(w):
    """per trajectory-step, forward+backward (SURVEY.md section 8d): fwd+bwd = 3x flops, 2x SFU of one forward evaluation."""
    st = STAGES[w["method"]]
    if w["variant"] == "df":
        D = w["D_in"]
        f1 = 2 * (3 * w["S"] * D * D + w["M"] * (6 * D * D + 2 * D))
        s1 = 2 * w["S"] * D + w["M"] * D * D
    elif w["variant"] == "rbf_shared":
        f1 = 2 * (w["S"] + w["M"]) * (w["D_in"] + w["D_out"])
        s1 = w["S"] + w["M"]
    else:
        f1 = 2 * w["D_out"] * (w["S"] + w["M"]) * (w["D_in"] + 1)
        s1 = w["D_out"] * (w["S"] + w["M"])
    return dict(flops=3 * st * f1, sfu=2 * st * s1, hbm_bytes=3 * w["D_in"] * 4)


def pipe_model(w, tc_rates):
    """Per trajectory-step: the time each pipe needs at its peak / measured issue rate, in SM-cycles summed over the chip's SMs
    (divide by 148 x clock for seconds).  D <= 8 and DF: everything on the FP32 / MUFU pipes.  RBF at D > 8 on a chip-filling batch:
    the contractions run on tcgen05 WITH their precision splits (that is executed work, stated as such), per (128 states x 128 units)
    item, cycles as measured in isolation (tools/tc_probe2, tools/tc_probe3 -> profiles/tc_probe*_r02.json):
      forward  : kind::tf32, 3xTF32 along K = 56: 7 MMAs (128 x 128 x 8), ~452 cycles;
      reverse  : theta = 3 kind::f16 MMAs (fp16 head / remainder) + 1 kind::tf32 for the offsets, ~400 cycles;
                 Q = tau P: 16 kind::f16 (bf16 head + remainder planes) k-steps of N = 48, ~710 cycles (bound by reading the 64 KB tau tile);
                 PG = tau^T X' (inducing items only): 16 k-steps, ~810 cycles -- the parameter-gradient statistics come from the SAME tau,
                 so nothing is evaluated a third time (round 1: a separate recomputation pass).
    SFU: 2 transcendentals per (state, k, unit) and stage (SURVEY 8d), executed = algorithmic."""
    st = STAGES[w["method"]]
    work = algorithmic_work(w)
    out = {"sfu_alg_cycles": work["sfu"] / 16.0, "fp32_alg_cycles": work["flops"] / 256.0, "tensor_cycles": 0.0, "smem_cycles": 0.0,
           "fp32_residual_cycles": work["flops"] / 256.0}
    tensor_path = w["variant"] != "df" and w["D_in"] > 8 and w["N"] * w["L"] >= 32768
    if tensor_path:
        units = w["D_out"] * (w["S"] + w["M"])
        items_s, items_m = w["D_out"] * -(-w["S"] // 128), w["D_out"] * -(-w["M"] // 128)        # items per evaluation of a 128-state tile
        fwd = st * units / 16384.0 * 7 * tc_rates["tcgen05_tf32_n128_cycles_per_mma"]
        bwd = st * (items_s * (tc_rates["bwd_theta_cycles"] + tc_rates["bwd_q_cycles"]) +
                    items_m * (tc_rates["bwd_theta_cycles"] + tc_rates["bwd_q_cycles"] + tc_rates["bwd_pg_cycles"])) / 128.0
        out["tensor_cycles"] = fwd + bwd
        # L1 / shared-memory data pipe (128 B per cycle per SM), bytes the DESIGN moves per (128 states x 128 units) item:
        #   reverse: tau tile stored once by the epilogue warps (64 KB: bf16 head + remainder planes) and read by Q (64 KB) and, inducing
        #            items, PG (64 KB); theta: the 4 MMAs' unit operands 4 x 4 KB (the state operand comes from tensor memory); P tile
        #            16 k-steps x 1.5 KB; X' 16 x 1.5 KB (inducing); bulk-copy writes of the operand tiles 24 KB
        #   forward: per block of 256 units x 2 state tiles: 4 accumulators x 7 k-steps x (4 + 4 KB), bulk-copy write 42 KB, weights read by
        #            16 warps x 2 halves x 16 broadcast LDS.128 (one 128-B wavefront each)  -> per item-equivalent a quarter of it
        KB = 1024.0
        smem_bwd_s = (64 + 64 + 16 + 24 + 24) * KB / 128.0
        smem_bwd_m = smem_bwd_s + (64 + 24) * KB / 128.0
        smem_fwd = ((4 * 7 * 8 + 42) * KB / 128.0 + 16 * 2 * 16) / 4.0
        n_items = items_s + items_m
        out["smem_cycles"] = st * (items_s * smem_bwd_s + items_m * smem_bwd_m + n_items * smem_fwd) / 128.0
        out["tensor_split"] = {"forward": "3xTF32 (K = 56 for D_in = 16), tcgen05 kind::tf32",
                               "reverse_sweep": "theta: fp16 head + remainder, 3 kind::f16 + 1 kind::tf32 MMA; Q = tau P and PG = tau^T X': bf16 head + remainder "
                                                "planes of tau from shared memory, 16 kind::f16 k-steps each (fused: one tau per stage)"}
        # what stays on the FP32 pipe algorithmically: everything except the D_in-long dot products (forward 1x, backward 2x)
        moved = 3 * st * 2 * units * w["D_in"]
        out["fp32_residual_cycles"] = max(work["flops"] - moved, 0) / 256.0
        out["sfu_exec_cycles"] = work["sfu"] / 16.0
    else:
        rbf = w["variant"] != "df"
        ind = w["D_out"] * w["M"] if rbf else w["M"] * w["D_in"] ** 2
        out["sfu_exec_cycles"] = (work["sfu"] + (st * ind if rbf else 0)) / 16.0
    return out


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            return json.load(fh), "measured"
    return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0}, "fallback"


class ClockSampler:
    """nvidia-smi clock / throttle-reason samples while the timed region runs (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "200", "-f", self.path], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        try:
            rows = [r.strip().split(",") for r in open(self.path) if r.strip()]
            os.unlink(self.path)
        except Exception:
            return out
        sm, reasons, mx, pw = [], set(), None, []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                pw.append(float(r[2]))
                for nm, v in zip(names, r[3:7]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        if sm:
            busy = [s for s in sm if s > 0.5 * max(sm)] or sm
            out.update(sm_mhz=float(np.median(busy)), sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm),
                       power_w_max=max(pw) if pw else None)
        return out


def seeded_draw_patch(seed):
    """Seed the drop-in's host RNG helpers (same three helpers the reference has)."""
    from gpode_b200.core import kernels as K
    from gpode_b200.core import svpy as SV
    rng = np.random.RandomState(seed)
    K.sample_normal = lambda shape, seed=None: torch.tensor(rng.normal(size=shape).astype(np.float32))
    K.sample_uniform = lambda shape, seed=None: torch.tensor(rng.uniform(size=shape).astype(np.float32))
    SV.sample_normal = lambda shape, seed=None: torch.tensor(rng.normal(size=shape).astype(np.float32))


def build_model(w, device, seed):
    from gpode_b200.core.flow import Flow
    from gpode_b200.core.svpy import SVGP_Layer
    from gpode_b200.misc.constraint_utils import invsoftplus
    np.random.seed(seed)
    gp = SVGP_Layer(D_in=w["D_in"], D_out=w["D_out"], M=w["M"], S=w["S"], q_diag=False, dimwise=w["variant"] != "rbf_shared",
                    device=device, kernel=w["kernel"])
    with torch.no_grad():
        gp.kern.unconstrained_lengthscales.copy_(invsoftplus(torch.full_like(gp.kern.unconstrained_lengthscales, w["ell"])))
        gp.kern.unconstrained_variance.copy_(invsoftplus(torch.full_like(gp.kern.unconstrained_variance, w["var"])))
    flow = Flow(diffeq=gp, order=w["order"], solver=w["method"], use_adjoint=False)
    return gp, flow


def tc_forward(w):
    """mirrors rbf_fwd_use_tc (csrc/rbf.h): the tensor-memory forward adds one launch (its operand-tile pack) per step"""
    if w["variant"] == "df" or w["D_in"] <= 8 or w["N"] * w["L"] < 32768:
        return False
    units = (-(-w["S"] // 256) + -(-w["M"] // 256)) * 256
    return units * 100 <= (w["S"] + w["M"]) * 115


def kernel_launches(w):
    """kernels of libgpode.so launched by one forward + backward rollout call (csrc/api.cu):
    RBF forward: k_rbf_pack [+ k_rbf_pack_tc] + k_rollout_fwd; backward: k_rbf_pack + k_rollout_bwd + (D <= 8: k_rbf_pgrad; D > 8 on a chip-filling
    batch: k_rbf_pack_tcb, the parameter gradients come out of the fused reverse sweep) + 2 finalize kernels;
    DF forward: k_df_pack + k_rollout_fwd; backward: k_df_pack + k_rollout_bwd + k_df_pgrad + finalize."""
    if w["variant"] == "df":
        return 6
    return 8 if tc_forward(w) else 7


def run_ours(args):
    import torch.distributed as dist
    import gpode_b200  # noqa: F401  (fails loudly if libgpode.so is missing)
    from gpode_b200.core.svpy import FieldSample
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device; there is no CPU fallback (use --impl reference for the CPU baseline)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    w = dict(WORKLOADS[args.workload])
    if args.scale != 1.0:
        w["N"] = max(1, int(w["N"] * args.scale))
    from gpode_b200.parallel import shard_bounds
    N_total = w["N"]
    if args.scaling == "strong" and world > 1:
        lo, hi = shard_bounds(N_total, rank, world)     # contiguous trajectory shard of ONE global problem
    else:
        lo, hi = 0, N_total
    w["N"] = hi - lo
    N, L, T, D = w["N"], w["L"], w["T"], w["D_in"]
    steps_per_pass = N * L * (T - 1)                      # this rank's share
    steps_job = (N_total * L * (T - 1)) if (args.scaling == "strong" or world == 1) else world * N_total * L * (T - 1)
    work = algorithmic_work(w)

    # ---- resident inputs: L function samples (seeds 10..), z0, dL/dtraj ----------------------------------
    gp, flow = build_model(w, dev, seed=1)
    samples = []
    with torch.no_grad():
        for l in range(L):
            seeded_draw_patch(10 + l)
            gp.build_cache()
            samples.append(gp.field_sample())
    fs = FieldSample.stack(samples)
    leaf = lambda v: v.detach().clone().requires_grad_(True)
    Z, nu, ell, var = leaf(fs.Z), leaf(fs.nu), leaf(fs.ell), leaf(fs.var)
    # ONE seeded global z0 / upstream gradient (the same on every rank); strong scaling slices this rank's trajectories out of it,
    # weak scaling gives every rank its own draw
    gen = torch.Generator(device=dev).manual_seed(1000 if args.scaling == "strong" else 1000 + rank)
    z0 = torch.randn(N_total, D, device=dev, generator=gen)[lo:hi].contiguous().requires_grad_(True)
    dtraj = torch.randn(L, N_total, T, D, device=dev, generator=gen)[:, lo:hi].contiguous()
    ts = 0.1 * torch.arange(T, dtype=torch.float, device=dev)
    from gpode_b200 import gp_rollout

    from gpode_b200.parallel import allreduce_gradients

    def allreduce_grads(tensors):
        """one flat NCCL all-reduce of the gradient buffers (in place); no-op on a single GPU"""
        if world > 1:
            allreduce_gradients(tensors)
            return True
        return None

    ev = lambda: torch.cuda.Event(enable_timing=True)

    last = {}       # --dump-outputs: what the last timed step of each path returned

    def kernel_step(record):
        for v in (z0, Z, nu, ell, var):
            v.grad = None
        e0, e1, e2, e3 = ev(), ev(), ev(), ev()
        e0.record()
        traj = gp_rollout(z0, ts, Z, nu, fs.eps, fs.phase, fs.w, ell, var, w["variant"], w["order"], w["method"], fs.B)
        if args.dump_outputs and record is not None and len(record) == args.steps - 1:
            last["traj"] = traj.detach()          # the last timed step's output; sampled once the timed loop is over
        e1.record()
        traj.backward(dtraj)
        e2.record()
        allreduce_grads([Z.grad, nu.grad, ell.grad, var.grad] + ([fs.B.grad] if (fs.B is not None and fs.B.grad is not None) else []))
        e3.record()
        if record is not None:
            record.append((e0, e1, e2, e3))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn(None)
        barrier()
        sampler = ClockSampler(local)
        sampler.start()
        rec = []
        s, e = ev(), ev()
        s.record()
        for _ in range(steps):
            fn(rec)
        e.record()
        barrier()
        clocks = sampler.stop()
        ms = s.elapsed_time(e)
        if world > 1:
            tms = torch.tensor([ms], device=dev)
            dist.all_reduce(tms, op=dist.ReduceOp.MAX)
            ms = tms.item()
        return ms, rec, clocks

    ms_total, rec, clocks = timed(kernel_step, args.steps, args.warmup)
    if args.dump_outputs:
        last["traj"] = dump_rows(last["traj"].reshape(-1, T, D))
    ms_step = ms_total / args.steps
    fwd_ms = float(np.mean([a.elapsed_time(b) for a, b, _, _ in rec]))
    bwd_ms = float(np.mean([b.elapsed_time(c) for _, b, c, _ in rec]))
    allreduce_ms = float(np.mean([c.elapsed_time(d) for _, _, c, d in rec]))
    if world > 1:   # the slowest rank's phases (the step time already is the max over ranks)
        ph = torch.tensor([fwd_ms, bwd_ms, allreduce_ms], device=dev)
        dist.all_reduce(ph, op=dist.ReduceOp.MAX)
        fwd_ms, bwd_ms, allreduce_ms = [float(v) for v in ph.tolist()]
    value = steps_job / (ms_step * 1e-3)

    # ---- end to end through the drop-in API, host buffers in the timed region --------------------------
    z0_host = z0.detach().cpu().pin_memory()
    h2d = [0]
    d2h = [0]
    params = [gp.kern.unconstrained_lengthscales, gp.kern.unconstrained_variance, gp.inducing_loc.optvar, gp.Um.optvar,
              gp.Us_sqrt.optvar]
    # function-sample draws on the device (gpode_b200.set_rng: one Philox launch per rollout instead of host numpy + H2D copies; the
    # reference's own host draws are unseeded, so no number of them is pinned anywhere): the step's host input is z0
    import gpode_b200
    gpode_b200.set_rng("device", seed=77 if args.scaling == "strong" else 77 + rank)   # strong: every rank draws the SAME function samples

    def e2e_step(record):
        for p_ in params:
            p_.grad = None
        z = z0_host.to(dev, non_blocking=True).requires_grad_(True)
        traj = flow.forward_samples(z, ts, L)                 # L function samples (device draws, batched setup), one rollout launch
        loss = (traj * dtraj).sum() + flow.kl()
        loss.backward()
        flat = allreduce_grads([p_.grad for p_ in params])
        host = [loss.detach().cpu()] + [p_.grad.cpu() for p_ in params] + [z.grad.cpu()]
        if args.dump_outputs:
            last["e2e"] = host
        if record is not None and not h2d[0]:
            h2d[0] = z0_host.numel() * 4
            d2h[0] = sum(h.numel() * 4 for h in host)

    e2e_warm = min(args.warmup, 3)
    ms_e2e, _, _ = timed(e2e_step, args.steps, e2e_warm)
    e2e_value = steps_job / (ms_e2e / args.steps * 1e-3)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last, dict(z0=z0, Z=Z, nu=nu, ell=ell, var=var, B=fs.B), rank)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks, peak_src = measured_peaks()
    sm_max = float(peaks.get("sm_max_mhz", 1965.0)) * 1e6
    fp32_peak = 148 * 128 * 2 * sm_max          # FFMA lanes x 2 flop x max SM clock
    sfu_peak = 148 * 16 * sm_max
    per_gpu_rate = steps_per_pass / (ms_step * 1e-3)
    achieved_tflops = work["flops"] * per_gpu_rate / 1e12
    # measured issue rates of the tensor pipes (tools/tc_probe2, tools/mma_peak; fallbacks = the round-2 measurements under profiles/)
    tc_rates = {"tcgen05_tf32_n128_cycles_per_mma": 452.0 / 7.0, "bwd_theta_cycles": 400.0, "bwd_q_cycles": 710.0, "bwd_pg_cycles": 810.0,
                "source": "profiles/tc_probe2_r02.json, tools/tc_probe3 (csrc/rbf_bwd_tc.cuh header)"}
    probe = os.path.join(ROOT, "tools", "tc_probe2")
    if world == 1 and os.path.exists(probe) and not args.no_cpu_baseline:
        try:
            pj = json.loads(subprocess.check_output([probe], timeout=120).decode().strip().splitlines()[-1])
            tc_rates["tcgen05_tf32_n128_cycles_per_mma"] = pj["cycles_per_rep"]["theta_7xSS_tf32_N128"][0] / 7.0
            tc_rates["source"] = "tools/tc_probe2 run inside this bench; tools/tc_probe3 (csrc/rbf_bwd_tc.cuh header)"
        except Exception:
            pass
    pm = pipe_model(w, tc_rates)
    chip_cycles_per_s = 148 * sm_max
    pipes = {"sfu": round(pm["sfu_alg_cycles"] * per_gpu_rate / chip_cycles_per_s, 4),
             "sfu_executed": round(pm["sfu_exec_cycles"] * per_gpu_rate / chip_cycles_per_s, 4),
             "tensor": round(pm["tensor_cycles"] * per_gpu_rate / chip_cycles_per_s, 4),
             "smem": round(pm["smem_cycles"] * per_gpu_rate / chip_cycles_per_s, 4),
             "fp32_residual": round(pm["fp32_residual_cycles"] * per_gpu_rate / chip_cycles_per_s, 4)}
    binding = max(("sfu", "tensor", "smem", "fp32_residual"), key=lambda k: pipes[k])
    frac_fp32_alg = round(work["flops"] * per_gpu_rate / fp32_peak, 4)
    roof = {"bound": {"sfu": "sfu", "tensor": "tensor", "smem": "smem_pipe", "fp32_residual": "fp32_fma"}[binding], "frac": pipes[binding], "pipes": pipes,
            "achieved": round(achieved_tflops, 3), "peak": round(fp32_peak / 1e12, 2), "unit": "TFLOP/s",
            "frac_fp32_algorithmic": frac_fp32_alg,
            "traffic": TRAFFIC.get(args.workload, (None, None))[0], "traffic_source": TRAFFIC.get(args.workload, (None, None))[1],
            "peak_source": "FP32: 148 SM x 128 lanes x 2 x sm_max_mhz of MEASURED_PEAKS.json (%s); SFU: 148 x 16 / clk; tensor: measured issue rates (%s); "
                           "not an HBM-bound path" % (peak_src, tc_rates["source"]),
            "note": ("frac = the fraction of the measured time the BINDING pipe needs at its peak rate (pipes: sfu = algorithmic transcendentals, "
                     "sfu_executed = what the kernels evaluate (D <= 8: incl. the re-evaluation in the separate parameter-gradient pass; D > 8: fused, "
                     "equal to algorithmic), tensor = the executed MMAs incl. their precision splits "
                     "at the measured issue rates, smem = the bytes the tcgen05 kernels move through the L1 / shared-memory data pipe by design "
                     "(tau tile stored once and read by two products, operand tiles) at 128 B per cycle per SM -- ncu of the fused reverse sweep: "
                     "l1tex data pipe 97.6 % busy (tensor-core operand reads 52.5 % + LSU 45.1 %, profiles/ncu_r02_cfg5_t3_bwd_tc.txt), "
                     "fp32_residual = algorithmic FP32 work that stays on the FMA pipe).  achieved / peak / "
                     "frac_fp32_algorithmic keep the SURVEY 8(d) definition: ALL algorithmic flops over the FP32-pipe peak (can exceed what the "
                     "FP32 pipe really executes once the dot products run on tensor cores)."),
            "tensor_split": pm.get("tensor_split"),
            "sfu_achieved_tops": round(work["sfu"] * per_gpu_rate / 1e12, 4), "sfu_peak_tops": round(sfu_peak / 1e12, 3),
            "hbm_achieved_gbs": round(work["hbm_bytes"] * per_gpu_rate / 1e9, 3), "hbm_peak_gbs": peaks.get("hbm_gbs"),
            "hbm_frac": round(work["hbm_bytes"] * per_gpu_rate / 1e9 / float(peaks.get("hbm_gbs", 6650.0)), 6),
            "flops_per_traj_step": work["flops"], "sfu_per_traj_step": work["sfu"], "bytes_per_traj_step": work["hbm_bytes"],
            "fwd_call_ms": round(fwd_ms, 3), "bwd_call_ms": round(bwd_ms, 3), "allreduce_ms": round(allreduce_ms, 3)}
    peaks_bin = os.path.join(ROOT, "tools", "peaks")
    if world == 1 and os.path.exists(peaks_bin) and not args.no_cpu_baseline:
        try:
            pk = json.loads(subprocess.check_output([peaks_bin], timeout=120).decode().strip().splitlines()[-1])
            roof["ffma_measured_tflops"] = pk["ffma_tflops"]
            roof["mufu_measured_tops"] = pk["ex2_tops"]
        except Exception as exc:  # the microbenchmark is informative only
            roof["ffma_measured_tflops"] = "unavailable: %s" % exc

    line = {"metric": "GP-ODE RK4 latent traj-steps/s fwd+bwd", "value": round(value, 1), "unit": "traj-steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_step, 3), "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "dtype_note": ("fp32 inputs, outputs, accumulation and transcendentals; where dot products run on tensor cores (RBF, D_in > 8) the operands are "
                           "split so that >= 16-21 mantissa bits enter every product: forward 3xTF32; fused reverse sweep: fp16 head + 2^11-scaled remainder "
                           "for theta, bf16 head + remainder planes of tau (fp32 exponent range) for the state- and parameter-gradient products, fp32 "
                           "accumulation in tensor memory; the per-rollout setup (K(Z,Z), Cholesky, solves) runs in fp64"),
            "config": {"workload": args.workload, "per_gpu": {k: w[k] for k in ("N", "L", "T", "D_in", "D_out", "M", "S", "method", "order", "variant")},
                       "total_trajectories": N_total if args.scaling == "strong" or world == 1 else world * N_total,
                       "traj_steps_per_gpu_per_step": steps_per_pass, "traj_steps_per_job_per_step": steps_job,
                       "parallelism": "dp%d (%s: trajectory shards of one seeded problem, params and function samples replicated, one all-reduce of the kernel-level gradients)" % (world, args.scaling),
                       "cache": "inputs and saves (%.1f GB) far exceed the 126 MB L2; no flush needed" %
                                ((T - 1) * STAGES[w["method"]] * (2 * D + w["D_out"]) * N * L * 4 / 1e9)},
            "roofline": roof,
            "e2e": {"value": round(e2e_value, 1), "unit": "traj-steps/s", "h2d_bytes_per_step": int(h2d[0]), "d2h_bytes_per_step": int(d2h[0]),
                    "ms_per_step": round(ms_e2e / args.steps, 3), "draws": "device (Philox4x32-10, gpode_b200.set_rng('device'))"},
            "gpu_launches": kernel_launches(w) * args.steps, "clocks": clocks}
    if world == 1 and not args.no_cpu_baseline:
        try:
            line["cpu_baseline"] = cpu_baseline(w, reps=3, warmup=1)
        except Exception as exc:
            line["cpu_baseline"] = {"value": None, "unit": "traj-steps/s", "cores": os.cpu_count(), "kind": "reference", "sample": "failed: %s" % exc}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


DUMP_ROWS = 4096
DUMP_MAX_BYTES = 64 << 20


def dump_rows(x):
    """a fixed sample of DUMP_ROWS rows of x (all rows if fewer): drawn by RandomState(0), in ascending order"""
    if x.shape[0] <= DUMP_ROWS:
        return x
    idx = np.sort(np.random.RandomState(0).choice(x.shape[0], size=DUMP_ROWS, replace=False))
    return x[torch.as_tensor(idx, device=x.device)]


def dump_outputs(out_dir, last, leaves, rank):
    """Writes what the timed paths returned in their last step as <out_dir>/<name>.npy (float32), rank 0 only, at most
    DUMP_MAX_BYTES in all.  Per-trajectory outputs are sampled by dump_rows: the trajectories over their (MC sample, trajectory)
    rows (the whole (L,N,T,D) tensor is 2 GB at the default workload), the z0 gradients over the trajectories.
    Kernel path: trajectories, gradients of z0 and of every kernel-level leaf.  End-to-end path (prefix e2e_): the loss, the
    gradients of the five model parameters and of z0; its device draws advance with every step, so these depend on --steps and
    --warmup as well.  At N > 1 GPUs the trajectories and z0 gradients are rank 0's shard; the parameter gradients are all-reduced."""
    if rank != 0:
        return
    arrays = {"traj_sample": last["traj"]}
    for k, v in leaves.items():
        if v is not None and v.grad is not None:
            arrays["grad_" + k] = dump_rows(v.grad) if k == "z0" else v.grad
    names = ["loss", "grad_unconstrained_lengthscales", "grad_unconstrained_variance", "grad_inducing_loc", "grad_Um", "grad_Us_sqrt", "grad_z0"]
    for k, v in zip(names, last["e2e"]):
        arrays["e2e_" + k] = dump_rows(v) if k == "grad_z0" else v
    total = sum(v.numel() * 4 for v in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit("--dump-outputs: %d bytes exceed the %d-byte limit" % (total, DUMP_MAX_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v.detach().float().cpu().numpy())


def cpu_sample_shape(w):
    """bounded sample of the workload for the CPU arm: BASELINE.md section 3 asks for 1,024 trajectories x 1 MC sample at the workload's
    own T; the reference keeps the whole unrolled solve in its autograd graph (~1.1 GB per 64 trajectories x 60 evaluations at
    D = 16, M = 512), so the trajectory count is halved until the estimate fits in a quarter of the host's free memory."""
    s = dict(w)
    s["L"] = 1
    s["N"] = min(1024, w["N"])
    s["T"] = min(64, w["T"])
    try:
        import psutil
        avail = psutil.virtual_memory().available
    except Exception:
        avail = 32 << 30
    per_eval_state = 4.0 * w["D_out"] * (w["M"] * (36 if w["variant"] == "df" else 1) + w["S"]) * 6     # bytes: ~6 saved (D_out, M, N)-sized temporaries
    evals = (s["T"] - 1) * STAGES[w["method"]]
    while s["N"] > 32 and per_eval_state * evals * s["N"] > 0.25 * avail:
        s["N"] //= 2
    return s


def cpu_baseline(w, reps, warmup):
    """The reference's CPU path on this box's host cores, on a bounded sample of the workload, in a subprocess with CUDA hidden (the
    reference puts its parameters on cuda:0 whenever a GPU is visible).  kind = "reference": the reference's OWN SVGP_Layer / Flow
    modules (oracle/_ref, the verbatim copy oracle/fetch_ref.py makes; oracle/ref_timing.py) -- timed region build_cache + rollout +
    backward; falls back to the bit-identical port (oracle/port_fp32.py, kind = "port") only where that copy is absent."""
    cores = os.cpu_count() or 1
    s = cpu_sample_shape(w)
    sys.path.insert(0, ROOT)
    from oracle import reference_harness as rh
    kind = "reference" if rh.reference_available() else "port"
    call = ("from oracle import ref_timing as R; sec = R.time_reference(" if kind == "reference" else "from oracle import port_fp32 as R; sec = R.time_rollout(")
    code = ("import sys, json, warnings; warnings.filterwarnings('ignore'); sys.path.insert(0, %r); import torch; %s%r, %d, %d, %d, %d, %d, %d, %d, %r, "
            "reps=%d, warmup=%d, threads=%d); print(json.dumps(sec))"
            % (ROOT, call, s["variant"], s["N"], s["D_in"], s["D_out"], s["M"], s["S"], s["T"], s["order"], s["method"], reps, warmup, cores))
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    proc = subprocess.run([sys.executable, "-c", code], env=env, timeout=1500, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    if proc.returncode != 0:
        raise RuntimeError("cpu baseline subprocess failed: %s" % proc.stderr.decode()[-2000:])
    sec = json.loads(proc.stdout.decode().strip().splitlines()[-1])
    n_steps = s["N"] * (s["T"] - 1)
    try:
        cpu_model = [ln.split(":", 1)[1].strip() for ln in open("/proc/cpuinfo") if ln.startswith("model name")][0]
    except Exception:
        cpu_model = "unknown"
    what = ("the reference's own SVGP_Layer + Flow (oracle/_ref, unmodified; torchdiffeq replaced by the restated fixed-grid loop), build_cache + rollout + backward"
            if kind == "reference" else "oracle/port_fp32.py (the reference's op sequence; oracle/_ref absent), rollout + backward")
    return {"value": round(n_steps / sec, 1), "unit": "traj-steps/s", "cores": cores, "kind": kind,
            "sample": "%d trajectories x 1 MC sample, T=%d, same D=%d M=%d S=%d %s %s; best of %d after %d warm-up; %s; torch CPU fp32, %d threads on %s" % (
                s["N"], s["T"], s["D_in"], s["M"], s["S"], s["variant"], s["method"], reps, warmup, what, cores, cpu_model),
            "seconds_per_pass": round(sec, 3)}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path (the reference's modules from oracle/_ref; the port only if
    that copy is absent), all host threads, same metric / unit / config; a bounded sample per step (cpu_sample_shape)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = dict(WORKLOADS[args.workload])
    base = cpu_baseline(w, reps=args.steps, warmup=args.warmup)
    value = base["value"]
    line = {"impl": "reference", "metric": "GP-ODE RK4 latent traj-steps/s fwd+bwd", "value": value, "unit": "traj-steps/s",
            "n_gpus": int(os.environ.get("WORLD_SIZE", str(args.gpus))), "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(base["seconds_per_pass"] * 1e3, 3), "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": args.workload, "per_gpu": {k: w[k] for k in ("N", "L", "T", "D_in", "D_out", "M", "S", "method", "order", "variant")}},
            "cpu_baseline": base, "e2e": {"value": value, "unit": "traj-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--scale", type=float, default=1.0, help="scale the trajectory count (debugging only; not a valid bench line)")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="N > 1 GPUs: strong = the workload's trajectories are sharded over the ranks (SURVEY 8d row 5); weak = every rank runs the full workload")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed paths computed in their last step to DIR/<name>.npy (float32, a fixed sample of the trajectories)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
