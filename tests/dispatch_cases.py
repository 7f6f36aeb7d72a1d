"""The dispatch matrix: one row per kernel instantiation the launch heuristics can pick (rbf_inst.cu: rbf_use_small,
rbf_small_cluster, rbf_fwd_use_tc, rbf_fwd_use_mma, rbf_bwd_use_tc, rbf_pick_shape; df_inst.cu: df_use_small, df_cluster,
df_pick_shape), each at a shape that reaches it.

tests/test_gpu_dispatch_matrix.py checks every row against the fp64 oracle and records which kernels the row launches;
tests/test_cpu_dispatch_matrix.py pins the family and cluster size of every row through the CPU-callable ABI queries, so a retuned
heuristic names the row that no longer reaches its kernel.

Row fields:
  family        what the row targets
  variant, order, D_in, D_out, M, S, N, L, methods (none: a field-only row, D_in is neither D_out nor 2 D_out)
  flags         None (default selection) or "mma" / "tc": the D > 8 tensor-path kernels forced through GpodeProblem.flags
  fwd_kernel    gpode_forward_kernel(): 0 FFMA, 1 mma.sync, 2 tcgen05
  cluster       gpode_cluster_size(): CTAs per thread-block cluster of the small-batch policies (grid z of their launches)
  fwd, bwd      sweep policy of the forward (k_field_fwd / k_rollout_fwd) and reverse (k_field_bwd / k_rollout_bwd) kernels, as it
                appears in the demangled kernel name with whitespace removed (default template arguments optional)
  fwd_per, bwd_per  states per CTA of those launches (grid x = ceil(N / per)); None where the row does not pin it
  extra         other kernels the backward must launch (parameter-gradient passes)
  grids         True: also run the irregular time grids (non-uniform, decreasing, T = 1, T = 2) on this row
  seed          seed of the row's parameters, states and upstream gradients
"""
import collections

Row = collections.namedtuple("Row", "family variant order D_in D_out M S N L methods flags fwd_kernel cluster fwd bwd fwd_per bwd_per "
                                    "extra grids seed")

FLAG_BITS = {None: 0, "mma": 1 | 4, "tc": 2 | 16}      # GPODE_FLAG_FWD_MMA | BWD_MMA, GPODE_FLAG_FWD_TCGEN05 | BWD_TCGEN05


def _pol(name, *args):
    """regex of a policy in a whitespace-free demangled name; DfPolicy's defaulted third argument (W = 0) may or may not be printed"""
    s = "%s<%s" % (name, ",".join(str(a) for a in args))
    return s + ("(,0)?>" if name == "DfPolicy" and len(args) == 2 else ">")


def _rbf(family, N, D_in, D_out, M, S, fwd, bwd, fwd_per, bwd_per, L=1, variant="rbf_dimwise", order=1, methods=("rk4",), flags=None,
         fwd_kernel=0, cluster=1, extra=(), grids=False, seed=0):
    return Row(family, variant, order, D_in, D_out, M, S, N, L, tuple(methods), flags, fwd_kernel, cluster, fwd, bwd, fwd_per, bwd_per,
               tuple(extra), grids, seed)


def _df(family, N, D, fwd, bwd, fwd_per, bwd_per, M=100, S=256, cluster=1, methods=("rk4",), grids=False):
    return Row(family, "df", 1, D, D, M, S, N, 1, tuple(methods), None, 0, cluster, fwd, bwd, fwd_per, bwd_per, ("k_df_pgrad<%d>" % D,),
               grids, 0)


def _small(DP):
    return _pol("RbfSmallPolicy", DP)


def _ffma(DP, R):
    return _pol("RbfPolicy", DP, R)


PG6 = "k_rbf_pgrad<6,1>"
PG_MMA = r"k_rbf_pgrad_mma<2,[12]>"

ROWS = [
    # ---- RBF small-batch policy (32 states per CTA, outputs split over a cluster along z) ----
    _rbf("rbf_small C=2", 2000, 6, 6, 100, 256, _small(6), _small(6), 32, 32, cluster=2, methods=("euler", "rk4"), grids=True),
    _rbf("rbf_small C=7 dimwise", 25, 7, 7, 100, 256, _small(8), _small(8), 32, 32, cluster=7, methods=("euler", "midpoint", "rk4"),
         grids=True),
    _rbf("rbf_small C=7 shared", 25, 7, 7, 100, 256, _small(8), _small(8), 32, 32, variant="rbf_shared", cluster=7),
    _rbf("rbf_small C=1 148 CTAs", 4736, 6, 6, 100, 256, _small(6), _small(6), 32, 32),
    _rbf("rbf_small C=1 148 CTAs L=2", 2368, 6, 6, 100, 256, _small(6), _small(6), 32, 32, L=2),
    _rbf("rbf_small DP=2 M=1 S=1", 100, 1, 1, 1, 1, _small(2), _small(2), 32, 32, methods=("euler", "rk4")),
    _rbf("rbf_small order2 16->8 C=8", 25, 16, 8, 64, 64, _small(16), _small(16), 32, 32, order=2, cluster=8, methods=("midpoint", "rk4")),
    # ---- RBF FFMA policy, D <= 8 (R states per thread; rbf_pick_shape) ----
    _rbf("rbf_ffma first non-small", 4737, 6, 6, 100, 256, _ffma(6, 1), _ffma(6, 1), 32, 32, extra=(PG6,), grids=True),
    _rbf("rbf_ffma R=2 fwd+bwd", 70001, 6, 6, 100, 256, _ffma(6, 2), _ffma(6, 2), 64, 128, extra=(PG6,)),
    _rbf("rbf_ffma R=4 bwd", 300000, 6, 6, 100, 256, _ffma(6, 4), _ffma(6, 4), 256, 512, extra=(PG6,)),
    _rbf("rbf_ffma DP4 R=4", 300000, 3, 3, 40, 50, _ffma(4, 4), _ffma(4, 4), 128, 128, extra=("k_rbf_pgrad<4,1>",)),
    _rbf("rbf_ffma order2 6->3", 6000, 6, 3, 100, 256, _ffma(6, 1), _ffma(6, 1), 32, 32, order=2, methods=("midpoint", "rk4"), extra=(PG6,)),
    _rbf("rbf_ffma shared", 9000, 6, 6, 100, 256, _ffma(6, 1), _ffma(6, 1), 32, 32, variant="rbf_shared", extra=(PG6,)),
    # ---- RBF FFMA policy, D > 8: the reverse sweep on FFMA, the parameter gradients on mma.sync ----
    _rbf("rbf_ffma DP16 + pgrad_mma N=25", 25, 16, 16, 512, 256, _ffma(16, 1), _ffma(16, 1), 32, 32, extra=(PG_MMA,), grids=True),
    _rbf("rbf_ffma DP16 + pgrad_mma N=32000", 32000, 16, 16, 512, 256, _ffma(16, 1), _ffma(16, 1), 32, 64, extra=(PG_MMA,)),
    _rbf("rbf_ffma DP16 L=2", 4099, 16, 16, 64, 48, _ffma(16, 1), _ffma(16, 1), 32, 32, L=2, extra=(PG_MMA,)),
    _rbf("rbf_ffma DP12 12->5 field", 20000, 12, 5, 101, 33, _ffma(12, 1), _ffma(12, 1), 32, 32, methods=(), extra=(PG_MMA,)),
    _rbf("rbf_ffma DP16 last FFMA N*L=32767", 32767, 16, 16, 64, 64, _ffma(16, 1), _ffma(16, 1), 32, 32, extra=(PG_MMA,)),
    _rbf("tensor DP16 first tensor N*L=32768", 32768, 16, 16, 64, 64, _pol("RbfMmaFwdPolicy", 16), _pol("RbfTcBwdPolicy", 16), None, 128,
         fwd_kernel=1),
    # ---- tensor path, both kernel families through GpodeProblem.flags ----
    _rbf("tc_bwd order2 16->8", 33000, 16, 8, 128, 128, _pol("RbfTcFwdPolicy", 16), _pol("RbfTcBwdPolicy", 16), 256, 128, order=2, flags="tc",
         fwd_kernel=2, methods=("midpoint", "rk4")),
    _rbf("mma_bwd order2 16->8", 33000, 16, 8, 128, 128, _pol("RbfMmaFwdPolicy", 16), _pol("RbfMmaBwdPolicy", 16), None, None, order=2,
         flags="mma", fwd_kernel=1, methods=("midpoint", "rk4"), extra=(PG_MMA,)),
    # (seed 1: at seed 0 the one shared variance gradient of the field VJP is a sum whose terms cancel 4,568-fold, see
    #  test_gpu_dispatch_matrix.variance_cancellation)
    _rbf("tc shared DP16", 33000, 16, 16, 100, 100, _pol("RbfTcFwdPolicy", 16), _pol("RbfTcBwdPolicy", 16), 256, 128, variant="rbf_shared",
         flags="tc", fwd_kernel=2, seed=1),
    _rbf("mma shared DP16", 33000, 16, 16, 100, 100, _pol("RbfMmaFwdPolicy", 16), _pol("RbfMmaBwdPolicy", 16), None, None,
         variant="rbf_shared", flags="mma", fwd_kernel=1, extra=(PG_MMA,), seed=1),
    _rbf("tc fwd at 15% padding M=190", 32768, 16, 16, 190, 256, _pol("RbfTcFwdPolicy", 16), _pol("RbfTcBwdPolicy", 16), 256, 128,
         fwd_kernel=2),
    _rbf("mma fwd above 15% padding M=189", 32768, 16, 16, 189, 256, _pol("RbfMmaFwdPolicy", 16), _pol("RbfTcBwdPolicy", 16), None, 128,
         fwd_kernel=1),
    # ---- DF small-batch policy (warp-split, 32 states per CTA, the rows of every chunk split over a cluster along z) ----
    _df("df_small C=7", 600, 6, _pol("DfPolicy", 6, 1, 8), _pol("DfPolicy", 6, 1, 8), 32, 32, cluster=7, methods=("euler", "midpoint", "rk4"),
        grids=True),
    _df("df_small C=6 D=8", 700, 8, _pol("DfPolicy", 8, 1, 8), _pol("DfPolicy", 8, 1, 8), 32, 32, cluster=6),
    _df("df_small C=5 D=5", 800, 5, _pol("DfPolicy", 5, 1, 8), _pol("DfPolicy", 5, 1, 8), 32, 32, cluster=5),
    _df("df_small C=3 D=7", 1200, 7, _pol("DfPolicy", 7, 1, 8), _pol("DfPolicy", 7, 1, 8), 32, 32, cluster=3),
    _df("df_small C=2", 1600, 6, _pol("DfPolicy", 6, 1, 8), _pol("DfPolicy", 6, 1, 8), 32, 32, cluster=2),
    _df("df_small C=8 M=3 S=1", 25, 6, _pol("DfPolicy", 6, 1, 8), _pol("DfPolicy", 6, 1, 8), 32, 32, M=3, S=1, cluster=8,
        methods=("euler", "rk4")),
    # ---- DF thread <-> state policy ----
    _df("df_large 32 threads", 4737, 6, _pol("DfPolicy", 6, 1), _pol("DfPolicy", 6, 1), 32, 32, grids=True),
    _df("df_large 64 threads D=8", 20000, 8, _pol("DfPolicy", 8, 1), _pol("DfPolicy", 8, 1), 64, 64),
    _df("df_large 128 threads", 40000, 6, _pol("DfPolicy", 6, 1), _pol("DfPolicy", 6, 1), 128, 128),
    _df("df_large fwd R=2", 80000, 6, _pol("DfPolicy", 6, 2), _pol("DfPolicy", 6, 1), 256, 128, methods=("midpoint", "rk4")),
]


def row_id(row):
    return row.family.replace(" ", "_")


def problem_fields(row):
    """(variant, L, N, D_in, D_out, M, S, flags) of the row's GpodeProblem"""
    return row.variant, row.L, row.N, row.D_in, row.D_out, row.M, row.S, FLAG_BITS[row.flags]
