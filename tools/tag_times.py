"""Where a solve spends its time (dev tool): builds a -DMPC_TIMING copy of the library, runs one batch and prints the cycles
between the driver's tags (mpc_solve.h: ex.tag(n)), summed over all problems.  python tools/tag_times.py N B [early]

Settings: bench.py's headline (SolverSettings.early_certified: polish_retry 4, stateless) with early polish on or off; termination
checks every CHECK iterations (environment, default 50 with early polish as the bench, 25 without).  CUDAMPC_TIMING_LIB names another
timing build (e.g. the parent commit's) instead of the in-tree one."""
import ctypes as C, dataclasses, os, subprocess, sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
dbg = os.environ.get("CUDAMPC_TIMING_LIB") or os.path.join(ROOT, "rrt_mpc_b200", "libcudampc_timing.so")
if "--build" in sys.argv or not os.path.exists(dbg):
    import __graft_entry__ as G
    G.build_cuda(dbg, extra=["-DMPC_TIMING"], tag="_timing")
    if "--build" in sys.argv: sys.exit(0)
import rrt_mpc_b200._lib as L
L.LIB_PATH = dbg
import torch
from rrt_mpc_b200 import MPCController, SolverSettings, MPCConfig
from rrt_mpc_b200.synthetic import make_batch
N, B = int(sys.argv[1]), int(sys.argv[2]); early = bool(int(sys.argv[3])) if len(sys.argv) > 3 else True
par = MPCConfig(horizon=N).to_parameters(0.8)
if N == 50: par = dataclasses.replace(par, du_bounds=((-12., 12.), (-0.02, 0.02)))
x0, ref, up = make_batch(B, N, seed=3 if N == 50 else 2)
check = int(os.environ.get("CHECK", "50" if early else "25"))
ctl = MPCController(par, SolverSettings.early_certified(early_polish=early, check_termination=check), max_batch=B)
lib = L.load()
d = lambda a: torch.as_tensor(a).cuda()
dx0, dref, dup = d(x0), d(ref), d(up)
out = (C.c_ulonglong * 32)()
r = ctl.solve_batch(dx0, dref, u_prev=dup); torch.cuda.synchronize()
lib.cudampc_debug_tag_cycles(ctl._handle(1).ptr, out, 1)
r = ctl.solve_batch(dx0, dref, u_prev=dup); torch.cuda.synchronize()
lib.cudampc_debug_tag_cycles(ctl._handle(1).ptr, out, 1)
names = ["setup", "-", "update (odd: expand + A1, even: A1)", "residuals/check", "-", "factor (ADMM)", "rhs (odd: A2 + t, even: A2 + b')", "final/outputs",
         "save iterate", "polish: activity+assemble", "polish: factor", "polish: 4x(rhs, solve, dual, primal)", "polish: residuals+decision",
         "resume: load+assemble", "resume: factor", "early probe", "sweep forward + middle", "diagonal step", "sweep backward", "-",
         "  block: forward", "  block: diagonal", "  block: backward", "  block: B_a, expand (odd), B_b", "  block: update (A1 + own A2), B_c", "  block: rhs (+ t_o), B_d", "  block: fixup"] + ["-"] * 5
v = np.array(list(out), dtype=np.float64); it = r.iters.double().mean().item(); info = r.info.double().mean(0).cpu().numpy()
print(f"N={N} B={B} early={early} check={check}: mean iters {it:.1f}, factorisations {info[1]:.2f}, solves {info[3]:.1f}, total {v.sum()/B/1e3:.0f} k cycles per problem")
for n, c in sorted(zip(names, v), key=lambda t: -t[1]):
    print(f"  {n:40s} {c/B/1e3:9.1f} k cycles/problem  {100*c/v.sum():5.1f} %")
