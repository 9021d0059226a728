#!/usr/bin/env python
"""bench.py — IP-iterations/sec of the KKT path (BASELINE.json metric).

One "step" = the KKT work of one interior-point iteration, issued through the reference-facing
AbstractKKTSolver boundary exactly as `solve!` issues it (src/solver.jl:278-323):
    kktsolver_update!(cones)                    value scatter + static reg + numeric LDL'
    3 x (kktsolver_setrhs! ; kktsolver_solve!)  constant-RHS, affine and combined solves, each
                                                with iterative refinement
on cone states / right-hand sides recorded from a COMPLETE interior-point solve of the synthetic
instance on the GPU backend (the replayed set mixes the first, a middle and the last two iterates,
so the late, badly scaled systems are timed and checked too).

  value : steps/s over the SAME recorded inputs staged in HBM beforehand (cb200_set_resident: the
          boundary calls then take device pointers; results stay on the device)
  e2e   : steps/s through the C-ABI with HOST buffers (H2D of the cone state and the three
          right-hand sides and D2H of the three solutions inside the timed region)
  parity: after the timed region the last recorded system is solved once more; reported are the
          relative residual against the UNREGULARISED K (host SpMV, independent of the factor),
          IR rounds, dynamically regularised pivots and, when the CPU leg ran, the relative
          difference to the CPU QDLDL-path solution of the same three right-hand sides
  cpu_baseline : the CPU oracle (QDLDL-algorithm restatement, 1 thread like
          directldl_qdldl.jl:37) on the SAME full-size instance and the same recorded system:
          one full step, timed; no extrapolation.  It runs after the GPU line has been printed
          (and flushed) once, under a wall-clock limit; the completed line is printed last.
Timing: CUDA events on the library's own stream, max over ranks, W >= 3 warm-up steps.  The
factor/solve working set (panel storage) is far larger than the 126 MB L2 for every workload
except C1, so no explicit L2 flush is done ("inputs larger than L2").

--impl reference : the reference's CPU path on the SAME full-size instance (no sampling, no flop
ratio): the oracle runs the real interior-point iterations and the KKT sections of the first
iterations are timed.  When a single step costs more than the time budget allows (C5: ~2.5 min
per factorisation), the one step that is timed is the solver's own first factorisation
(solver_default_start!, identity scaling) + 3 solves; `steps` in the line says how many were timed.

--dump-outputs DIR : after the timed steps, writes what the last timed step computed, as its caller
reads it back: solve<k>_x.npy and solve<k>_z.npy (lhsx / lhsz of the step's k-th solve), float64,
at most 64 MB in all (a longer array is replaced by a fixed, seeded sample of its entries).
--replay-inputs PATH : the replayed systems are iterates of this build's own GPU solve, so they
depend on the build (a different summation order moves the trajectory, even the iteration count)
and, for C2, on the run (FP64 atomics in its root-front assembly).  With --replay-inputs the first
run stores its replayed systems (cone states and right-hand sides) in PATH and every later run with
the same PATH replays those instead: runs with the same arguments then solve the same systems, on any
build, and their dumps can be compared output for output.  C2's outputs can still differ in the last
bits from run to run (the same atomics, in the timed factorisations).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "IP-iterations/sec (KKT assemble+factor+solve)"

WORKLOADS = {
    # name: (generator, kwargs).  C1..C5 are the BASELINE.json configs at their stated sizes;
    # C4r / C4t are reduced SDPs kept for development runs.
    "C1": ("c1_random_qp", {}),
    "C2": ("c2_portfolio", {}),
    "C3": ("c3_socp", {}),
    "C4": ("c4_sdp", {}),
    "C4r": ("c4_sdp", {"ncones": 40, "side": 40, "n": 8000, "vars_per_cone": 300}),
    "C4t": ("c4_sdp", {"ncones": 12, "side": 20, "n": 1500, "vars_per_cone": 100}),     # compute-sanitizer size
    "C5": ("c5_block_angular", {}),
}
ORDERING_NAMES = {0: "amd", 1: "nested-dissection", 2: "natural", 3: "user", 4: "cone-block-dissection"}
CPU_LEG_LIMIT_S = float(os.environ.get("CB200_CPU_LEG_LIMIT", "330"))      # wall clock, b200 arm
REF_ARM_BUDGET_S = float(os.environ.get("CB200_REF_BUDGET", "200"))        # timed CPU work, reference arm


def make_problem(name):
    from clarabel_jl_b200 import problems
    gen, kw = WORKLOADS[name]
    return getattr(problems, gen)(**kw)


def workload_config(name, data, N, nnzK):
    """Identical in both arms: what the instance is, nothing about how an arm solves it."""
    gen, kw = WORKLOADS[name]
    # factor storage per step: C3 0.4 GB, C4 4.2 GB, C5 1.6 GB (>> the 126 MB L2); C1 2 MB, C2 58 MB
    l2 = ("working set fits in the 126 MB L2 and is NOT flushed between steps (latency-bound parity config)"
          if name in ("C1", "C2", "C4t") else "inputs larger than L2 (no flush)")
    return dict(workload=name, generator=gen, generator_kwargs=kw, n=int(data.n), m=int(data.m),
                N=int(N), nnzK=int(nnzK), l2=l2)


class Recorder:
    """Wraps a KKT solver and records the inputs of every boundary call of an IP run."""
    def __init__(self, ks):
        self.ks = ks
        self.steps = []          # list of dict(state=..., rhs=[(rx, rz), ...])
        self._u, self._s, self._r = ks.update, ks.solve, ks.setrhs
        ks.update, ks.solve, ks.setrhs = self.update, self.solve, self.setrhs
        self._rhs = None

    def update(self, cones):
        st = {k: np.array(v, copy=True) for k, v in cones.export_state().items()}
        self.steps.append(dict(state=st, rhs=[]))
        return self._u(cones)

    def setrhs(self, rx, rz):
        self._rhs = (np.array(rx, copy=True), np.array(rz, copy=True))
        return self._r(rx, rz)

    def solve(self, lx, lz):
        if self.steps:
            self.steps[-1]["rhs"].append(self._rhs)
        return self._s(lx, lz)

    def detach(self):
        self.ks.update, self.ks.solve, self.ks.setrhs = self._u, self._s, self._r


class FakeCones:
    def __init__(self, st):
        self.st = st

    def export_state(self):
        return self.st


def apply_state_to_oracle_cones(cones, st):
    """Overwrite the scaling state of a CompositeCone with a recorded one (CPU oracle replay)."""
    cones.w[:] = st["w"]; cones.soc_eta[:] = st["soc_eta"]; cones.soc_d[:] = st["soc_d"]
    cones.soc_u[:] = st["soc_u"]; cones.soc_v[:] = st["soc_v"]
    if len(st["psd_R"]):
        off = 0
        pos = {}
        for g in cones.psd_groups:
            for j, ci in enumerate(g["cones"]):
                pos[ci] = (g, j)
        for ci in [i for i, t in enumerate(cones.types) if t == 3]:
            g, j = pos[ci]; n = g["n"]
            g["R"][j] = st["psd_R"][off:off + n * n].reshape(n, n, order="F"); off += n * n
    return cones


def pick_replay(steps):
    """first / middle / last two complete IP iterations (each with its 3 right-hand sides)."""
    full = [(i, s) for i, s in enumerate(steps) if len(s["rhs"]) == 3]
    if not full:
        return [(len(steps) - 1, steps[-1])]
    k = len(full)
    idx = sorted(set([0, k // 2, max(0, k - 2), k - 1]))
    return [full[i] for i in idx]


def sample_clocks(stop, out):
    q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    while not stop.is_set():
        try:
            r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i",
                                os.environ.get("LOCAL_RANK", "0")], capture_output=True, text=True, timeout=5)
            f = [x.strip() for x in r.stdout.strip().split("\n")[0].split(",")]
            out.append(f)
        except Exception:
            pass
        stop.wait(0.2)


def clocks_summary(samples):
    if not samples:
        return dict(sm_mhz=None, sm_max_mhz=None, reasons=["unavailable"])
    sm = [float(s[1]) for s in samples if len(s) > 2]
    reasons = set()
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    for s in samples:
        for k, nm in enumerate(names):
            if len(s) > 5 + k and s[5 + k].lower().startswith("active"):
                reasons.add(nm)
    return dict(sm_mhz=float(np.median(sm)) if sm else None,
                sm_max_mhz=float(samples[0][2]) if len(samples[0]) > 2 else None,
                reasons=sorted(reasons))


def sym_matvec(K):
    """x -> K x for the symmetric matrix stored as upper-triangular scipy CSC."""
    import scipy.sparse as sp
    Ku = sp.triu(K, 1).tocsr()
    Kt = K.T.tocsr()
    return lambda x: Kt @ x + Ku @ x


# --------------------------------------------------------------------------------------------
# CPU oracle legs (the ONLY places bench.py executes oracle/)
# --------------------------------------------------------------------------------------------
def oracle_solver(problem):
    import clarabel_jl_b200 as cb
    from oracle.kktsolver_oracle import OracleDirectLDLKKTSolver
    cb.register_kktsolver("qdldl", OracleDirectLDLKKTSolver)
    P, q, A, b, K = problem
    t0 = time.perf_counter()
    s = cb.Solver(P, q, A, b, K, cb.Settings(direct_solve_method="qdldl"))
    return s, time.perf_counter() - t0


def cpu_full_step(problem, step, out):
    """One full-size step of the CPU QDLDL path on a recorded system; fills `out` (runs in a thread)."""
    try:
        s, t_setup = oracle_solver(problem)
        ks = s.kktsystem.kktsolver
        n, m = s.data.n, s.data.m
        apply_state_to_oracle_cones(s.cones, step["state"])
        sols = []
        t0 = time.perf_counter()
        ok = ks.update(s.cones)
        t_fac = time.perf_counter() - t0
        for rx, rz in step["rhs"]:
            lx, lz = np.zeros(n), np.zeros(m)
            ks.setrhs(rx, rz); ok &= bool(ks.solve(lx, lz))
            sols.append(np.concatenate([lx, lz]))
        dt = time.perf_counter() - t0
        out.update(ok=bool(ok), seconds=dt, factor_seconds=t_fac, setup_seconds=t_setup, sols=sols,
                   nnzL=int(ks.ldl.nnzL), factor_flops=float(ks.ldl.sum_lnz_sq))
    except Exception as e:                                   # reported, never fatal for the GPU line
        out.update(error=f"{type(e).__name__}: {e}")


class _BudgetExhausted(Exception):
    pass


def reference_arm(name, steps, warmup):
    """The reference's CPU path on the full-size instance: real IP iterations, KKT sections timed."""
    problem = make_problem(name)
    s, t_setup = oracle_solver(problem)
    ks = s.kktsystem.kktsolver
    n, m = s.data.n, s.data.m
    u0, s0, r0 = ks.update, ks.solve, ks.setrhs
    acc = dict(t=0.0, updates=0, per_iter=[], cur=0.0, last_rhs=None, nsolve=0)
    want_warm = min(max(0, warmup), 1)

    def upd(cones):
        # an update opens a new step; the previous one (if any) is complete
        if acc["updates"] > 0:
            acc["per_iter"].append((acc["cur"], acc["nsolve"]))
        timed_done = len(acc["per_iter"]) - 1 - want_warm       # entry 0 is solver_default_start!
        spent = sum(t for t, _ in acc["per_iter"][1 + want_warm:])
        nxt = acc["per_iter"][-1][0] if acc["per_iter"] else 0.0
        if acc["per_iter"] and (timed_done >= steps or spent + nxt > REF_ARM_BUDGET_S
                                or (timed_done < 0 and acc["per_iter"][0][0] > REF_ARM_BUDGET_S / 3)):
            raise _BudgetExhausted()
        acc["updates"] += 1; acc["cur"] = 0.0; acc["nsolve"] = 0
        t = time.perf_counter(); r = u0(cones); acc["cur"] += time.perf_counter() - t
        return r

    def setrhs(rx, rz):
        acc["last_rhs"] = (np.array(rx, copy=True), np.array(rz, copy=True))
        t = time.perf_counter(); r = r0(rx, rz); acc["cur"] += time.perf_counter() - t
        return r

    def sol(lx, lz):
        t = time.perf_counter(); r = s0(lx, lz); acc["cur"] += time.perf_counter() - t
        acc["nsolve"] += 1
        return r
    ks.update, ks.solve, ks.setrhs = upd, sol, setrhs
    status = None
    try:
        res = s.solve(max_iter=want_warm + steps + 1)
        status = res.status_name
        if acc["updates"] > len(acc["per_iter"]):
            acc["per_iter"].append((acc["cur"], acc["nsolve"]))
    except _BudgetExhausted:
        pass
    ks.update, ks.solve, ks.setrhs = u0, s0, r0
    per = acc["per_iter"]
    timed = per[1 + want_warm:1 + want_warm + steps]
    timed = [t for t in timed if t[1] >= 3]
    if timed:
        what = (f"IP iterations {1 + want_warm}..{want_warm + len(timed)} of the full-size solve "
                f"(update + 3 solves each), after solver_default_start! and {want_warm} untimed iteration(s)")
        tt = [t for t, _ in timed]
    else:
        # a single step is all the budget allows: solver_default_start!'s factorisation (identity
        # scaling) + its solves, completed to 3 solves with the same right-hand side
        t_extra = 0.0
        nso = per[0][1]
        lx, lz = np.zeros(n), np.zeros(m)
        while nso < 3:
            t = time.perf_counter(); r0(*acc["last_rhs"]); s0(lx, lz); t_extra += time.perf_counter() - t
            nso += 1
        tt = [per[0][0] + t_extra]
        what = ("1 step = solver_default_start!'s factorisation (identity scaling) + 3 solves; one such "
                f"step takes {tt[0]:.0f} s on this instance, more would exceed the time budget")
    dt = float(np.sum(tt))
    v = len(tt) / dt
    N = s.kktsystem.kktsolver.KKT.shape[0]
    line = dict(metric=METRIC, value=v, unit="it/s", n_gpus=1, steps=len(tt), warmup=want_warm if timed else 0,
                ms_per_step=1e3 / v, higher_is_better=True, scaling="strong", vs_baseline=None,
                dtype="f64", data="synthetic", impl="reference",
                config=workload_config(name, s.data, N, ks.KKT.nnz),
                cpu_baseline=dict(value=v, unit="it/s", cores=1, kind="port",
                                  sample="FULL-SIZE instance, " + what,
                                  engine="oracle/qdldl_oracle.c (QDLDL algorithm, 1 thread like "
                                         "directldl_qdldl.jl:37), AMD-class ordering with the reference's "
                                         "amd_dense_scale = 1.5",
                                  nnzL=int(ks.ldl.nnzL), factor_flops=float(ks.ldl.sum_lnz_sq),
                                  setup_seconds=t_setup, step_seconds=tt, status_after=status),
                e2e=dict(value=v, unit="it/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    return line


DUMP_BUDGET_BYTES = 64_000_000


def fit_dump_budget(outs, budget=DUMP_BUDGET_BYTES):
    """float64 copies of `outs` that together stay within `budget` bytes: an array longer than its
    equal share is replaced by a fixed sample of its entries (seed 0, ascending indices), so the
    same array sizes always give the same sample."""
    cap = (budget - 4096 * len(outs)) // (8 * len(outs))      # 4 KB per file for the .npy header
    fitted = {}
    for name, a in outs.items():
        a = np.asarray(a, dtype=np.float64)
        if a.size > cap:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, cap, replace=False))]
        fitted[name] = a
    return fitted


def dump_outputs(out_dir, ks, rhs_t, write):
    """The solutions of the last timed step (device-resident leg).  The step leaves only its last
    solution on the device; the earlier ones are solved again from the same factorisation and
    right-hand sides (a solve reads the factorisation, it does not change it).  Every rank takes part
    in the solves; only `write` ranks write."""
    N, n, m = ks.KKT.shape[0], ks.n, ks.m
    sols = [None] * len(rhs_t)
    sols[-1] = ks.ldl.download(6, N)
    for k, (tx, tz) in enumerate(rhs_t[:-1]):
        ks.setrhs_staged(tx.data_ptr() if tx.numel() else 0, tz.data_ptr() if tz.numel() else 0)
        ks.solve(None, None)
        sols[k] = ks.ldl.download(6, N)
    if not write:
        return
    outs = {}
    for k, x in enumerate(sols, 1):
        outs[f"solve{k}_x"], outs[f"solve{k}_z"] = x[:n], x[n:n + m]
    os.makedirs(out_dir, exist_ok=True)
    for name, a in fit_dump_budget(outs).items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def save_replay(path, name, n, m, replay_ids, replay):
    arrs = dict(workload=np.array(name), n_m=np.array([n, m]), replay_ids=np.array(replay_ids))
    for i, s_ in enumerate(replay):
        for k, v in s_["state"].items():
            arrs[f"s{i}_state_{k}"] = v
        for j, (rx, rz) in enumerate(s_["rhs"]):
            arrs[f"s{i}_rx{j}"], arrs[f"s{i}_rz{j}"] = rx, rz
    with open(path, "wb") as f:
        np.savez(f, **arrs)


def load_replay(path, name, n, m):
    """(replay_ids, replay) as save_replay stored them; the file must hold systems of this instance."""
    with np.load(path) as z:
        if str(z["workload"]) != name or z["n_m"].tolist() != [n, m]:
            raise SystemExit(f"{path} holds systems of {z['workload']} (n, m = {z['n_m'].tolist()}), "
                             f"not of {name} (n, m = {[n, m]})")
        ids = z["replay_ids"].tolist()
        replay = []
        for i in range(len(ids)):
            pre = f"s{i}_state_"
            st = {f[len(pre):]: z[f] for f in z.files if f.startswith(pre)}
            nrhs = sum(f.startswith(f"s{i}_rx") for f in z.files)
            replay.append(dict(state=st, rhs=[(z[f"s{i}_rx{j}"], z[f"s{i}_rz{j}"]) for j in range(nrhs)]))
    return ids, replay


def _watchdog(seconds):
    """A hung collective must not hang the caller: dump stacks and exit non-zero."""
    import faulthandler
    faulthandler.dump_traceback_later(seconds, exit=True)


def load_traffic(name):
    """ncu dram__bytes of the kernel classes (per call), committed under profiles/ (see
    profiles/r02_summary.md for the command); None when no capture exists for the workload."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json"))).get(name)
    except Exception:
        return None


def main():
    _watchdog(int(os.environ.get("CB200_BENCH_TIMEOUT", "1500")))
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=os.environ.get("CB200_WORKLOAD", "C5"))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the solutions of the last timed step to DIR/<name>.npy")
    ap.add_argument("--replay-inputs", metavar="PATH",
                    help="replay the systems stored in PATH; if PATH does not exist, store this run's there")
    args = ap.parse_args()
    if (args.dump_outputs or args.replay_inputs) and args.impl == "reference":
        ap.error("--dump-outputs and --replay-inputs apply to --impl b200")
    # decided before any rank can have written PATH
    load_inputs = bool(args.replay_inputs) and os.path.exists(args.replay_inputs)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    name = args.workload

    if args.impl == "reference":
        if rank != 0:
            return
        print(json.dumps(reference_arm(name, max(1, args.steps), max(0, args.warmup))), flush=True)
        return

    args.warmup = max(args.warmup, 3)
    import torch
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    import clarabel_jl_b200 as cb
    problem = make_problem(name)
    P, q, A, b, K = problem
    t0 = time.perf_counter()
    solver = cb.Solver(P, q, A, b, K, cb.Settings(direct_solve_method="b200"))
    t_setup = time.perf_counter() - t0
    ks = solver.kktsystem.kktsolver
    # ---- a complete IP solve on the GPU backend, every boundary call recorded
    rec = Recorder(ks)
    t0 = time.perf_counter()
    sol = solver.solve()
    t_ipsolve = time.perf_counter() - t0
    rec.detach()
    picked = pick_replay(rec.steps)
    replay_ids = [i for i, _ in picked]
    replay = [s_ for _, s_ in picked]
    n_recorded = len(rec.steps)
    rec.steps = None
    n, m = solver.data.n, solver.data.m
    N = ks.KKT.shape[0]
    if load_inputs:
        replay_ids, replay = load_replay(args.replay_inputs, name, n, m)
    elif args.replay_inputs and rank == 0:
        save_replay(args.replay_inputs, name, n, m, replay_ids, replay)

    def pinned(a):
        """copy of `a` in page-locked host memory (the e2e copies are then true DMA transfers)"""
        t = torch.empty(a.shape, dtype=torch.float64, pin_memory=True)
        v = t.numpy(); v[...] = a
        pinned.keep.append(t)
        return v
    pinned.keep = []
    for s_ in replay:
        s_["state"] = {k: pinned(v) for k, v in s_["state"].items()}
        s_["rhs"] = [(pinned(rx), pinned(rz)) for rx, rz in s_["rhs"]]
    lx, lz = pinned(np.zeros(n)), pinned(np.zeros(m))
    stream = torch.cuda.ExternalStream(ks.ldl.stream_ptr(), device=torch.device("cuda", local))

    # the same inputs once more, staged in HBM for the device-resident timing (cb200_set_resident:
    # pointer arguments are then device pointers, copied device-to-device on the solver's stream)
    dev = torch.device("cuda", local)
    staged = []
    for s_ in replay:
        st_t = {k: torch.from_numpy(np.ascontiguousarray(s_["state"][k], dtype=np.float64)).to(dev)
                for k in ks.STATE_KEYS}
        rhs_t = [(torch.from_numpy(rx).to(dev), torch.from_numpy(rz).to(dev)) for rx, rz in s_["rhs"]]
        staged.append((st_t, rhs_t))
    torch.cuda.synchronize()

    def step(i):
        k = i % len(replay)
        s_ = replay[k]
        if ks.ldl.resident:
            st_t, rhs_t = staged[k]
            ok = ks.update_staged([st_t[key].data_ptr() if st_t[key].numel() else 0 for key in ks.STATE_KEYS])
            for tx, tz in rhs_t:
                ks.setrhs_staged(tx.data_ptr() if tx.numel() else 0, tz.data_ptr() if tz.numel() else 0)
                ok &= ks.solve(None, None)
            return ok
        ok = ks.update(FakeCones(s_["state"]))
        for rx, rz in s_["rhs"]:
            ks.setrhs(rx, rz); ok &= ks.solve(lx, lz)
        return ok

    def timed(nsteps, offset):
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(nsteps):
            step(offset + i)
        e1.record(stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            import torch.distributed as dist
            t = torch.tensor([ms], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    state_bytes = sum(v.nbytes for v in replay[0]["state"].values())
    nrhs = len(replay[0]["rhs"])
    h2d = state_bytes + nrhs * (n + m) * 8
    d2h = nrhs * (n + m) * 8
    # ---- e2e (host buffers through the C-ABI)
    for i in range(args.warmup):
        step(i)
    stop = threading.Event(); samples = []
    th = threading.Thread(target=sample_clocks, args=(stop, samples), daemon=True)
    th.start()
    ks.ldl.reset_timers()
    ms_e2e = timed(args.steps, args.warmup)
    # ---- device-resident
    ks.ldl.set_resident(True)
    for i in range(args.warmup):
        step(i)
    ks.ldl.reset_timers(); ks.ir_rounds = 0; ks.n_solves = 0
    ms_res = timed(args.steps, args.warmup)
    tm = ks.ldl.timers()
    ir_per_solve = ks.ir_rounds / max(1, ks.n_solves)
    stop.set(); th.join(timeout=2)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, ks, staged[(args.warmup + args.steps - 1) % len(replay)][1], rank == 0)
    ks.ldl.set_resident(False)
    # ---- per-kernel-class timing of the factorisation (events around each launch group; graph
    # replay is off for these extra steps, they are not part of the timed regions above).  In
    # multi-GPU mode EVERY rank must execute them (they contain collectives).
    ks.ldl.set_detail(True); ks.ldl.set_resident(True)
    step(0)
    ks.ldl.reset_timers()
    nd_steps = len(replay)
    for i in range(nd_steps):
        step(i)
    td = ks.ldl.timers()
    ks.ldl.set_detail(False); ks.ldl.set_resident(False)
    # ---- parity solves (every rank takes part; rank 0 evaluates): the LAST recorded system
    last = replay[-1]
    ks.ir_rounds = 0; ks.n_solves = 0
    ok_par = ks.update(FakeCones(last["state"]))
    nzv = ks.device_nzval()                     # unregularised K values as the device holds them
    gsol, gfull = [], []
    for rx, rz in last["rhs"]:
        gx, gz = np.zeros(n), np.zeros(m)
        ks.setrhs(rx, rz); ok_par &= ks.solve(gx, gz)
        gsol.append(np.concatenate([gx, gz]))
        gfull.append(ks.ldl.download(6, N))     # [x; z; expansion variables] as the device holds it
    par_ir = ks.ir_rounds / max(1, ks.n_solves)
    # the device-resident leg must compute the same thing: the same system once more from the staged
    # (HBM) copies of its inputs, solutions compared with the host-buffer path above
    res_diff = None
    try:
        ks.ldl.set_resident(True)
        st_t, rhs_t = staged[-1]
        okr = ks.update_staged([st_t[key].data_ptr() if st_t[key].numel() else 0 for key in ks.STATE_KEYS])
        res_diff = 0.0
        for (tx, tz), xh in zip(rhs_t, gfull):
            ks.setrhs_staged(tx.data_ptr() if tx.numel() else 0, tz.data_ptr() if tz.numel() else 0)
            okr &= ks.solve(None, None)
            xr = ks.ldl.download(6, N)
            res_diff = max(res_diff, float(np.abs(xr - xh).max() / max(1e-300, np.abs(xh).max())))
        if not okr:
            res_diff = float("inf")
    except Exception as e:        # never lose the line over the cross-check
        res_diff = f"failed: {e}"
    finally:
        ks.ldl.set_resident(False)
    nreg = int(ks.ldl.download(5, 1)[0])
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    import scipy.sparse as sp
    Kd = sp.csc_matrix((nzv, ks.KKT.indices, ks.KKT.indptr), shape=ks.KKT.shape)
    mv = sym_matvec(Kd)
    resid = []
    for (rx, rz), xf in zip(last["rhs"], gfull):
        bb = np.concatenate([rx, rz, np.zeros(N - n - m)])
        r = bb - mv(xf)
        resid.append(float(np.abs(r).max() / max(1e-300, np.abs(bb).max())))
    parity = dict(system=f"IP iteration {replay_ids[-1]} of {n_recorded - 1} (the last one recorded)",
                  ok=bool(ok_par), rel_residual_unregularised_K=resid, ir_rounds_per_solve=par_ir,
                  regularised_pivots=nreg, gpu_solve=dict(status=sol.status_name, iterations=int(sol.iterations),
                                                          obj_val=float(sol.obj_val), obj_val_dual=float(sol.obj_val_dual),
                                                          r_prim=float(sol.r_prim), r_dual=float(sol.r_dual)),
                  resident_vs_host_rel_diff=res_diff, cpu_rel_diff=None)
    info = ks.ldl.info()
    stats = ks.ldl.stats()
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
    nfac, nsol = max(1, tm["nfactor"]), max(1, tm["nsolve"])
    nnzL, nnzK = int(info.nnzL), int(ks.KKT.nnz)
    # ---- FP64 compute calibration on this box (no FP64 figure in MEASURED_PEAKS.json): cuBLAS DGEMM
    fp64_peak = None
    try:
        a_ = torch.randn(4096, 4096, dtype=torch.float64, device="cuda")
        b_ = torch.randn(4096, 4096, dtype=torch.float64, device="cuda")
        for _ in range(2):
            torch.matmul(a_, b_)
        torch.cuda.synchronize()
        best = 1e9
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); torch.matmul(a_, b_); e1.record(); torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        fp64_peak = 2 * 4096 ** 3 / (best * 1e-3) / 1e12
        del a_, b_
    except Exception:
        pass
    nfd = max(1, td["nfactor"])
    b_solve = 16.0 * nnzL + 48.0 * N                 # SURVEY.md section 8(d)
    b_spmv = 8.0 * nnzK + 24.0 * N
    t_solve = tm["solve_ms"] / nsol * 1e-3
    t_fac = tm["factor_ms"] / nfac * 1e-3
    t_spmv = tm["spmv_ms"] / nsol * 1e-3
    t_schur = td["schur_ms"] / nfd * 1e-3
    rank_flops = stats.get("rank_flops", stats["flops"]) if world > 1 else stats["flops"]
    traffic = load_traffic(name) or {}
    kernels = dict(
        triangular_solve_sweeps=dict(bound="hbm", ms_per_call=t_solve * 1e3, calls_per_step=nsol / args.steps,
                                     achieved=b_solve / t_solve / 1e9, unit="GB/s", peak=hbm_peak,
                                     algorithmic_bytes=b_solve, traffic=traffic.get("triangular_solve_sweeps")),
        spmv_residual=dict(bound="hbm", ms_per_call=t_spmv * 1e3, calls_per_step=nsol / args.steps,
                           achieved=b_spmv / max(t_spmv, 1e-12) / 1e9, unit="GB/s", peak=hbm_peak,
                           algorithmic_bytes=b_spmv, traffic=traffic.get("spmv_residual")),
        factor_total=dict(bound="fp64", ms_per_call=t_fac * 1e3, calls_per_step=nfac / args.steps,
                          achieved=rank_flops / t_fac / 1e12, unit="TFLOP/s", peak=fp64_peak,
                          algorithmic_flops=rank_flops),
        schur_gemm=dict(bound="fp64", ms_per_call=t_schur * 1e3, calls_per_step=1.0,
                        achieved=(stats["schur_flops"] / t_schur / 1e12) if t_schur > 0 else None,
                        unit="TFLOP/s", peak=fp64_peak, algorithmic_flops=stats["schur_flops"],
                        traffic=traffic.get("schur_gemm")),
        factor_pivot_blocks=dict(ms_per_call=td["panel_ms"] / nfd), factor_small_fronts=dict(ms_per_call=td["small_ms"] / nfd),
        factor_assembly=dict(ms_per_call=td["asm_ms"] / nfd))
    for k in kernels.values():
        if k.get("peak") and k.get("achieved") is not None:
            k["frac"] = k["achieved"] / k["peak"]
    if world > 1:
        for k in ("schur_gemm", "factor_total"):
            kernels[k]["note"] = "flops of the fronts THIS rank factors (own subtrees + replicated top) / this rank's time"
        # the sweeps stream the WHOLE factor once per job (each rank its subtrees + the replicated top), so the
        # whole-job bytes are held against the aggregate bandwidth of the N GPUs
        for k in ("triangular_solve_sweeps", "spmv_residual"):
            kernels[k]["peak"] = hbm_peak * world
            kernels[k]["frac"] = kernels[k]["achieved"] / kernels[k]["peak"]
            kernels[k]["note"] = f"whole-job algorithmic bytes / max-over-ranks time, peak = {world} x the single-GPU figure"
    # dominant kernel class of the step: the largest (time per call x calls per step) among the measured ones
    cand = {"triangular_solve_sweeps": t_solve * nsol / args.steps, "schur_gemm": t_schur,
            "spmv_residual": t_spmv * nsol / args.steps}
    dom = max(cand, key=cand.get)
    kd = kernels[dom]
    roofline = dict(bound=kd["bound"] if kd["bound"] == "hbm" else "tensor", kernel=dom, achieved=kd["achieved"],
                    peak=kd["peak"], unit=kd["unit"], frac=kd.get("frac"), traffic=kd.get("traffic"),
                    peak_source=(peak_src if kd["bound"] == "hbm" else
                                 "on-box cuBLAS DGEMM 4096^3 (float64) - MEASURED_PEAKS.json has no FP64 figure"),
                    note="FP64 throughout: bound 'tensor' means the FP64 tensor-core path (DMMA; tcgen05 has no f64 "
                         "kind, DESIGN.md section 4) measured against an on-box DGEMM",
                    kernels=kernels)
    config = workload_config(name, solver.data, N, nnzK)
    line = dict(metric=METRIC, value=args.steps / (ms_res * 1e-3), unit="it/s", n_gpus=args.gpus,
                steps=args.steps, warmup=args.warmup, ms_per_step=ms_res / args.steps,
                higher_is_better=True, scaling="strong", vs_baseline=None, dtype="f64",
                data="synthetic", impl="b200", config=config,
                details=dict(nnzL=nnzL, factor_flops=stats["flops"], nsuper=int(stats["nsuper"]),
                             nlevels=int(stats["nlevels"]),
                             ordering=ORDERING_NAMES.get(int(stats.get("ordering_used", -1)), "?"),
                             setup_s=t_setup, ip_solve_s=t_ipsolve, recorded_ip_iterations=n_recorded - 1,
                             replayed_ip_iterations=replay_ids,
                             solves_per_step=nsol / args.steps, ir_rounds_per_solve=ir_per_solve),
                e2e=dict(value=args.steps / (ms_e2e * 1e-3), unit="it/s", ms_per_step=ms_e2e / args.steps,
                         h2d_bytes_per_step=int(h2d), d2h_bytes_per_step=int(d2h)),
                gpu_launches=int(tm["nlaunch"]), clocks=clocks_summary(samples), roofline=roofline,
                parity=parity,
                cpu_baseline=dict(value=None, unit="it/s", cores=1, kind="port",
                                  sample="pending: the full-size CPU step runs after this line"))
    if world > 1 or args.no_cpu_baseline:
        line["cpu_baseline"]["sample"] = "not run (the CPU arm is timed at N = 1 only)" if world > 1 else "not run (--no-cpu-baseline)"
        print(json.dumps(line), flush=True)
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()
        return
    # the GPU measurement is on record before the (long) CPU leg starts
    print(json.dumps(line), flush=True)
    out = {}
    thc = threading.Thread(target=cpu_full_step, args=(problem, last, out), daemon=True)
    t0 = time.perf_counter()
    thc.start(); thc.join(CPU_LEG_LIMIT_S)
    what = (f"FULL-SIZE instance, one step (update + 3 solves with refinement) on the system of IP iteration "
            f"{replay_ids[-1]}; oracle/qdldl_oracle.c, 1 thread, AMD-class ordering with amd_dense_scale = 1.5")
    if thc.is_alive() or "seconds" not in out:
        why = out.get("error") or f"not finished within the {CPU_LEG_LIMIT_S:.0f} s wall-clock limit of the CPU leg"
        line["cpu_baseline"] = dict(value=None, unit="it/s", cores=1, kind="port", sample=what + " -- " + why)
    else:
        line["cpu_baseline"] = dict(value=1.0 / out["seconds"], unit="it/s", cores=1, kind="port", sample=what,
                                    step_seconds=out["seconds"], factor_seconds=out["factor_seconds"],
                                    setup_seconds=out["setup_seconds"], nnzL=out["nnzL"],
                                    factor_flops=out["factor_flops"])
        diffs = [float(np.abs(g - c).max() / max(1e-300, np.abs(c).max())) for g, c in zip(gsol, out["sols"])]
        line["parity"]["cpu_rel_diff"] = diffs
        line["parity"]["cpu_ok"] = out["ok"]
    print(json.dumps(line), flush=True)
    if thc.is_alive():
        os._exit(0)          # the C factorisation cannot be interrupted; everything is already printed


if __name__ == "__main__":
    main()
