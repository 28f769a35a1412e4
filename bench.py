#!/usr/bin/env python
"""bench.py -- moment-match rollout steps/s of the B200-native PILCO engine (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--config metric|inverted_pendulum|inv_double_pendulum|smgpr|swimmer|test_cascade]
                    [--restarts R] [--through-api] [--dump-outputs DIR]

One bench "step" = one pass of the hot path over one batch: an H-step moment-matching rollout
(policy moment match -> squash -> joint -> dynamics moment match -> glue -> reward, pilco.py:118-153)
for R independent policy restarts per GPU.  value = R*H*N_gpus rollout steps / second.

Default workload = the metric config of BASELINE.json (SURVEY.md section 8d): N=300 training points, E=Ds=10, U=2, D=12,
H=40, RBF policy with 50 basis functions, fp64, synthetic seeded data, R=32 restarts per GPU (weak scaling).
`--config` selects one of BASELINE.json's `configs` shapes instead (same JSON line, its own roofline / CPU leg).
`--through-api` (any config) drives `PILCO.optimize_policy(restarts=R*N)` itself -- lock-step L-BFGS-B,
taped forward + reverse sweep per evaluation, one all_gather of [loss | params] -- and reports wall-clock
loss-evaluations x R x H / s.
`--dump-outputs DIR` writes, after the timed steps, what the last timed step of each arm returned (trajectories, rewards,
policy gradients; rank 0's restarts) as DIR/<name>.npy: the inputs are seeded, so two builds can be compared output
for output.

Rank 0 prints ONE JSON line.  `--impl reference` times the reference-equivalent CPU path
(oracle/torch_port.py, all host threads it can use) on bounded samples of the same workload.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# rank 0 must print exactly ONE line on stdout: keep NCCL's "NCCL version ..." banner (NCCL_DEBUG=VERSION) off it
if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
    os.environ["NCCL_DEBUG"] = "WARN"

# BASELINE.json `configs` as code-derived shapes (SURVEY.md section 8d): E = Ds, D = Ds + U.  R = restarts per GPU.
CONFIGS = {
    "metric": dict(N=300, Ds=10, U=2, bf=50, H=40, R=32, S0=0.1,
                   name="metric config: N=300 E=Ds=10 U=2 D=12 H=40, RBF policy bf=50"),
    "test_cascade": dict(N=100, Ds=2, U=1, bf=0, H=30, R=1, S0=0.1,
                         name="test_cascade.py: N=100 D=3 E=2 H=30, linear policy, single restart"),
    "inverted_pendulum": dict(N=300, Ds=4, U=1, bf=10, H=40, R=1, S0=0.1,
                              name="inverted_pendulum.py: N=300 E=4 D=5 H=40, RBF bf=10, single restart"),
    "inv_double_pendulum": dict(N=400, Ds=6, U=1, bf=40, H=40, R=32, S0=0.1,
                                name="inv_double_pendulum.py: N=400 E=6 D=7 H=40, RBF bf=40, 32 restarts batched"),
    "smgpr": dict(N=2000, M=200, Ds=10, U=2, bf=50, H=40, R=32, S0=0.1,
                  name="SMGPR sparse path: N=2000 M=200 E=10 D=12 H=40, RBF bf=50"),
    "swimmer": dict(N=500, Ds=8, U=2, bf=40, H=50, R=32, S0=0.005,
                    name="swimmer.py: N=500 E=8 D=10 H=50, RBF bf=40, 256 restarts over 8 GPUs (32 per GPU)"),
}
UNIT = "rollout-steps/s"
EXP_FLOP_EQ = 14.0          # fp64 flop-equivalents of one exp: exp_shifted()'s 7 fp64-pipe instructions (3 DADD, 3 DFMA, DMUL), 2 each


def metric_name(cfg):
    if cfg is CONFIGS["metric"]:
        return "moment-match rollout steps/sec (N=300, E=10, H=40, fp64)"
    n = ("M=%d of N=%d" % (cfg["M"], cfg["N"])) if "M" in cfg else "N=%d" % cfg["N"]
    return "moment-match rollout steps/sec (%s, E=%d, H=%d, fp64)" % (n, cfg["Ds"], cfg["H"])


def make_workload(cfg, seed=0):
    """Seeded synthetic problem (SURVEY.md section 8d recipe; deviations documented in BASELINE.md section 6: state differences
    and signal variances scaled by 0.05, noise 1e-3, so that a 40-50 step rollout with UNTRAINED hyper-parameters stays
    finite).  Restart r uses RandomState(seed+1+r), so any sharding over ranks sees the same per-restart policies."""
    N, Ds, U = cfg["N"], cfg["Ds"], cfg["U"]
    D = Ds + U
    rng = np.random.RandomState(seed)
    X = rng.rand(N, D)
    A = rng.rand(D, Ds)
    Y = 0.05 * (np.sin(X).dot(A) + 1e-3 * (rng.rand(N, Ds) - 0.5))     # state differences
    ell = 1.0 + rng.rand(Ds, D)
    sf2 = 0.05 * (1.0 + rng.rand(Ds))
    sn2 = 1e-3 * np.ones(Ds)
    wl = dict(X=X, Y=Y, ell=ell, sf2=sf2, sn2=sn2, m0=X[0, :Ds].copy(), S0=cfg["S0"] * np.eye(Ds), W=np.eye(Ds), t=np.zeros(Ds))
    if "M" in cfg:
        wl["Z"] = np.random.RandomState(seed + 7).rand(cfg["M"], D)        # smgpr.py:20
    return wl


def make_policies(cfg, restart_ids, seed=0):
    Ds, U, bf = cfg["Ds"], cfg["U"], cfg["bf"]
    if bf == 0:                                                             # linear policy (test_cascade.py)
        Ws, bs = [], []
        for r in restart_ids:
            rng = np.random.RandomState(seed + 1 + int(r))
            Ws.append(rng.rand(U, Ds)); bs.append(rng.rand(U))
        return dict(W=np.stack(Ws), b=np.stack(bs))
    Xc, Yc, lc = [], [], []
    for r in restart_ids:
        rng = np.random.RandomState(seed + 1 + int(r))
        Xc.append(rng.randn(bf, Ds) * 0.5 + 0.5)
        Yc.append(0.1 * rng.randn(bf, U))
        lc.append(1.0 + 0.1 * rng.randn(U, Ds))
    return dict(Xc=np.stack(Xc), Yc=np.stack(Yc), lc=np.stack(lc))


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, restart_ids, arrays):
    """``--dump-outputs``: each array (leading dimension = restart) as ``<out_dir>/<name>.npy`` in float64, and the
    global ids of the dumped restarts as ``restarts.npy``.  Above 64 MB in all, a fixed seeded sample of the
    restarts is written instead, the same rows for every array."""
    rows = np.arange(len(restart_ids))
    row_bytes = 8 * sum(a[0].size for a in arrays.values())
    if row_bytes * len(rows) > DUMP_LIMIT_BYTES:
        keep = max(1, DUMP_LIMIT_BYTES // row_bytes)
        rows = np.sort(np.random.RandomState(0).choice(len(rows), keep, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "restarts.npy"), np.asarray(restart_ids, dtype=np.float64)[rows])
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64)[rows])


def step_counts(cfg):
    """SURVEY.md section 8d / BASELINE.md section 5: algorithmic flops, exps and compulsory bytes of ONE rollout step
    (dynamics call over n centres + policy call over bf centres)."""
    def mm(n, D, E, trace):
        P = E * (E + 1) // 2
        F = P * (2 * n * n * D + 2 * n * D * D) + 4 * P * n * n + (2 * E * n * n if trace else 0) + E * (2 * n * D * D + 6 * n * D)
        Xe = P * n * n + E * n
        B = 8 * (n * D + E * n + (E * n * n if trace else 0) + 2 * E * D + D * D + D + E + E * E + D * E)
        return F, Xe, B
    n = cfg.get("M", cfg["N"])
    Ds, U, bf = cfg["Ds"], cfg["U"], cfg["bf"]
    F, Xe, B = mm(n, Ds + U, Ds, True)
    if bf:
        F2, X2, B2 = mm(bf, Ds, U, False)
        F, Xe, B = F + F2, Xe + X2, B + B2
    return F, Xe, B


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: oracle torch port on the host cores
# ------------------------------------------------------------------------------------------------
_THREADS = None


def pick_cpu_threads():
    """All the host threads the CPU path can USE: torch's intra-op pool stops scaling (and on a shared
    128-core box collapses) beyond a few tens of threads on these [E,E,N,N] elementwise ops, so calibrate
    once on a small probe and keep the fastest of {8,16,32,64,all} <= os.cpu_count()."""
    global _THREADS
    if _THREADS is not None:
        return _THREADS
    import torch
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 64, ncpu) if c <= ncpu} or {ncpu})
    x = torch.rand(10, 10, 200, 200, dtype=torch.float64)
    best, best_t = cands[0], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        torch.exp(x)                                  # warm the pool
        t0 = time.perf_counter()
        for _ in range(3):
            y = torch.exp(x + 1.0) @ x[0, 0]          # noqa: F841
        dt = time.perf_counter() - t0
        if dt < best_t * 0.9:                         # prefer fewer threads unless clearly faster
            best, best_t = c, dt
    _THREADS = best
    return best


class CpuRollout:
    """The reference-equivalent CPU path (oracle/torch_port.py) for restart 0 of a config: one rollout of
    ``h`` steps, factorisations recomputed inside every step as the reference does (mgpr.py:77-79, smgpr.py,
    controllers.py:115); ``grad=True`` also runs torch autograd back to the policy parameters (what
    gpflow.optimizers.Scipy differentiates, pilco.py:84-90)."""

    def __init__(self, cfg, wl, threads=None):
        import torch
        from oracle import torch_port as tp
        self.torch, self.tp, self.cfg, self.wl = torch, tp, cfg, wl
        self.threads = threads or pick_cpu_threads()
        torch.set_num_threads(self.threads)
        T = lambda a: torch.as_tensor(np.asarray(a), dtype=torch.float64)
        self.T = T
        self.X, self.Y, self.ell, self.sf2, self.sn2 = map(T, (wl["X"], wl["Y"], wl["ell"], wl["sf2"], wl["sn2"]))
        self.Z = T(wl["Z"]) if "Z" in wl else None
        pol = make_policies(cfg, [0])
        self.pol = {k: T(v[0]) for k, v in pol.items()}
        self.maxa = torch.ones((1, cfg["U"]), dtype=torch.float64)
        self.W, self.t = T(wl["W"]), T(wl["t"])[None]

    def run(self, h, grad=False):
        torch, tp = self.torch, self.tp
        ps = {k: v.clone().requires_grad_(grad) for k, v in self.pol.items()}

        def dyn(m, s):
            if self.Z is not None:
                iK, beta = tp.fitc_factorizations(self.X, self.Z, self.Y, self.ell, self.sf2, self.sn2)
                return tp.predict_given_factorizations(self.Z, self.ell, self.sf2, m, s, iK, beta)
            iK, beta = tp.calculate_factorizations(self.X, self.Y, self.ell, self.sf2, self.sn2)
            return tp.predict_given_factorizations(self.X, self.ell, self.sf2, m, s, iK, beta)
        if "W" in ps:
            act = lambda m, s: tp.linear_action(ps["W"], ps["b"][None], m, s, self.maxa)
        else:
            act = lambda m, s: tp.rbf_action(ps["Xc"], ps["Yc"], ps["lc"], m, s, self.maxa)
        rew = lambda m, s: tp.exponential_reward(m, s, self.W, self.t)
        ctx = torch.enable_grad() if grad else torch.no_grad()
        with ctx:
            _, _, total = tp.predict(self.T(self.wl["m0"])[None], self.T(self.wl["S0"]), h, act, dyn, rew)
            if grad:
                total[0, 0].backward()
        return float(total.detach())

    def steps_per_s(self, reps=2, h=4, grad=False, budget_s=30.0):
        self.run(2 if grad else 1, grad)                    # warm-up (the reward of step 0 does not depend on the policy)
        t0 = time.perf_counter()
        done = 0
        for _ in range(reps):
            self.run(h, grad)
            done += 1
            if time.perf_counter() - t0 > budget_s:
                break
        dt = time.perf_counter() - t0
        what = "forward+backward (torch autograd)" if grad else "forward"
        return done * h / dt, "R=1, %d rollouts of %d steps (of H=%d), %s, factorisations recomputed per step as in the reference" % (
            done, h, self.cfg["H"], what)


_REAL_REF_SCRIPT = r"""
import json, sys, time
import numpy as np
import tensorflow as tf            # noqa: F401  (ImportError -> the caller falls back to the port)
import gpflow                      # noqa: F401
from pilco.models import PILCO
from pilco.controllers import RbfController
from pilco.rewards import ExponentialReward
wl = np.load(sys.argv[1]); h, reps = int(sys.argv[2]), int(sys.argv[3])
Ds, U = wl["Y"].shape[1], wl["X"].shape[1] - wl["Y"].shape[1]
ctrl = RbfController(Ds, U, int(wl["Xc"].shape[0]), max_action=1.0)
p = PILCO((wl["X"], wl["Y"]), controller=ctrl, horizon=h, reward=ExponentialReward(Ds, W=wl["W"], t=wl["t"]),
          m_init=wl["m0"][None], S_init=wl["S0"])
for i, m in enumerate(p.mgpr.models):
    m.kernel.lengthscales.assign(wl["ell"][i]); m.kernel.variance.assign(wl["sf2"][i]); m.likelihood.variance.assign(wl["sn2"][i])
ctrl.set_data((wl["Xc"], wl["Yc"]))
for i, m in enumerate(ctrl.models):
    m.kernel.lengthscales.assign(wl["lc"][i])
p.predict(wl["m0"][None], wl["S0"], h)
t0 = time.perf_counter()
for _ in range(reps):
    p.predict(wl["m0"][None], wl["S0"], h)
print(json.dumps({"steps_per_s": reps * h / (time.perf_counter() - t0)}))
"""


def real_reference_steps_per_s(cfg, wl, reps=2, h_sample=4):
    """BASELINE.md section 2: if a reference install ever appears under baseline/_ref (TensorFlow + GPflow + the reference's
    own ``pilco`` package), time the UNMODIFIED reference through its public API (PILCO.predict, pilco.py:118-136)
    in a separate interpreter (its package name collides with this repo's alias package).  Returns None when it is
    not there or does not import -- the normal case: nothing in /opt/wheelhouse provides tensorflow or gpflow."""
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref_dir, "pilco")) or cfg["bf"] == 0 or "M" in cfg:
        return None
    import tempfile
    try:
        pol = make_policies(cfg, [0])
        with tempfile.TemporaryDirectory() as td:
            np.savez(os.path.join(td, "wl.npz"), Xc=pol["Xc"][0], Yc=pol["Yc"][0], lc=pol["lc"][0], **wl)
            open(os.path.join(td, "run.py"), "w").write(_REAL_REF_SCRIPT)
            env = dict(os.environ, PYTHONPATH=ref_dir)
            out = subprocess.run([sys.executable, os.path.join(td, "run.py"), os.path.join(td, "wl.npz"), str(h_sample), str(reps)],
                                 capture_output=True, text=True, timeout=900, cwd=td, env=env)
        if out.returncode != 0:
            return None
        return float(json.loads(out.stdout.strip().splitlines()[-1])["steps_per_s"])
    except Exception:
        return None


def workload_string(cfg, R):
    return "%s, R=%d restarts/GPU, forward rollout" % (cfg["name"], R)


def run_reference(args, cfg):
    """`--impl reference`: each bench step = ONE bounded sample of the workload (restart 0, the first `h` of the H
    rollout steps) through the reference-equivalent CPU path; W untimed + K timed samples; `steps`/`ms_per_step` are
    the real ones of this run (the run is cut after two minutes, `steps` then says how many samples were timed)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = make_workload(cfg)
    h = 4 if cfg.get("M", cfg["N"]) >= 200 else min(cfg["H"], 10)
    cpu = CpuRollout(cfg, wl)
    nwarm = max(1, min(args.warmup, 2))
    for _ in range(nwarm):
        cpu.run(h)
    K = max(1, args.steps)
    t0 = time.perf_counter()
    done = 0
    for _ in range(K):
        cpu.run(h)
        done += 1
        if time.perf_counter() - t0 > 120.0:              # bounded: never let the CPU arm run past two minutes
            break
    dt = time.perf_counter() - t0
    v = done * h / dt
    kind, note = "port", "reference-equivalent CPU restatement (oracle/torch_port.py); TensorFlow/GPflow are not installable offline"
    sample = "each step = restart 0, first %d of H=%d rollout steps, forward, factorisations recomputed per step as in the reference" % (h, cfg["H"])
    cores = cpu.threads
    real = real_reference_steps_per_s(cfg, wl, reps=max(1, min(done, 3)), h_sample=h)
    if real is not None:
        v, cores, kind = real, os.cpu_count() or 1, "reference"
        note = "the unmodified reference from baseline/_ref through PILCO.predict (TensorFlow/GPflow on the host cores)"
    R = args.restarts or cfg["R"]
    line = {
        "impl": "reference", "metric": metric_name(cfg), "value": v, "unit": UNIT, "n_gpus": args.gpus,
        "steps": done, "warmup": nwarm, "ms_per_step": 1e3 * dt / done, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_string(cfg, R), "restarts_per_gpu": R},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "rollout_steps_per_bench_step": h, "host_cpus": os.cpu_count(),
        "note": note,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.05)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        sm = sorted(float(s[0]) for s in self.samples)
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            for nme, val in zip(names, s[2:]):
                if val.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.samples[0][1]), "reasons": sorted(reasons)}


def build_pilco(cfg, wl, pol):
    """The workload as the reference's own objects (drop-in class API): PILCO + RbfController/LinearController +
    ExponentialReward with the synthetic hyper-parameters assigned (no training)."""
    from pilco.models import PILCO
    from pilco.controllers import RbfController, LinearController
    from pilco.rewards import ExponentialReward
    Ds, U = cfg["Ds"], cfg["U"]
    np.random.seed(0)
    if cfg["bf"]:
        ctrl = RbfController(Ds, U, cfg["bf"], max_action=1.0)
        ctrl.set_data((pol["Xc"][0], pol["Yc"][0]))
        for i, m in enumerate(ctrl.models):
            m.kernel.lengthscales.assign(pol["lc"][0][i])
    else:
        ctrl = LinearController(Ds, U, max_action=1.0)
        ctrl.W.assign(pol["W"][0]); ctrl.b.assign(pol["b"][0][None])
    kw = dict(num_induced_points=cfg["M"]) if "M" in cfg else {}
    p = PILCO((wl["X"], wl["Y"]), controller=ctrl, horizon=cfg["H"], reward=ExponentialReward(Ds, W=wl["W"], t=wl["t"]),
              m_init=wl["m0"][None], S_init=wl["S0"], **kw)
    for i, m in enumerate(p.mgpr.models):
        m.kernel.lengthscales.assign(wl["ell"][i]); m.kernel.variance.assign(wl["sf2"][i]); m.likelihood.variance.assign(wl["sn2"][i])
        if "M" in cfg:
            m.inducing_variable.Z.assign(wl["Z"])
    return p


def run_through_api(args, cfg):
    """`--through-api`: PILCO.optimize_policy(restarts = R x world) under torchrun -- the real sharded path: restart
    r on rank r % world, lock-step SciPy L-BFGS-B, every evaluation one captured graph (policy factorisation, taped
    H-step forward, reverse sweep), ONE all_gather of [loss | params] at the end (NCCL)."""
    import contextlib
    import io
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    if world > 1:
        dist.init_process_group("nccl")
    from pilco_b200 import policy_opt
    R = args.restarts or cfg["R"]
    wl = make_workload(cfg)
    p = build_pilco(cfg, wl, make_policies(cfg, [0]))
    sink = io.StringIO()
    with contextlib.redirect_stdout(sink):                 # (randomize() / optimize_policy() print per restart)
        p.optimize_policy(maxiter=2, restarts=R * world)   # warm-up: builds the evaluator, captures its graph
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        reward = p.optimize_policy(maxiter=args.maxiter, restarts=R * world)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
    st = dict(policy_opt.LAST_STATS)
    tt = torch.tensor([dt, float(st.get("rollout_steps", st["evals"] * st["restarts_local"] * st["horizon"]))], dtype=torch.float64, device="cuda")
    if world > 1:
        tmax = tt.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = tt.clone(); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        dt, steps = float(tmax[0]), float(tsum[1])
    else:
        steps = float(tt[1])
    if rank == 0:
        print(json.dumps({
            "metric": metric_name(cfg) + " through PILCO.optimize_policy", "value": steps / dt, "unit": UNIT, "n_gpus": world,
            "steps": args.maxiter, "warmup": 2, "ms_per_step": 1e3 * dt / max(st["evals"], 1), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "%s; PILCO.optimize_policy(maxiter=%d, restarts=%d): lock-step L-BFGS-B, forward + reverse sweep per evaluation, wall clock incl. SciPy and host<->device copies"
                                   % (cfg["name"], args.maxiter, R * world), "restarts_per_gpu": R},
            "loss_evaluations": st["evals"], "lockstep_groups": st.get("groups", 1), "wall_s": dt, "best_reward": float(reward),
        }))
    if world > 1:
        dist.destroy_process_group()


def run_ours(args, cfg):
    import torch
    import torch.distributed as dist
    from pilco_b200 import engine, _lib
    from pilco_b200._lib import lib
    from pilco_b200.engine import ptr, stream_ptr

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl")
    d = engine.device()
    R, H = args.restarts or cfg["R"], cfg["H"]
    Ds, U, bf = cfg["Ds"], cfg["U"], cfg["bf"]
    D = Ds + U
    wl = make_workload(cfg)

    def timeit(fn, reps=3):
        fn(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record(); torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps
    if "M" in cfg:                                          # FITC over M inducing points (once per set_data / hyper change)
        gp = engine.fitc_factorize(wl["X"], wl["Z"], wl["Y"], wl["ell"], wl["sf2"], wl["sn2"])
        fact_ms = timeit(lambda: engine.fitc_factorize(wl["X"], wl["Z"], wl["Y"], wl["ell"], wl["sf2"], wl["sn2"]))
    else:
        gp = engine.gp_factorize(wl["X"], wl["Y"], wl["ell"], wl["sf2"], wl["sn2"])      # once per set_data
        fact_ms = timeit(lambda: engine.gp_refactorize(gp))
    n_c = gp.n                                              # centres of the moment match (N, or M for SMGPR)
    my_ids = np.arange(rank * R, (rank + 1) * R)            # weak scaling: R per GPU
    pol = make_policies(cfg, my_ids)
    ones, noise = np.ones((R, U)), 1e-4 * np.ones((R, U))
    maxa = np.ones(U)
    rew = [dict(kind=_lib.REWARD_EXP, coef=1.0, W=wl["W"], t=wl["t"])]
    nsplit = max(1, min(args.nsplit, R))

    def policy_spec(lo, hi, store):
        if bf == 0:
            return dict(kind=_lib.POLICY_LINEAR, Ds=Ds, U=U, squash=True, max_action=maxa, W=pol["W"][lo:hi], b=pol["b"][lo:hi])
        pg = engine.gp_factorize(pol["Xc"][lo:hi], pol["Yc"][lo:hi], pol["lc"][lo:hi], ones[lo:hi], noise[lo:hi], need_iK=False, mode=1)
        store[(lo, hi)] = pg
        return dict(kind=_lib.POLICY_RBF, Ds=Ds, U=U, squash=True, max_action=maxa, gp=pg)

    # ---- device-resident arm: policy parameters already in HBM, rollout only --------------------------
    # The H-step loop of all R restarts is ONE CUDA graph: nsplit sub-batches on parallel streams (their
    # latency-bound per-step kernels overlap each other's tile kernels).
    pgps = {}

    def make_plan(lo, hi, grad=False):
        return engine.RolloutPlan(gp, policy_spec(lo, hi, pgps), rew, wl["m0"], wl["S0"], H, R=hi - lo, grad=grad)

    split = engine.SplitRollout(make_plan, R, nsplit=nsplit)
    flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device=d)       # > L2 (126 MB)
    gathered = [torch.empty(R, dtype=torch.float64, device=d) for _ in range(world)]

    def step_resident():
        rw = split.replay()
        if world > 1:
            dist.all_gather(gathered, rw)

    # ---- end-to-end arm: host buffers in, host result out -----------------------------------------
    # What one optimiser evaluation does through the public engine objects: pinned host policy parameters ->
    # device, policy factorisation (beta = (K+sn2 I)^-1 Y, pilco_gp_factorize), H-step rollout, rewards -> host.
    # Device work is one captured CUDA graph (refactorise + cascade, same sub-batch split) replayed per step.
    keys = ("W", "b") if bf == 0 else ("Xc", "Yc", "lc")
    hbuf = {k: torch.as_tensor(pol[k]).pin_memory() for k in keys}
    h_out = torch.empty(R, dtype=torch.float64).pin_memory()
    h2d = sum(v.numel() for v in hbuf.values()) * 8
    d2h = R * 8

    def plan_factory(pgs, plans, grad):
        def make(lo, hi):
            pl = engine.RolloutPlan(gp, policy_spec(lo, hi, pgs), rew, wl["m0"], wl["S0"], H, R=hi - lo, grad=grad)
            plans[(lo, hi)] = pl
            if bf:
                pg = pgs[(lo, hi)]
                fwd = pl.forward
                pl.forward = lambda: (engine.gp_refactorize(pg), fwd())[1]      # refactorise inside the captured graph
            return pl
        return make

    pg2, plans2 = {}, {}
    split2 = engine.SplitRollout(plan_factory(pg2, plans2, False), R, nsplit=nsplit)

    def upload(plans, pgs):
        for (lo, hi), pl in plans.items():
            if bf == 0:
                pl.W.copy_(hbuf["W"][lo:hi], non_blocking=True); pl.b.copy_(hbuf["b"][lo:hi], non_blocking=True)
            else:
                pg = pgs[(lo, hi)]
                pg.X.copy_(hbuf["Xc"][lo:hi], non_blocking=True); pg.Y.copy_(hbuf["Yc"][lo:hi], non_blocking=True)
                pg.ell.copy_(hbuf["lc"][lo:hi], non_blocking=True)

    def step_e2e():
        upload(plans2, pg2)
        rw = split2.replay()
        h_out.copy_(rw, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    def timed(fn, K, W):
        for _ in range(W):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        tot = 0.0
        for _ in range(K):
            flush.fill_(1.0)                                   # L2 flush between timed iterations (untimed)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            tot += e0.elapsed_time(e1)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t = torch.tensor([tot], dtype=torch.float64, device=d)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)           # max over ranks
        return float(t.item()) / K                             # ms per step

    # ---- forward + reverse sweep (policy gradient): the loop optimize_policy runs ------------------------
    # taped forward (pilco_rollout.tape) + tape-driven reverse sweep; device resident and end to end
    # (host parameters in, [reward | gradient] out), one captured graph each
    split3 = split4 = None
    nsplit_b = max(1, min(args.nsplit_bwd, R))
    if args.with_backward:
        split3 = engine.SplitRollout(lambda lo, hi: make_plan(lo, hi, grad=True), R, nsplit=nsplit_b, backward=True)
        pg4, plans4 = {}, {}
        split4 = engine.SplitRollout(plan_factory(pg4, plans4, True), R, nsplit=nsplit_b, backward=True)
        gkeys = ("W", "b") if bf == 0 else ("X", "Y", "ell")
        first = plans4[next(iter(plans4))]
        gsz = sum(int(np.prod(first.gbuf[k].shape[1:])) for k in gkeys)
        h_grad = torch.empty((R, 1 + gsz), dtype=torch.float64).pin_memory()
        d_grad = torch.empty((R, 1 + gsz), dtype=torch.float64, device=d)

    # The restarts are independent optimisation problems: policy_opt deals them to lock-step GROUPS that only wait for
    # their own previous evaluation, half an evaluation out of phase, so one group's latency-bound reverse sweep runs
    # under the other's tile kernels.  The grouped arms time exactly that: K evaluations per group, back to back on the
    # group's stream, the phase offset INSIDE the timed region.
    G = max(1, min(args.groups, R // 8)) if args.with_backward else 1
    gsplit3 = gsplit4 = None
    if G > 1:
        gb = [round(k * R / G) for k in range(G + 1)]
        gsl = [(gb[k], gb[k + 1]) for k in range(G)]

        def shifted(make, off):
            return lambda lo, hi: make(lo + off, hi + off)
        gsplit3 = [engine.SplitRollout(shifted(lambda lo, hi: make_plan(lo, hi, grad=True), lo), hi - lo, nsplit=nsplit_b, backward=True)
                   for lo, hi in gsl]
        pg5, plans5 = [dict() for _ in gsl], [dict() for _ in gsl]
        gsplit4 = [engine.SplitRollout(shifted(plan_factory(pg5[k], plans5[k], True), lo), hi - lo, nsplit=nsplit_b, backward=True)
                   for k, (lo, hi) in enumerate(gsl)]
        gstreams = [torch.cuda.Stream() for _ in gsl]
        group_ms = timeit(gsplit3[0].replay)                   # one group alone: sets the phase offset
        stagger_ms = args.stagger_ms if args.stagger_ms > 0 else group_ms / G

    def pipeline(K, e2e):
        """K evaluations of every group; returns the elapsed device time [ms] (events on the main stream, which the
        group streams fork from and join into)."""
        import threading
        cur = torch.cuda.current_stream()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0.record()
        for st in gstreams:
            st.wait_stream(cur)
        if not e2e:
            for g, st in enumerate(gstreams):
                if g:
                    with torch.cuda.stream(st):
                        torch.cuda._sleep(int(g * stagger_ms * 1.9e6))     # ~SM cycles
            for _ in range(K):
                for g, st in enumerate(gstreams):
                    with torch.cuda.stream(st):
                        gsplit3[g].replay()
        else:
            def drive(g):
                torch.cuda.set_device(local)
                (lo, hi), st = gsl[g], gstreams[g]
                time.sleep(g * stagger_ms * 1e-3)
                with torch.cuda.stream(st):
                    for _ in range(K):                             # what one lock-step group does per evaluation
                        upload(plans5[g], pg5[g])
                        rw = gsplit4[g].replay()
                        d_grad[lo:hi, 0] = rw
                        for (a, b), pl in plans5[g].items():
                            d_grad[a:b, 1:] = torch.cat([pl.gbuf[k].reshape(b - a, -1) for k in gkeys], dim=1)
                        h_grad[lo:hi].copy_(d_grad[lo:hi], non_blocking=True)
                        st.synchronize()                           # the host optimiser needs the values
            ths = [threading.Thread(target=drive, args=(g,)) for g in range(G)]
            for t in ths:
                t.start()
            for t in ths:
                t.join()
        for st in gstreams:
            cur.wait_stream(st)
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=d)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def step_fwd_bwd():
        split3.replay()

    def step_fwd_bwd_e2e():
        upload(plans4, pg4)
        rw = split4.replay()
        d_grad[:, 0] = rw
        for (lo, hi), pl in plans4.items():
            d_grad[lo:hi, 1:] = torch.cat([pl.gbuf[k].reshape(hi - lo, -1) for k in gkeys], dim=1)
        h_grad.copy_(d_grad, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    ms_res = timed(step_resident, args.steps, args.warmup)
    ok = int(split.info.max().item()) == 0 and bool(torch.isfinite(split.reward).all().item())
    ms_e2e = timed(step_e2e, args.steps, args.warmup)
    ms_fb = ms_fb_e2e = ms_fbg = ms_fbg_e2e = None
    if split3 is not None:
        ms_fb = timed(step_fwd_bwd, args.steps, 3)
        ms_fb_e2e = timed(step_fwd_bwd_e2e, args.steps, 3)
        if G > 1:
            pipeline(3, False)
            ms_fbg = pipeline(args.steps, False) / args.steps
            pipeline(3, True)
            ms_fbg_e2e = pipeline(args.steps, True) / args.steps
    if sampler:
        sampler.stop_flag = True
        sampler.join(timeout=2)
    if args.dump_outputs and rank == 0:
        out = {"rollout_traj_m": torch.cat([p.traj_m for p in split.plans]),
               "rollout_traj_S": torch.cat([p.traj_S for p in split.plans]),
               "rollout_reward": split.reward, "e2e_reward": h_out}
        if split3 is not None:
            fb_plans = [p for sp in gsplit3 for p in sp.plans] if G > 1 else split3.plans
            out["fwd_bwd_reward"] = torch.cat([p.reward for p in fb_plans])
            for k in gkeys:
                out["fwd_bwd_grad_" + k] = torch.cat([p.gbuf[k] for p in fb_plans])
            out["fwd_bwd_e2e_reward_grad"] = h_grad
        dump_outputs(args.dump_outputs, my_ids, {k: v.cpu().numpy() for k, v in out.items()})

    total_steps = R * H * world
    value = total_steps / (ms_res * 1e-3)
    e2e_value = total_steps / (ms_e2e * 1e-3)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- class-API line: PILCO.predict(m, S, H) with host arrays in / out (one restart, the reference's call) ----
    api = None
    if args.api_line:
        try:
            p = build_pilco(cfg, wl, make_policies(cfg, [0]))
            p.predict(wl["m0"][None], wl["S0"], H)             # builds + captures the cached plan
            reps = 20
            t0 = time.perf_counter()
            for _ in range(reps):
                p.predict(wl["m0"][None], wl["S0"], H)
            dt = (time.perf_counter() - t0) / reps
            api = {"call": "pilco.models.PILCO.predict(m, S, %d) -- numpy in, numpy out, R=1" % H, "ms_per_call": 1e3 * dt,
                   "value": H / dt, "unit": UNIT, "us_per_rollout_step": 1e6 * dt / H}
        except Exception as exc:                               # pragma: no cover
            api = {"error": repr(exc)}

    # ---- roofline of the dominant kernel (dynamics tile kernel: plain forward, and taped) ----------------------
    ms3 = (C.c_float * 3)()
    g = gp.struct()
    E = Ds
    Mo = torch.empty((R, E), dtype=torch.float64, device=d); So = torch.empty((R, E, E), dtype=torch.float64, device=d)
    Vo = torch.empty((R, D, E), dtype=torch.float64, device=d); info = torch.zeros(R, dtype=torch.int32, device=d)
    wsb = lib.pilco_mm_workspace_bytes(n_c, D, E, R)
    ws = torch.empty(wsb // 8, dtype=torch.float64, device=d)
    tb = lib.pilco_mm_tape_bytes(n_c, D, E, R)
    tape = torch.empty(max(tb // 8, 2), dtype=torch.float64, device=d)
    mj = engine.dev(np.tile(np.concatenate([wl["m0"], np.zeros(U)]), (R, 1)))
    sj = engine.dev(np.tile(0.1 * np.eye(D), (R, 1, 1)))
    tile_ms, setup_ms, ttile_ms = [], [], []
    for i in range(8):
        flush.fill_(1.0)
        _lib.check(lib.pilco_mm_forward_profile(C.byref(g), R, ptr(mj), ptr(sj), ptr(Mo), ptr(So), ptr(Vo), ptr(info),
                                                ptr(ws), wsb, ms3, stream_ptr()))
        if i >= 3:
            setup_ms.append(ms3[0]); tile_ms.append(ms3[1])
        if tb:
            flush.fill_(1.0)
            _lib.check(lib.pilco_mm_forward_taped_profile(C.byref(g), R, ptr(mj), ptr(sj), ptr(Mo), ptr(So), ptr(Vo), ptr(info),
                                                          ptr(ws), wsb, ptr(tape), tb, ms3, stream_ptr()))
            if i >= 3:
                ttile_ms.append(ms3[1])
    tile_ms = float(np.mean(tile_ms)); setup_ms = float(np.mean(setup_ms))
    ttile_ms = float(np.mean(ttile_ms)) if ttile_ms else None
    # fp64 pipe peaks measured live (DFMA and DMMA microbenchmarks, same process): 8 DMMA.8x8x4 per warp and iteration,
    # 256 FMA = 512 flop each
    sink = torch.zeros(8, dtype=torch.float64, device=d)
    msf = C.c_float()
    iters, blocks = 20000, 148 * 4
    _lib.check(lib.pilco_microbench_fp64(0, iters, blocks, ptr(sink), C.byref(msf), stream_ptr()))
    dfma_tf = 2 * blocks * 256 * iters * 8.0 / (msf.value * 1e-3) / 1e12
    _lib.check(lib.pilco_microbench_fp64(1, iters, blocks, ptr(sink), C.byref(msf), stream_ptr()))
    dmma_tf = blocks * 8 * iters * 8.0 * 512 / (msf.value * 1e-3) / 1e12
    # independent library denominator (NOT on the product path): cuBLAS DGEMM through torch.matmul
    lib_tf, nmm = None, 6144
    try:
        a_ = torch.randn(nmm, nmm, dtype=torch.float64, device=d); b_ = torch.randn(nmm, nmm, dtype=torch.float64, device=d)
        torch.matmul(a_, b_); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); torch.matmul(a_, b_); torch.matmul(a_, b_); e1.record(); torch.cuda.synchronize()
        lib_tf = 2 * 2.0 * nmm ** 3 / (e0.elapsed_time(e1) * 1e-3) / 1e12
        del a_, b_
    except Exception:
        pass
    P = E * (E + 1) // 2
    nn = float(n_c) * n_c
    ks = (D + 3) // 4

    def tile_block(ms, elems, dmma_extra, dfma_extra, label, trace_elems):
        dot = 2.0 * D * elems                                  # Q-contraction U'.zeta (DMMA)
        hz = dmma_extra * elems                                # second product H.[Z,1] (taped only, DMMA)
        other = (EXP_FLOP_EQ + dfma_extra) * elems + 2.0 * trace_elems
        flops = dot + hz + other
        ach = flops / (ms * 1e-3) / 1e12
        peak = flops / ((dot + hz) / dmma_tf + other / dfma_tf)   # time-weighted fp64 peak for this kernel's op mix
        return {"kernel": label, "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                "tensor_flops_share": (dot + hz) / flops, "q_contraction_tflops": dot / (ms * 1e-3) / 1e12, "kernel_ms": ms}
    # plain forward: symmetric (a == a) pairs need only half of their n x n elements; A'+B ride in the DMMA C operand /
    # rounding constant, so per element: the dot, one exp, one weighted add (+ trace term on diagonal pairs)
    rf = tile_block(tile_ms, (float(P) - 0.5 * E) * nn * R, 0.0, 2.0,
                    "mm_tile_kernel<%d,3,true> (dynamics GP: fp64 DMMA Q-contraction + table exp + beta/iK-weighted sums)" % ks,
                    0.5 * E * nn * R)
    # compulsory bytes per launch (SURVEY 8d): iK once (shared by the batch) + per restart X-m, beta, hypers, s, outputs
    alg_bytes = 8.0 * (E * nn + R * (n_c * D + E * n_c + 2 * E * D + D * D + D + E + E * E + D * E))
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    traffic = tsrc = None                # dram bytes per launch of the same kernel/config from the committed ncu --set full capture
    if cfg is CONFIGS["metric"] and R == 32:
        for fn in ("r02_tile_traffic.json", "r01_tile_traffic.json"):
            try:
                traffic = json.load(open(os.path.join(ROOT, "profiles", fn)))["dram_bytes_per_launch"]
                tsrc = "profiles/" + fn + " (ncu --set full, same kernel and config; cold caches: in the pipeline the operands written by the setup kernel are L2 hits)"
                break
            except Exception:
                pass
    roofline = dict(rf)
    roofline.update({
        "bound": "tensor", "traffic": traffic, "traffic_source": tsrc,
        "algorithmic_bytes": alg_bytes, "traffic_over_algorithmic": (traffic / alg_bytes) if traffic else None,
        "peak_source": "fp64 pipe measured live by pilco_microbench_fp64 (DFMA %.1f, DMMA %.1f TFLOP/s: 512 flop per warp-level DMMA.8x8x4), "
                       "time-weighted for this kernel's op mix; MEASURED_PEAKS.json holds no fp64 figure" % (dfma_tf, dmma_tf),
        "fp64_library_tflops": lib_tf,
        "fp64_library_note": "cuBLAS DGEMM %d^3 through torch.matmul in this process: independent denominator only, not on the product path" % nmm,
        "frac_of_library": (rf["achieved"] / lib_tf) if lib_tf else None,
        "setup_kernel_ms": setup_ms,
        "hbm": {"achieved_gbs": alg_bytes / (tile_ms * 1e-3) / 1e9, "peak_gbs": hbm_peak,
                "frac": alg_bytes / (tile_ms * 1e-3) / 1e9 / hbm_peak,
                "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback"},
    })
    # whole step: SURVEY 8d flop + exp count of one rollout step x steps / measured time
    F, Xe, Bs = step_counts(cfg)
    step_flop_eq = F + EXP_FLOP_EQ * Xe
    pipe_peak = min(dfma_tf, dmma_tf)
    roofline["whole_step"] = {"flop_eq_per_rollout_step": step_flop_eq, "achieved": step_flop_eq * R * H / (ms_res * 1e-3) / 1e12,
                              "peak": pipe_peak, "unit": "TFLOP/s", "frac": step_flop_eq * R * H / (ms_res * 1e-3) / 1e12 / pipe_peak,
                              "compulsory_bytes_per_rollout_step": Bs}
    fb = None
    if ms_fb is not None:
        fb = {"value": total_steps / (ms_fb * 1e-3), "unit": UNIT, "ms_per_step": ms_fb,
              "what": "taped forward cascade + tape-driven reverse sweep (policy gradient), device resident, %d sub-batches on parallel streams" % nsplit_b,
              "e2e": {"value": total_steps / (ms_fb_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_fb_e2e,
                      "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": int(h_grad.numel()) * 8,
                      "what": "pinned host policy parameters -> device, policy factorisation, taped forward, reverse sweep, [reward | gradient] -> host"}}
        if ms_fbg is not None:
            # headline = the grouped pipeline (what policy_opt runs); the single lock-step batch is kept beside it
            fb["single_group"] = {"value": fb["value"], "ms_per_step": fb["ms_per_step"], "what": fb["what"],
                                  "e2e_value": fb["e2e"]["value"], "e2e_ms_per_step": fb["e2e"]["ms_per_step"],
                                  "l2": "flushed between timed iterations"}
            fb.update({"value": total_steps / (ms_fbg * 1e-3), "ms_per_step": ms_fbg, "steps": args.steps, "groups": G,
                       "what": "taped forward cascade + tape-driven reverse sweep (policy gradient), device resident: %d lock-step groups of %d restarts "
                               "(x %d sub-batches on parallel streams), each group's evaluations back to back on its own stream, "
                               "groups %.1f ms out of phase (offset inside the timed region) -- the schedule policy_opt.optimize runs"
                               % (G, R // G, nsplit_b, stagger_ms),
                       "l2": "no flush between the pipelined steps: a step writes and re-reads its tape (%.1f GB per step over all restarts), far beyond the 126 MB L2"
                             % (1e-9 * sum(pl.tape.numel() * 8 for sp in gsplit3 for pl in sp.plans if pl.tape is not None))})
            fb["e2e"].update({"value": total_steps / (ms_fbg_e2e * 1e-3), "ms_per_step": ms_fbg_e2e,
                              "what": fb["e2e"]["what"] + "; one host thread per group, stream-synchronised after every evaluation"})
        if ttile_ms:
            # taped tile pass: every pair over its full square; per element the dot, the exp, the weight and column-sum
            # updates (2 DFMA-class ops) and the second product H.[Z,1] (2 (D+1) flop)
            fb["roofline"] = tile_block(ttile_ms, float(P) * nn * R, 2.0 * (D + 1), 4.0,
                                        "mm_tape_tile_kernel<%d> (taped dynamics pass: Q-contraction + exp + H.[Z,1] product + column sums)" % ks, 0.0)
            fb["roofline"]["bound"] = "tensor"
    cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": "skipped (--no-cpu-baseline)"}
    if args.cpu_baseline:
        cr = CpuRollout(cfg, wl)
        hs = 4 if n_c >= 200 else min(H, 10)
        v, sample = cr.steps_per_s(reps=2, h=hs, budget_s=20.0)
        cpu = {"value": v, "unit": UNIT, "cores": cr.threads, "kind": "port", "sample": sample, "host_cpus": os.cpu_count()}
        if fb is not None:
            vb, sb = cr.steps_per_s(reps=1, h=2 if n_c >= 200 else min(H, 6), grad=True, budget_s=20.0)
            fb["cpu_baseline"] = {"value": vb, "unit": UNIT, "cores": cr.threads, "kind": "port", "sample": sb}
    launches_per_rollout = (H * (8 if bf else 4) + 1) + 1 + 2  # per sub-batch: ro_state + [policy: setup1, setup2, tile, ro_policy] + dyn (setup1, setup2, tile); + memset; + ro_reward, ro_reward_sum
    line = {
        "metric": metric_name(cfg), "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_res, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_string(cfg, R), "restarts_per_gpu": R,
                   "graph": "one CUDA graph per rollout batch, %d sub-batches on parallel streams" % nsplit,
                   "l2": "flushed between timed iterations (256 MiB write)", "finite": ok},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": ms_e2e, "what": "pinned host policy parameters -> device, policy factorisation, H-step rollout, rewards -> host"},
        "fwd_bwd": fb,
        "api_predict": api,
        "factorize_ms": fact_ms,
        "gpu_launches": nsplit * launches_per_rollout * args.steps,
        "roofline": roofline,
        "cpu_baseline": cpu,
        "clocks": sampler.summary() if sampler else None,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="metric", choices=sorted(CONFIGS))
    ap.add_argument("--restarts", type=int, default=0, help="policy restarts per GPU (default: the config's)")
    ap.add_argument("--no-backward", dest="with_backward", action="store_false", help="skip the forward+backward lines")
    ap.add_argument("--no-cpu-baseline", dest="cpu_baseline", action="store_false", help="tuning runs: skip the CPU legs")
    ap.add_argument("--no-api-line", dest="api_line", action="store_false", help="skip the PILCO.predict class-API line")
    ap.add_argument("--nsplit", type=int, default=8, help="sub-batches on parallel streams inside the captured graph (forward arms)")
    ap.add_argument("--nsplit-bwd", type=int, default=4, help="... for the forward+backward arms (measured: 4 beats 8 for the reverse sweep)")
    ap.add_argument("--groups", type=int, default=2, help="lock-step groups of the forward+backward arms (policy_opt.GROUPS); 1 = one batch")
    ap.add_argument("--stagger-ms", type=float, default=0.0, help="phase offset between the groups (default: one group's evaluation time / groups)")
    ap.add_argument("--through-api", action="store_true", help="drive PILCO.optimize_policy itself (lock-step L-BFGS-B, sharded restarts)")
    ap.add_argument("--maxiter", type=int, default=10, help="--through-api: L-BFGS-B iterations")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step of each arm returned as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.through_api):
        ap.error("--dump-outputs applies to the default arm (not --impl reference or --through-api)")
    cfg = CONFIGS[args.config]
    # Exactly ONE line on stdout (the JSON): everything any library writes to file descriptor 1 meanwhile (NCCL's
    # "NCCL version ..." banner is written by C code, not through sys.stdout) is sent to stderr; the JSON line is
    # printed through the saved descriptor.
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    real_stdout = os.fdopen(saved, "w")
    import builtins
    _print = builtins.print

    def print_json(*a, **k):
        k.setdefault("file", real_stdout)
        _print(*a, **k)
        real_stdout.flush()
    g = globals()
    g["print"] = print_json                                  # the run_* functions print only the JSON line
    try:
        if args.impl == "reference":
            run_reference(args, cfg)
        elif args.through_api:
            run_through_api(args, cfg)
        else:
            run_ours(args, cfg)
    finally:
        g.pop("print", None)
        sys.stdout.flush()


if __name__ == "__main__":
    main()
