#!/usr/bin/env python
"""bench.py -- PPO update throughput (BASELINE.json metric) on synthetic HalfCheetah-shaped batches.

  python bench.py --gpus N --steps K --warmup W            # our arm (one rank per GPU under torchrun for N > 1)
  python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port) on the host cores

A "step" = one full PPO.train()-equivalent on one batch: value inference on N+E rows -> GAE/return scan ->
normalisation -> 80 policy-gradient steps (+ final KL pass) -> old-policy sync -> 80 value steps
(early stop disabled: max_kl = inf, so the work is fixed; SURVEY.md section 8d).
Workload at N GPUs: 1024 envs x 1000 steps PER GPU (BASELINE configs[1]; configs[4] at N = 8) -- weak scaling.

  value : transitions/s with the batch already resident in HBM (engine.update only).
  e2e   : same through the public API, PPO.train(experience) with a PackedExperience in pinned host memory (the
          rollout store a sampler fills): host -> device copies of the batch, parameter / optimizer-state upload, the
          update, and the device -> host read-back of parameters, optimizer state and the logged scalars, all inside the
          timed region.

The CPU legs (`cpu_baseline` of the default run, `--impl reference`) run the UNMODIFIED reference, pip-installed from
/root/reference into git-ignored baseline/_ref by __graft_entry__.build() (kind "reference"); only if that package is
absent they fall back to oracle/torch_port.py (kind "port").  The measured arm imports neither: it builds its learners
and synthetic data from `rl_replicas_b200.synthetic` alone.

  --dump-outputs DIR : after the timed steps, write what the last step of each timed leg computed as DIR/<name>.npy
                       (parameters, Adam moments and update statistics; inputs are seeded, so two builds can be compared
                       output for output).
"""
from __future__ import annotations

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
sys.path.insert(0, os.path.join(ROOT, "tests"))

OBS, ACT, HID = 17, 6, 64
POLICY_SIZES, VALUE_SIZES = [OBS, HID, HID, ACT], [OBS, HID, HID, 1]
N_POLICY, N_VALUE = 80, 80
# algorithmic fp32-equivalent FLOPs per row (2*MAC), SURVEY.md section 8: policy fwd 11136 / bwd 20096, value 10496 / 18816
FLOP_POLICY_STEP = 11136 + 20096
FLOP_VALUE_STEP = 10496 + 18816
FLOP_FUSED_STEP = FLOP_POLICY_STEP + FLOP_VALUE_STEP  # one mlp_tc3 launch = policy step + value step
FLOP_PER_TRANSITION = (N_POLICY + 1) * 11136 + N_POLICY * 20096 + (N_VALUE + 1) * 10496 + N_VALUE * 18816


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm=p["hbm_gbs"], tf_burst=p["bf16_tflops"], tf_sust=p["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback")


def make_nets(seed=0):
    rng = np.random.default_rng(seed)
    mk = lambda sz: [(rng.standard_normal((o, i)).astype(np.float32) / np.sqrt(i), np.zeros(o, np.float32))
                     for i, o in zip(sz[:-1], sz[1:])]
    return mk(POLICY_SIZES), mk(VALUE_SIZES), np.full(ACT, -0.5, np.float32)


def make_batch(n_envs, horizon, pl, seed):
    from rl_replicas_b200 import synthetic

    def mean_fn(o):  # on-policy-like actions: mu_theta0(obs) + sigma * noise (SURVEY 8d config 2)
        h = o
        for i, (w, b) in enumerate(pl):
            h = h @ w.T + b
            if i < len(pl) - 1:
                h = np.tanh(h)
        return h

    return synthetic.fixed_batch(n_envs, horizon, OBS, ACT, seed=seed, frac_not_done=0.1, mean_fn=mean_fn)


# UpdateStats fields that are results of the update (kernel_launches / fused describe how it ran, not what it computed)
STAT_FIELDS = ("policy_loss_before", "entropy_before", "logp_std_before", "kl_divergence", "value_loss_mean",
               "policy_steps_applied", "value_steps_applied", "adv_mean", "adv_std", "value_loss_first", "value_loss_last")


def stats_array(stats):
    return np.array([float(getattr(stats, f)) for f in STAT_FIELDS], dtype=np.float64)


def learner_outputs(prefix, ppo):
    """What PPO.train leaves its caller: the networks' parameters, the Adam moments and step, the update statistics."""
    from rl_replicas_b200.algorithms._onpolicy import describe_mlp, flat_params, read_adam_state
    out = {f"{prefix}_stats": stats_array(ppo.last_update_stats)}
    for name, module in (("policy", ppo.policy), ("value", ppo.value_function)):
        linears = describe_mlp(module.network)[3]
        m, v, step = read_adam_state(module.optimizer, linears)
        out.update({f"{prefix}_{name}_params": flat_params(linears), f"{prefix}_{name}_adam_exp_avg": m,
                    f"{prefix}_{name}_adam_exp_avg_sq": v, f"{prefix}_{name}_adam_step": np.float64(step)})
    return out


def engine_outputs(prefix, engine, stats):
    """What OnPolicyEngine.update leaves its caller: the returned statistics and the device-resident parameters and
    Adam state, read back."""
    from rl_replicas_b200.engine import POLICY, VALUE
    out = {f"{prefix}_stats": stats_array(stats)}
    for name, which in (("policy", POLICY), ("value", VALUE)):
        m, v, step = engine.get_adam(which)
        out.update({f"{prefix}_{name}_params": engine.get_params(which), f"{prefix}_{name}_adam_exp_avg": m,
                    f"{prefix}_{name}_adam_exp_avg_sq": v, f"{prefix}_{name}_adam_step": np.float64(step)})
    return out


def dump_outputs(directory, arrays):
    """DIR/<name>.npy per array, as float32 or float64."""
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        np.save(os.path.join(directory, name + ".npy"), a if a.dtype in (np.float32, np.float64) else a.astype(np.float64))


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_evt = index, [], threading.Event()

    def run(self):
        while not self.stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop_evt.wait(0.2)

    def summary(self):
        self.stop_evt.set()
        self.join(timeout=3)
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


def _numa0_cpus():
    """CPUs of NUMA node 0 (the reference arm is pinned there: no cross-socket traffic, repeatable timings)."""
    try:
        txt = open("/sys/devices/system/node/node0/cpulist").read().strip()
        cpus = []
        for part in txt.split(","):
            lo, _, hi = part.partition("-")
            cpus += list(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0)
        cpus = [c for c in cpus if c in allowed]
        return cpus or sorted(allowed)
    except Exception:
        return sorted(os.sched_getaffinity(0))


def _import_reference():
    """The unmodified reference from baseline/_ref (None if it was not installed).  gymnasium is not in the image and the
    update path uses it for type annotations only (SURVEY 8c): a stub module stands in."""
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref_dir, "rl_replicas")):
        return None
    import types
    if "gymnasium" not in sys.modules:
        gym, spaces = types.ModuleType("gymnasium"), types.ModuleType("gymnasium.spaces")
        for name in ("Env", "Space"):
            setattr(gym, name, type(name, (), {}))
        for name in ("Box", "Discrete"):
            setattr(spaces, name, type(name, (gym.Space,), {}))
        gym.spaces, gym.make = spaces, (lambda *a, **k: None)
        sys.modules["gymnasium"], sys.modules["gymnasium.spaces"] = gym, spaces
    if ref_dir not in sys.path:
        sys.path.insert(0, ref_dir)
    try:
        import rl_replicas  # noqa: F401
        from rl_replicas.algorithms import PPO  # noqa: F401
        return rl_replicas
    except Exception:
        return None


def cpu_reference_run(steps, warmup, n_envs=64, horizon=1000):
    """The reference's CPU path for this workload: rl_replicas.algorithms.PPO.train(experience) itself when the package
    is installed under baseline/_ref, on a bounded sample of the same workload (n_envs x horizon transitions, the same
    80 + 80 full-batch steps; throughput is size-independent to first order), pinned to NUMA node 0 with a fixed thread
    count.  Returns (cpu_baseline dict, best seconds per step)."""
    import torch
    cpus = _numa0_cpus()
    try:
        os.sched_setaffinity(0, cpus)
    except Exception:
        pass
    threads = max(1, min(32, len(cpus) // 2 if len(cpus) >= 4 else len(cpus)))  # physical cores of the node, at most 32
    torch.set_num_threads(threads)  # torchrun exports OMP_NUM_THREADS=1 to every rank; this arm uses the host's cores
    pl, vl, log_std = make_nets()
    b = make_batch(n_envs, horizon, pl, seed=0)
    n = n_envs * horizon
    ref = _import_reference()
    if ref is not None:
        from rl_replicas.algorithms import PPO
        from rl_replicas.experience import Experience
        from rl_replicas.networks import MLP
        from rl_replicas.policies import GaussianPolicy
        from rl_replicas.value_function import ValueFunction
        from rl_replicas_b200 import synthetic

        def load(net, layers):
            linears = [m for m in net.modules() if isinstance(m, torch.nn.Linear)]
            with torch.no_grad():
                for lin, (w, bias) in zip(linears, layers):
                    lin.weight.copy_(torch.from_numpy(w))
                    lin.bias.copy_(torch.from_numpy(bias))

        pnet, vnet = MLP(POLICY_SIZES), MLP(VALUE_SIZES)
        load(pnet, pl)
        load(vnet, vl)
        policy = GaussianPolicy(pnet, torch.optim.Adam(pnet.parameters(), lr=3e-4),
                                torch.nn.Parameter(torch.from_numpy(log_std.copy())))
        vf = ValueFunction(vnet, torch.optim.Adam(vnet.parameters(), lr=1e-3))
        algo = PPO(policy, vf, None, None, num_policy_gradients=N_POLICY, num_value_gradients=N_VALUE,
                   max_kl_divergence=float("inf"))

        class _Sink:
            def record_scalar(self, *a, **k):
                pass

        algo.metrics_manager, algo.current_total_steps = _Sink(), 0
        exp = Experience(**synthetic.to_experience_lists(b, False))
        step_fn, kind = (lambda: algo.train(exp)), "reference"
        what = "rl_replicas 0.0.7 PPO.train(experience), unmodified, from baseline/_ref"
    else:
        from oracle import torch_port as T
        step_fn = lambda: T.ppo_train(b, pl, vl, "gaussian", log_std, max_kl=float("inf"), n_policy=N_POLICY,
                                      n_value=N_VALUE)
        kind, what = "port", "torch-CPU port of the reference (oracle/torch_port.py; baseline/_ref is not installed)"
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        step_fn()
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    best = float(np.min(times))
    return dict(value=n / best, unit="transitions/s", cores=int(threads), kind=kind, host_cpus=os.cpu_count(),
                numa0_cpus=len(cpus), mean_value=n / float(np.mean(times)),
                sample=f"{n_envs} envs x {horizon} steps = {n} transitions, {N_POLICY}+{N_VALUE} full-batch steps, "
                       f"{what}; {threads} threads pinned to NUMA node 0; best of {len(times)} run(s) after {warmup} "
                       f"warm-up (BASELINE.md section 3)"), best


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cb, sec = cpu_reference_run(args.steps, args.warmup)
    line = {"impl": "reference", "metric": "ppo_update_transitions_per_sec", "value": cb["value"],
            "unit": "transitions/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(args.gpus), "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": "transitions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def workload_config(n_gpus, envs=1024, horizon=1000):
    return {"workload": f"PPO synthetic HalfCheetah-shaped obs({OBS}) act({ACT}), {envs} envs x {horizon} steps per GPU"
                        f" ({envs * n_gpus} envs total), MLP(64,64) Gaussian policy + value, {N_POLICY}+{N_VALUE} "
                        f"full-batch Adam steps, max_kl=inf",
            "envs_per_gpu": envs, "horizon": horizon, "parallelism": f"dp{n_gpus} (shard by environment)",
            "l2": "L2 flushed (256 MiB write) before every timed step"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--envs", type=int, default=1024)
    ap.add_argument("--horizon", type=int, default=1000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the TRPO (config 3) / TD3 (config 4) side measurements")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step of each PPO leg computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the outputs of the GPU arm")
        return run_reference_arm(args)

    import torch
    import torch.distributed as dist
    from rl_replicas_b200 import _lib
    from rl_replicas_b200 import synthetic

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    distributed = world > 1
    if distributed:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    assert world == args.gpus or not distributed, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    lib = _lib.load()
    pk = peaks()

    pl, vl, log_std = make_nets()
    E, T = args.envs, args.horizon
    n_local = E * T
    batch = make_batch(E, T, pl, seed=rank)
    # pinned host staging for the e2e leg
    pinned = {}
    for k, v in batch.items():
        t = torch.from_numpy(np.ascontiguousarray(v if k != "ep_done" else v.astype(np.uint8)))
        pinned[k] = t.pin_memory().numpy()
    h2d = sum(pinned[k].nbytes for k in pinned) + 2 * (5702 * 4 * 3 + 5377 * 4 * 3) // 2 + 5702 * 4 + ACT * 4
    d2h = (5702 + 5377) * 4 * 3 + 13 * 8

    ppo = synthetic.onpolicy_learner("ppo", pl, vl, log_std, num_policy_gradients=N_POLICY, num_value_gradients=N_VALUE,
                                     max_kl_divergence=float("inf"), distributed=distributed)
    # the rollout store a sampler fills (SURVEY 8f-1), in pinned host memory: what the public train() is handed
    from rl_replicas_b200.experience import PackedExperience
    store = PackedExperience(n_local, OBS, ACT, pinned=True)
    off = batch["ep_offsets"]
    for ep in range(E):
        a, z = int(off[ep]), int(off[ep + 1])
        done_col = np.zeros(z - a, dtype=bool)
        done_col[-1] = bool(batch["ep_done"][ep])
        store.append_episode(batch["obs"][a:z], batch["act"][a:z], batch["rew"][a:z], done_col, batch["last_obs"][ep])
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def barrier():
        if distributed:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        total = 0.0
        for _ in range(steps):
            flush.fill_(1)  # L2 flush, outside the timed events
            torch.cuda.synchronize()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            fn()
            ev1.record()
            torch.cuda.synchronize()
            total += ev0.elapsed_time(ev1)
        barrier()
        t = torch.tensor([total], dtype=torch.float64, device="cuda")
        if distributed:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / steps  # ms per step, max over ranks

    # ---------------- e2e: public API with host buffers ----------------
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    l0 = lib.b200rl_launch_count()
    ms_e2e = timed(lambda: ppo.train(store), args.steps, args.warmup)  # the reference's boundary call (ppo.py:139)
    fused_path = int(ppo.last_update_stats.fused)
    launches_per_step = (lib.b200rl_launch_count() - l0) // (args.steps + args.warmup)
    dump = bool(args.dump_outputs) and rank == 0
    outputs = learner_outputs("e2e", ppo) if dump else {}

    # ---------------- value: batch resident in HBM ----------------
    engine = ppo._engine
    hp = ppo._hparams(engine, n_local * world if distributed else 0)
    last = {}

    def device_step():
        last["stats"] = engine.update(hp, "ppo", None, distributed)

    ms_dev = timed(device_step, args.steps, args.warmup)
    if dump:  # read back before the per-stage timings below move the engine's state on
        outputs.update(engine_outputs("update", engine, last["stats"]))
    clocks = sampler.summary() if sampler else None

    # ---------------- kernel-level rooflines (rank 0, N = 1 semantics: per-GPU kernels) ----------------
    def stage_ms(stage, reps):
        engine.run_stage(stage, hp)
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(reps):
            engine.run_stage(stage, hp)
        ev1.record()
        torch.cuda.synchronize()
        return ev0.elapsed_time(ev1) / reps

    engine.run_stage("preamble", hp)
    engine.run_stage("old_logp", hp)
    ms_pack = stage_ms("pack_obs", 10)
    ms_fused = stage_ms("fused_step_kernel", 10)
    ms_pol = stage_ms("policy_grad_kernel", 10)
    ms_val = stage_ms("value_grad_kernel", 10)
    tf_fused = FLOP_FUSED_STEP * n_local / (ms_fused * 1e-3) / 1e12
    ncu = {}
    try:  # dram bytes per launch of the dominant kernel, from the committed ncu --set full capture (tools/ncu_summary.py)
        with open(os.path.join(ROOT, "profiles", "r02_tc3_ncu.json")) as f:
            ncu = json.load(f)
    except Exception:
        pass
    ncu_scan = {}
    try:
        with open(os.path.join(ROOT, "profiles", "r02_scan_ncu.json")) as f:
            ncu_scan = json.load(f)
    except Exception:
        pass
    scan_reps = 20
    engine.run_stage("values", hp)
    ms_scan_pair = stage_ms("scan", scan_reps)
    tf_pol = FLOP_POLICY_STEP * n_local / (ms_pol * 1e-3) / 1e12
    tf_val = FLOP_VALUE_STEP * n_local / (ms_val * 1e-3) / 1e12
    scan_bytes = (8 + 4 + 4 + 4) * n_local  # f64 rewards + values in, adv + ret out
    gbs_scan = scan_bytes / (ms_scan_pair * 1e-3) / 1e9

    # the same scan kernel on a shape whose traffic (1.3 GB) cannot live in the 126 MB L2: the HBM-bandwidth figure
    def scan_large():
        import ctypes as C
        E2, T2 = 65536, 1000
        n2 = E2 * T2
        rew = torch.randn(n2, dtype=torch.float64, device="cuda")
        val = torch.randn(n2, dtype=torch.float32, device="cuda")
        lv = torch.randn(E2, dtype=torch.float32, device="cuda")
        off = torch.arange(E2 + 1, dtype=torch.int64, device="cuda") * T2
        done = (torch.rand(E2, device="cuda") < 0.9).to(torch.uint8)
        adv, ret = torch.empty(n2, dtype=torch.float32, device="cuda"), torch.empty(n2, dtype=torch.float32, device="cuda")
        st = torch.zeros(3, dtype=torch.float64, device="cuda")
        wsb = lib.b200rl_gae_scan_workspace_bytes(n2)
        ws = torch.zeros(wsb, dtype=torch.uint8, device="cuda")
        p = lambda t: C.c_void_p(t.data_ptr())
        strm = int(torch.cuda.current_stream().cuda_stream)

        def go():
            _lib.check(lib.b200rl_gae_scan(p(rew), 1, p(val), p(lv), p(off), p(done), n2, E2, 0.99, 0.97, p(adv), p(ret),
                                           p(st), p(ws), wsb, strm), "gae_scan")
        for _ in range(3):
            go()
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(10):
            go()
        ev1.record()
        torch.cuda.synchronize()
        ms = ev0.elapsed_time(ev1) / 10
        return n2, ms, 20.0 * n2 / (ms * 1e-3) / 1e9

    # ---------------- BASELINE configs 3 and 4 (rank 0 only; reported as extra fields, not the headline) ----------------
    def trpo_config3():
        """TRPO synthetic Ant-shaped obs(27) act(8), 1024 envs x 1000 steps, CG iters 10 (11 FVPs), 80 value steps."""
        rng = np.random.default_rng(1)
        ps, vs = [27, 64, 64, 8], [27, 64, 64, 1]
        mk = lambda sz: [(rng.standard_normal((o, i)).astype(np.float32) / np.sqrt(i), np.zeros(o, np.float32))
                         for i, o in zip(sz[:-1], sz[1:])]
        pl2, vl2 = mk(ps), mk(vs)
        trpo = synthetic.onpolicy_learner("trpo", pl2, vl2, np.full(8, -0.5, np.float32), num_value_gradients=N_VALUE)
        b = synthetic.fixed_batch(E, T, 27, 8, seed=9, frac_not_done=0.1,
                                  mean_fn=lambda o: synthetic.numpy_mlp(pl2, o))
        # e2e: the public TRPO.train on the rollout store a sampler fills, in pinned host memory (as the PPO e2e leg)
        from rl_replicas_b200.experience import PackedExperience
        store3 = PackedExperience(E * T, 27, 8, pinned=True)
        off3 = b["ep_offsets"]
        for ep in range(E):
            a3, z3 = int(off3[ep]), int(off3[ep + 1])
            dcol = np.zeros(z3 - a3, dtype=bool)
            dcol[-1] = bool(b["ep_done"][ep])
            store3.append_episode(b["obs"][a3:z3], b["act"][a3:z3], b["rew"][a3:z3], dcol, b["last_obs"][ep])
        for _ in range(2):
            trpo.train(store3)
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ms_e2e = []
        for _ in range(3):
            ev0.record()
            trpo.train(store3)
            ev1.record()
            torch.cuda.synchronize()
            ms_e2e.append(ev0.elapsed_time(ev1))
        ms_update = float(np.median(ms_e2e))
        eng = trpo._engine
        hp3 = trpo._hparams(eng, 0)
        # the update alone, batch resident in HBM (what `value` is for PPO): b200rl_trpo_update on the loaded batch
        cg_kw = trpo.policy.optimizer.hyper_parameters()
        eng.trpo_update(hp3, **cg_kw)
        torch.cuda.synchronize()
        ms_res = []
        for _ in range(3):
            ev0.record()
            eng.trpo_update(hp3, **cg_kw)
            ev1.record()
            torch.cuda.synchronize()
            ms_res.append(ev0.elapsed_time(ev1))
        ms_resident = float(np.median(ms_res))
        eng.run_stage("fvp", hp3)
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(10):
            eng.run_stage("fvp", hp3)
        ev1.record()
        torch.cuda.synchronize()
        ms_fvp = ev0.elapsed_time(ev1) / 10
        flop_fvp = 2 * 6336 * 2 + 2 * (6336 + 4608) + 2 * (6336 + 4608)  # tangent fwd (2 products/layer) + fwd + bwd
        ts = trpo.last_trpo_stats
        return {"workload": "TRPO synthetic Ant-shaped obs(27) act(8), 1024 envs x 1000 steps, 10 CG iterations",
                "ms_per_update": ms_resident, "transitions_per_s": E * T / (ms_resident * 1e-3),
                "ms_per_update_e2e": ms_update, "transitions_per_s_e2e": E * T / (ms_update * 1e-3),
                "e2e_note": "TRPO.train(PackedExperience) in pinned host memory: the 156 MB host-to-device copy is inside",
                "ms_per_fvp": ms_fvp, "fvp_per_s": 1e3 / ms_fvp, "fvp_launches": int(ts.fvp_launches),
                "fvp_tflops_fp32": flop_fvp * E * T / (ms_fvp * 1e-3) / 1e12,
                "accepted_ratio_index": int(ts.accepted_index), "rejected": int(ts.rejected), "kl": ts.kl,
                "kernel": "mlp_tc_fvp_kernel (tcgen05 fp16x2: forward + tangents + metric + backward, fp32 re-run predicated behind it)"}

    def td3_config4():
        """TD3 synthetic Hopper-shaped replay (obs 11, act 3), minibatch 256, 256-256 nets, 50 train steps per call."""
        rng = np.random.default_rng(2)
        H = 256
        mk = lambda sz: [(rng.standard_normal((o, i)).astype(np.float32) / np.sqrt(i), np.zeros(o, np.float32))
                         for i, o in zip(sz[:-1], sz[1:])]
        PSz, QSz = [11, H, H, 3], [14, H, H, 1]
        algo, rb = synthetic.offpolicy_learner(True, mk(PSz), [mk(QSz), mk(QSz)])
        n_rb = 1_000_000  # BASELINE config 4: a full 1 M-transition replay, device-resident (108 MB of HBM)
        from rl_replicas_b200.experience import PackedExperience
        obs_rb = rng.standard_normal((n_rb + 1, 11)).astype(np.float32)
        store = PackedExperience(n_rb, 11, 3)
        L = 1000
        for ep in range(n_rb // L):
            a = ep * L
            d = np.zeros(L, dtype=bool)
            d[-1] = True
            store.append_episode(obs_rb[a:a + L], rng.uniform(-1, 1, (L, 3)).astype(np.float32), rng.standard_normal(L), d,
                                 obs_rb[a + L])
        rb.add_experience(store)
        S4, B4 = 50, 256
        algo.train(rb, S4, B4)
        reps = 5
        calls = []
        for _ in range(12):
            t0 = time.perf_counter()
            algo.train(rb, S4, B4)  # returns after the read-back of the logged values: synchronous
            calls.append((time.perf_counter() - t0) * 1e3)
        ms_call = float(np.median(calls))
        # device part only: replay the last staged minibatches through the engine
        eng = algo._engine
        mbs = [rb.sample_minibatch(B4) for _ in range(S4)]
        st = lambda k: np.stack([np.asarray(m[k]) for m in mbs]).astype(np.float32)
        noise = torch.stack([torch.randn(B4, 3) for _ in range(S4)]).numpy()
        hp4 = algo._hparams(True, 2)
        args4 = (hp4, st("observations"), st("actions"), st("rewards"), st("next_observations"), st("dones"), noise)
        eng.train(*args4)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            eng.train(*args4)
        ms_dev = (time.perf_counter() - t0) * 1e3 / reps
        return {"workload": "TD3 synthetic Hopper-shaped (obs 11, act 3), minibatch 256, MLP(256,256), 50 train steps/call, "
                            "replay 1 M transitions (device-resident columns)",
                "ms_per_train_call_e2e": ms_call, "train_steps_per_s_e2e": S4 / (ms_call * 1e-3),
                "ms_per_train_call_e2e_mean": float(np.mean(calls)), "ms_per_train_call_e2e_max": float(np.max(calls)),
                "transitions_per_s_e2e": S4 * B4 / (ms_call * 1e-3),
                "ms_per_train_call_engine": ms_dev, "train_steps_per_s_engine": S4 / (ms_dev * 1e-3),
                "note": "e2e = TD3.train(replay_buffer, 50, 256): host index draws with the reference's numpy stream, "
                        "device-resident replay columns gathered on the GPU, CUDA-graph replay of the 50-step loop, "
                        "parameters / Adam state synchronised back to the host modules; engine = host-staged "
                        "minibatches: one upload + graph + one read-back"}

    if rank == 0:
        n_big, ms_big, gbs_big = scan_large()
        extras = {}
        if world == 1 and not args.no_extras:
            try:
                extras["config3_trpo"] = trpo_config3()
                extras["config4_td3"] = td3_config4()
            except Exception as exc:  # extras must never break the headline line
                extras["error"] = repr(exc)
    if rank == 0:
        total_transitions = n_local * world
        value = total_transitions / (ms_dev * 1e-3)
        e2e = total_transitions / (ms_e2e * 1e-3)
        line = {
            "metric": "ppo_update_transitions_per_sec", "value": value, "unit": "transitions/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(world, E, T),
            "e2e": {"value": e2e, "unit": "transitions/s", "ms_per_step": ms_e2e, "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h)},
            "dtype_note": "fp32 semantics (1e-5 parity vs the float32 reference); tensor-core products are 3 fp16 MMAs "
                          "on two-way fp16 splits with fp32 accumulation, range-checked (a trip redoes the update on "
                          "the wide-range kernels)",
            "tc_wide_range_reruns": int(_lib.load().b200rl_tc_fallback_count()),
            "gpu_launches": int(launches_per_step * args.steps),
            "gpu_launches_per_step": int(launches_per_step),
            "fused_step_path": fused_path,
            "roofline": {"kernel": "mlp_tc3_kernel (tcgen05 fp16x2: policy fwd + PPO-clip loss + bwd AND value fwd + MSE + "
                                   "bwd over the same 128-row tile, one launch per PPO iteration; observations packed "
                                   "once per update and staged by cp.async.bulk)",
                         "bound": "tensor", "achieved": tf_fused, "peak": pk["tf_sust"], "unit": "TFLOP/s",
                         "frac": tf_fused / pk["tf_sust"],
                         "traffic": ncu.get("dram_bytes_per_launch") if (E, T) == (1024, 1000) else None,
                         "traffic_note": "dram__bytes_read.sum + dram__bytes_write.sum per launch of one ncu --set full "
                                         "capture at this shape (profiles/r02_tc3_ncu.json); algorithmic: 104 B per row "
                                         "of reference data (fp32 obs 68 + act 24 + adv 4 + old log-prob 4 + return 4) "
                                         "= 106.5 MB; the kernel reads the packed fp16-pair observations (128 B per row) "
                                         "instead of the fp32 ones: 164 B per row = 167.9 MB",
                         "ncu": {k: ncu.get(k) for k in ("issue_active_pct", "tensor_pipe_active_pct", "duration_us",
                                                         "warp_instructions", "registers", "source")},
                         "note": f"fp32-equivalent algorithmic FLOPs ({FLOP_FUSED_STEP}/row: policy {FLOP_POLICY_STEP} + "
                                 f"value {FLOP_VALUE_STEP}) over the CUDA-event launch time; peak = 16-bit dense sustained "
                                 f"GEMM ({pk['src']}); the kernel executes 3 fp16 MMAs per logical fp32 product (2 for "
                                 f"weight gradients), so 100 % of this roofline is not reachable at fp32-grade accuracy",
                         "ms_per_launch": ms_fused},
            "pack_obs": {"ms_per_launch": ms_pack, "note": "once per update: fp32 observations -> packed fp16-pair tiles"},
            "roofline_policy_kernel": {"kernel": "mlp_tc2_kernel<true> (the two-loop path / VPG / TRPO surrogate)",
                                       "bound": "tensor", "achieved": tf_pol, "peak": pk["tf_sust"], "unit": "TFLOP/s",
                                       "frac": tf_pol / pk["tf_sust"], "ms_per_launch": ms_pol},
            "roofline_value_kernel": {"bound": "tensor", "achieved": tf_val, "peak": pk["tf_sust"], "unit": "TFLOP/s",
                                      "frac": tf_val / pk["tf_sust"], "ms_per_launch": ms_val},
            "roofline_scan": {"kernel": "gae_scan_episode_kernel<double> (single launch: scan + statistics)", "bound": "hbm", "achieved": gbs_scan,
                              "peak": pk["hbm"], "unit": "GB/s", "frac": gbs_scan / pk["hbm"], "traffic": None,
                              "bytes_per_transition": 20, "ms_per_launch": ms_scan_pair,
                              "note": "16.4 MB problem: launch-latency bound at this size (SURVEY 7.3-3)"},
            "roofline_scan_large": {"kernel": "gae_scan_episode_kernel<double>", "bound": "hbm", "achieved": gbs_big,
                                    "peak": pk["hbm"], "unit": "GB/s", "frac": gbs_big / pk["hbm"],
                                    "traffic": ncu_scan.get("dram_bytes_per_launch"),
                                    "traffic_note": "dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full "
                                                    "capture at this shape (profiles/r02_scan_ncu.json; algorithmic "
                                                    "1.311 GB, the last written lines are still in L2 when it ends)",
                                    "transitions": n_big, "bytes_per_transition": 20, "ms_per_launch": ms_big,
                                    "note": "65536 episodes x 1000 steps: 1.31 GB of algorithmic traffic (> L2)"},
            "update_flops_per_transition": FLOP_PER_TRANSITION,
            "update_tflops_fp32_equiv": FLOP_PER_TRANSITION * total_transitions / (ms_dev * 1e-3) / 1e12,
            "clocks": clocks,
            "other_configs": extras,
        }
        if not args.no_cpu_baseline and world == 1:
            cb, _ = cpu_reference_run(2, 1)
            line["cpu_baseline"] = cb
        if dump:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line))
    if distributed:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
