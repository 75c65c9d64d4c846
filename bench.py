#!/usr/bin/env python
"""bench.py — throughput of the fused rollout path (BASELINE.json metric: instance-steps/s and rollouts/s,
TSP/VRP/IRP-50 greedy, at 1/2/4/8 B200).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--kind tsp] [--nodes 50] [--batch B]
                    [--dump-outputs DIR]

One "step" = one full greedy rollout (encoder forward + every decode step + every environment transition) over one
batch of synthetic uniform instances; every timed GPU workload runs K steps (the cpu_baseline leg times one step of its
bounded CPU sample).  Rank 0 prints ONE JSON line.  See DESIGN.md §6.

  --dump-outputs DIR   after the timed steps, rank 0 writes what the headline workload computed in its last step as
             DIR/<name>.npy (float32 / float64): costs, log-probs, action tapes and embeddings of a fixed sample of
             instances for a rollout; rewards, log-probs, loss and the updated weights for --mode train.  The instances
             and weights follow from --seed, so two builds run with the same arguments can be compared array by array:
             a greedy rollout repeats bit for bit; a train step does not (float atomics in the backward perturb the
             warm-up updates, and the sampled rollouts follow), so its arrays agree to rounding and in distribution.

  value / ms_per_step / roofline / e2e / cpu_baseline   the HEADLINE workload: greedy TSP-50, 65,536 instances per GPU
      value      whole-job instance-steps/s with the instances already resident in HBM (Philox on device)
      e2e        the same through the public API with HOST buffers: pinned host arrays -> TSPEnv.from_arrays ->
                 agent.evaluate(env) -> costs back on the host, copies inside the timed region
      roofline   the decode loop: algorithmic bytes (512*N+100 per instance-step, SURVEY §8d) / the CUDA-event time of
                 the decode launches (on their launch stream), against the measured HBM copy bandwidth
      cpu_baseline   the reference's CPU implementation on a bounded sample (see --impl reference)
  workloads  the other configurations the metric and BASELINE.json name, each device-timed the same way with its own
             roofline and clocks: greedy VRP-50 and IRP-50 (65,536 per GPU), the C4 REINFORCE train step (TSP-50 x 65,536:
             sampled rollout + sampled baseline rollout + backward + Adam; under torchrun with the NCCL gradient
             all-reduce, timed separately) and C5 greedy VRP-100 x 131,072 per GPU.  `--no-extras` skips them.

  --impl reference   the reference's own CPU implementation on the host cores, all threads: the UNMODIFIED reference
             (oracle/_ref, a git-ignored copy of the reference's agents/ + gym_vrp/ made by __graft_entry__.build() where
             /root/reference exists; kind "reference") at its own batch size 256, else the oracle port (kind "port").
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
REF_DIR = os.path.join(ROOT, "oracle", "_ref")

import numpy as np  # noqa: E402
import torch  # noqa: E402

KINDS = ("tsp", "vrp", "irp")


def _use_product_paths():
    for p in (os.path.join(ROOT, "vrp-gym_b200"), ROOT):
        if p not in sys.path:
            sys.path.insert(0, p)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--kind", default="tsp", choices=KINDS)
    ap.add_argument("--nodes", type=int, default=50)
    ap.add_argument("--batch", type=int, default=65536, help="instances per GPU (weak scaling)")
    ap.add_argument("--coupling", type=int, default=-1, help="glimpse-mask coupling group; -1 = whole per-GPU batch")
    ap.add_argument("--cpu-batch", type=int, default=0, help="instances in the bounded CPU sample (0: 256 for the "
                                                               "unmodified reference, 4096 for the oracle port)")
    ap.add_argument("--cpu-impl", default="auto", choices=["auto", "reference", "port"])
    ap.add_argument("--gemm-path", type=int, default=0, help="0 tcgen05 f16-split (production), 1 fp32 SIMT cross-check")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="headline workload only")
    ap.add_argument("--no-split", action="store_true",
                    help="keep every decode step inside the persistent kernel (A/B against the split-step launches)")
    ap.add_argument("--seed", type=int, default=69)
    ap.add_argument("--mode", default="rollout", choices=["rollout", "train"],
                    help="headline = greedy rollout (default) or one REINFORCE step (BASELINE.json configs[3])")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the headline workload computed in its last timed step to DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


def _sample(n, k):
    """A fixed sorted sample of k of the indices 0..n-1 (all of them when n <= k), the same in every run."""
    if n <= k:
        return np.arange(n)
    return np.sort(np.random.RandomState(0).choice(n, k, replace=False))


def _to_host(t, rows=None):
    t = t.detach()
    if rows is not None:
        t = t[torch.as_tensor(rows, device=t.device)]
    t = t.cpu()
    return t.numpy().astype(np.float64 if t.dtype == torch.float64 else np.float32)


def write_outputs(d, arrays):
    """--dump-outputs: one float32/float64 .npy per array (well under 64 MB in all, see the two dump sites)."""
    os.makedirs(d, exist_ok=True)
    for name, arr in arrays.items():
        np.save(os.path.join(d, name + ".npy"), arr)


# ------------------------------------------------------------------------------------------------ CPU arms
def cpu_port_rate(kind, N, B, seed, steps=1):
    """Greedy rollout of the oracle port on host cores.  Returns (instance-steps/s, seconds per step, threads)."""
    _use_product_paths()
    from agents import IRPAgent, TSPAgent, VRPAgent
    from oracle import policy_oracle as po
    from oracle.env_oracle import EnvOracle

    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    rs = np.random.RandomState(seed)
    xy = rs.rand(B, N, 2)
    depot = rs.randint(0, N, size=B)
    C = 0.2449 * N + 26.12
    demand = rs.uniform(1, 10, size=(B, N)) / C
    demand[np.arange(B), depot] = 0
    agent = {"tsp": TSPAgent, "vrp": VRPAgent, "irp": IRPAgent}[kind](seed=seed)
    sd = {k: v.detach().float().cpu() for k, v in agent.model.state_dict().items()}
    total_steps, t0 = 0, time.perf_counter()
    with torch.no_grad():
        for _ in range(steps):
            env = EnvOracle(kind, xy, depot, demand)
            po.rollout(sd, env, greedy=True)
            total_steps += env.step_count * B
    dt = time.perf_counter() - t0
    return total_steps / dt, dt / steps, threads


def cpu_reference_rate(kind, N, B, seed, steps=1, warmup=0):
    """The UNMODIFIED reference (oracle/_ref + the two render-only stub modules): Env(N, B) -> Agent(seed).evaluate(env),
    the call reproduction.py:47 makes; fresh instances per step through env.reset() outside the timed region.
    Must run in a process that has not imported this repo's `agents` / `gym_vrp` packages (same module names)."""
    assert "agents" not in sys.modules and "gym_vrp" not in sys.modules
    sys.path[:0] = [os.path.join(ROOT, "oracle", "stubs"), REF_DIR]
    import logging

    logging.disable(logging.CRITICAL)
    from agents import IRPAgent, TSPAgent, VRPAgent  # the reference's
    from gym_vrp.envs import IRPEnv, TSPEnv, VRPEnv

    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    env = {"tsp": TSPEnv, "vrp": VRPEnv, "irp": IRPEnv}[kind](num_nodes=N, batch_size=B, num_draw=1, seed=seed)
    agent = {"tsp": TSPAgent, "vrp": VRPAgent, "irp": IRPAgent}[kind](seed=seed)
    total_steps, dt = 0, 0.0
    for i in range(warmup + steps):
        if i:
            env.reset()
        env.step_count = 0
        t0 = time.perf_counter()
        agent.evaluate(env)
        if i >= warmup:
            dt += time.perf_counter() - t0
            total_steps += env.step_count * B
    return total_steps / dt, dt / steps, threads


def pick_cpu_impl(a):
    have_ref = os.path.isdir(os.path.join(REF_DIR, "agents")) and os.path.isdir(os.path.join(REF_DIR, "gym_vrp"))
    if a.cpu_impl == "reference" and not have_ref:
        raise SystemExit("oracle/_ref is missing: run __graft_entry__.build() where /root/reference exists")
    impl = "reference" if (have_ref and a.cpu_impl != "port") else "port"
    batch = a.cpu_batch or (256 if impl == "reference" else 4096)
    return impl, batch


def run_reference_arm(a):
    """--impl reference: the reference's CPU implementation on the host cores, a bounded sample per step."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    impl, B = pick_cpu_impl(a)
    if impl == "reference":
        rate, sec, threads = cpu_reference_rate(a.kind, a.nodes, B, a.seed, steps=a.steps, warmup=min(a.warmup, 1))
        what = (f"greedy {a.kind.upper()}-{a.nodes} rollout of {B} instances per step by the UNMODIFIED reference "
                f"(oracle/_ref: networkx/numpy env + torch-CPU agent.evaluate, reproduction.py:47; its throughput is flat in the "
                f"batch size — per-instance Python loops — and it cannot hold 65,536 instances: 372 KB per graph)")
    else:
        for _ in range(min(a.warmup, 1)):
            cpu_port_rate(a.kind, a.nodes, 64, a.seed)
        rate, sec, threads = cpu_port_rate(a.kind, a.nodes, B, a.seed, steps=a.steps)
        what = (f"greedy {a.kind.upper()}-{a.nodes} rollout of {B} instances per step (oracle port of the reference: "
                f"vectorised numpy env + torch-CPU policy)")
    line = {
        "impl": "reference", "metric": "instance_steps_per_sec", "value": rate, "unit": "instance-steps/s",
        "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"greedy {a.kind.upper()}-{a.nodes} rollout, CPU sample batch {B}"},
        "cpu_baseline": {"value": rate, "unit": "instance-steps/s", "cores": threads, "kind": impl, "sample": what},
        "e2e": {"value": rate, "unit": "instance-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def cpu_baseline_subprocess(a):
    """The cpu_baseline leg of our own arm: the reference arm in a child process (the reference's packages share their
    names with this repo's), one bounded step."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "1", "--warmup", "0", "--kind", a.kind,
           "--nodes", str(a.nodes), "--seed", str(a.seed), "--cpu-impl", a.cpu_impl, "--cpu-batch", str(a.cpu_batch)]
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE")}
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env)
    for ln in reversed(out.stdout.strip().splitlines()):
        if ln.startswith("{"):
            return json.loads(ln)["cpu_baseline"]
    return {"value": None, "unit": "instance-steps/s", "cores": os.cpu_count(), "kind": "unavailable",
            "sample": "CPU arm failed: " + out.stderr[-300:]}


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def window(self, t0, t1):
        """Median SM clock and throttle reasons sampled between two perf_counter stamps (the timed region)."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        sm, smax, reasons = [], None, set()
        for ts, line in list(self.rows):
            if not (t0 <= ts <= t1 + 0.1):
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[0]))
                smax = float(f[1])
            except Exception:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}

    def close(self):
        if self.proc is not None:
            self.proc.terminate()


class Ctx:
    """Per-process bench context: device, ranks, collectives, clocks, measured peaks."""

    def __init__(self, a):
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist

            self.dist = dist
            dist.init_process_group("nccl", device_id=self.dev)
        self.clocks = ClockSampler(self.local) if self.rank == 0 else None
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            pk = json.load(open(peaks_path))
            self.hbm, self.hbm_src = float(pk["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (copy, burst)"
        else:
            self.hbm, self.hbm_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"

    def barrier(self):
        torch.cuda.synchronize()
        if self.dist is not None:
            self.dist.barrier()
        torch.cuda.synchronize()

    def reduce(self, max_vals, sum_vals):
        t = torch.tensor(list(max_vals), device=self.dev, dtype=torch.float64)
        s = torch.tensor(list(sum_vals), device=self.dev, dtype=torch.float64)
        if self.dist is not None:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            self.dist.all_reduce(s, op=self.dist.ReduceOp.SUM)
        return [float(x) for x in t.tolist()], [float(x) for x in s.tolist()]


def _classes(kind):
    from agents import IRPAgent, TSPAgent, VRPAgent
    from gym_vrp.envs import IRPEnv, TSPEnv, VRPEnv

    return ({"tsp": TSPEnv, "vrp": VRPEnv, "irp": IRPEnv}[kind], {"tsp": TSPAgent, "vrp": VRPAgent, "irp": IRPAgent}[kind])


def _traffic(kind, N, B):
    """DRAM bytes of the decode launches of one rollout, from the committed per-round ncu capture of this exact
    configuration (profiles/rollout_traffic_<kind><N>_b<B>.json names the ncu log it was summed from), else null."""
    tpath = os.path.join(ROOT, "profiles", f"rollout_traffic_{kind}{N}_b{B}.json")
    if os.path.exists(tpath):
        return float(json.load(open(tpath))["dram_bytes_per_launch"])
    return None


# ------------------------------------------------------------------------------------------------ greedy rollout
def rollout_workload(a, ctx, kind, N, B, steps, warmup, with_e2e, dump=None):
    import vrpx
    from agents.graph_encoder import run_encoder

    Env, Agent = _classes(kind)
    dev = ctx.dev
    agent = Agent(seed=a.seed)  # identical seed-initialised weights on every rank (no checkpoint in the reference tree)
    model = agent.model
    model.eval()
    model.encoder.gemm_path = a.gemm_path
    model.coupling = None if a.coupling < 0 else a.coupling
    env = Env(N, B, 0, seed=a.seed, instance_rng="philox", instance_offset=ctx.rank * B)  # shard = own reference batch
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def one_step(events=None, keep_emb=False):
        env.restart_episode()
        if events is not None:
            events[0].record()
        with torch.no_grad():
            h = run_encoder(model.encoder, env=env, depot=env._depot if model._USES_DEPOT_EMBED else None,
                            gemm_path=a.gemm_path)
            if events is not None:
                events[1].record()
            out = model.decoder.rollout_episode(env, h, greedy=True, coupling=model.coupling)
            if events is not None:
                events[2].record()
        if keep_emb:  # only the dumped step: an earlier step's h would stay alive during the next one
            out["emb"] = h
        return out

    for _ in range(max(warmup, 3)):
        out = one_step()
    T = out["steps"]
    ctx.barrier()
    launches0 = vrpx.launch_count()
    per_step_events = [[ev(), ev(), ev()] for _ in range(steps)]
    e0, e1 = ev(), ev()
    w0 = time.perf_counter()
    e0.record()
    total_inst_steps, useful_steps, kernel_ms = 0, 0.0, []
    if a.no_split:
        vrpx.lib().vrpx_debug_rollout_split(0)
    vrpx.lib().vrpx_debug_rollout_timing(1)  # CUDA events around the decode launches alone, on their launch stream
    for i in range(steps):
        out = one_step(per_step_events[i], keep_emb=dump is not None and i == steps - 1)
        total_inst_steps += out["steps"] * B  # includes the .item() sync on the step count
        kernel_ms.append(float(vrpx.lib().vrpx_debug_rollout_kernel_ms()))  # the step is already synchronised
    e1.record()
    ctx.barrier()
    w1 = time.perf_counter()
    elapsed_ms = e0.elapsed_time(e1)
    launches = vrpx.launch_count() - launches0
    enc_ms = float(np.mean([e[0].elapsed_time(e[1]) for e in per_step_events]))
    roll_ms = float(np.mean([e[1].elapsed_time(e[2]) for e in per_step_events]))
    mean_cost = float(out["cost"].mean().item())
    vrpx.lib().vrpx_debug_rollout_timing(0)
    kern_ms = float(np.mean(kernel_ms))
    if dump is not None:
        # per-instance results of up to 131,072 instances, the action tapes of 8,192 and the embeddings of 256:
        # at most 0.5 + 0.5 + 8.4 + 16.8 MB (N <= 128, at most 2N - 1 steps)
        inst, tape_rows, emb_rows = _sample(B, 1 << 17), _sample(B, 8192), _sample(B, 256)
        dump.update(cost=_to_host(out["cost"], inst), logp=_to_host(out["logp"], inst),
                    tape=_to_host(out["tape"].t(), tape_rows).T.copy(), emb=_to_host(out["emb"], emb_rows),
                    steps=np.array([out["steps"]], dtype=np.float64), instances=inst.astype(np.float64),
                    tape_instances=tape_rows.astype(np.float64), emb_instances=emb_rows.astype(np.float64))

    e2e_ms, e2e_inst_steps, n_e2e, h2d, d2h = 0.0, 0.0, 0, 0, 0
    if with_e2e:
        # public API with host buffers (pinned H2D of the instances, D2H of the costs inside the timed region)
        s = env.sampler
        xy_h = torch.from_numpy(s.get_graph_positions()).pin_memory()
        dep_h = torch.from_numpy(s.get_depots()[:, 0].astype(np.int64)).pin_memory()
        dem_h = torch.from_numpy(s.get_demands()[:, :, 0]).pin_memory()

        def e2e_step():
            e = Env.from_arrays(xy_h.numpy(), dep_h.numpy(), dem_h.numpy() if kind != "tsp" else None, device=dev)
            loss = agent.evaluate(e)
            return loss.cpu(), e.step_count

        for _ in range(2):
            e2e_step()
        ctx.barrier()
        f0, f1 = ev(), ev()
        f0.record()
        n_e2e = max(1, steps)
        for _ in range(n_e2e):
            loss_h, sc = e2e_step()
            e2e_inst_steps += sc * B
        f1.record()
        ctx.barrier()
        e2e_ms = f0.elapsed_time(f1)
        h2d = int(xy_h.numel() * 8 + dep_h.numel() * 4 + (dem_h.numel() * 8 if kind != "tsp" else 0))
        d2h = int(B * 4)

    (elapsed_ms, e2e_ms, roll_ms, enc_ms, kern_ms), (total_inst_steps, e2e_inst_steps) = ctx.reduce(
        [elapsed_ms, e2e_ms, roll_ms, enc_ms, kern_ms], [float(total_inst_steps), float(e2e_inst_steps)])
    res = None
    if ctx.rank == 0:
        bytes_per_step = 512.0 * N + 100.0                # per instance-step (SURVEY §8d, DESIGN.md §3.3)
        alg_bytes = bytes_per_step * B * T                # per rollout = per "launch" of the decode loop
        achieved = alg_bytes / (kern_ms * 1e-3) / 1e9
        value = total_inst_steps / (elapsed_ms * 1e-3)
        res = {
            "value": value, "unit": "instance-steps/s", "ms_per_step": elapsed_ms / steps, "steps": steps,
            "workload": f"greedy {kind.upper()}-{N} rollout (encoder + {T} fused decode/env steps, idle steps of finished "
                        f"instances included like the reference's loop), {B} Philox-uniform instances per GPU, "
                        f"seed-initialised {kind.upper()}Agent weights",
            "instances_per_gpu": B, "nodes": N, "steps_per_rollout": T,
            "coupling_group": B if model.coupling is None else model.coupling,
            "rollouts_per_sec": value / T, "mean_cost": mean_cost,
            "breakdown_ms": {"encoder": enc_ms, "score_tables": roll_ms - kern_ms, "decode_loop": kern_ms},
            "clocks": ctx.clocks.window(w0, w1), "gpu_launches": int(launches),
            "roofline": {"bound": "hbm",
                         "kernel": ("k_rollout (persistent decoder+env, every step)" if a.no_split else
                                    "decode loop: every launch between the score-table prologue and the end of the episode"),
                         "achieved": achieved, "peak": ctx.hbm, "unit": "GB/s", "frac": achieved / ctx.hbm,
                         "traffic": _traffic(kind, N, B), "peak_source": ctx.hbm_src,
                         "algorithmic_bytes_per_launch": alg_bytes, "launch_ms": kern_ms},
        }
        if with_e2e:
            res["e2e"] = {"value": e2e_inst_steps / (e2e_ms * 1e-3), "unit": "instance-steps/s", "h2d_bytes_per_step": h2d,
                          "d2h_bytes_per_step": d2h, "steps": n_e2e}
    del env, agent, model, out
    torch.cuda.empty_cache()
    return res


# ------------------------------------------------------------------------------------------------ train step
def train_workload(a, ctx, kind, N, B, steps, warmup, dump=None):
    """One step = the body of TSPAgent.train's epoch without baseline_update (graph_tsp_agent.py:176-186): reset,
    sampled rollout with grad (train-mode BatchNorm), sampled baseline rollout, REINFORCE loss, backward, gradient
    all-reduce over ranks (NCCL; a no-op on one GPU), Adam."""
    import vrpx

    Env, Agent = _classes(kind)
    agent = Agent(seed=a.seed)
    agent.model.encoder.gemm_path = agent.target_model.encoder.gemm_path = a.gemm_path
    env = Env(N, B, 0, seed=a.seed, instance_rng="philox", instance_offset=ctx.rank * B)
    ev = lambda: torch.cuda.Event(enable_timing=True)
    ar_events = []
    plain_allreduce = agent._allreduce_gradients

    def timed_allreduce():
        x0, x1 = ev(), ev()
        x0.record()
        plain_allreduce()
        x1.record()
        ar_events.append((x0, x1))

    agent._allreduce_gradients = timed_allreduce
    last = {}

    def one():
        agent.model.train()
        loss_m, loss_b, logp = agent.step(env, (False, True))
        adv = (loss_m - loss_b) * -1
        loss = agent.policy_gradient_step(adv, logp)
        last.update(reward=loss_m, baseline_reward=loss_b, logp=logp, loss=loss)
        return env.step_count, float(loss)

    for _ in range(max(warmup, 3)):
        T, loss = one()
    ctx.barrier()
    ar_events.clear()
    l0 = vrpx.launch_count()
    e0, e1 = ev(), ev()
    w0 = time.perf_counter()
    e0.record()
    inst_steps = 0
    for _ in range(steps):
        T, loss = one()
        inst_steps += 2 * T * B
    e1.record()
    ctx.barrier()
    w1 = time.perf_counter()
    ms = e0.elapsed_time(e1)
    ar_ms = sum(x0.elapsed_time(x1) for x0, x1 in ar_events) / steps
    if dump is not None:
        # per-instance rewards and log-probs of up to 131,072 instances (1.5 MB) and the updated weights (4.6 MB)
        inst = _sample(B, 1 << 17)
        dump.update({k: _to_host(last[k], inst) for k in ("reward", "baseline_reward", "logp")})
        dump.update(loss=_to_host(last["loss"].reshape(1)), instances=inst.astype(np.float64))
        dump.update({"param." + k: _to_host(v) for k, v in agent.model.state_dict().items() if v.is_floating_point()})
    (ms, ar_ms), (inst_steps,) = ctx.reduce([ms, ar_ms], [float(inst_steps)])
    res = None
    if ctx.rank == 0:
        # tensor-pipe roofline of the step: 2 encoder forwards + 1 backward (= 2 forwards) of 2*(589,824 N + 768 N^2)
        # FLOP per instance (SURVEY §8d), against the measured sustained dense bf16 rate; the f16 hi/lo split issues 3x
        enc_flop = 4.0 * 2.0 * (589824.0 * N + 768.0 * N * N) * B
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        tpeak = float(json.load(open(peaks_path)).get("bf16_tflops_sustained", 1408.5)) if os.path.exists(peaks_path) else 1408.5
        res = {"value": inst_steps / (ms * 1e-3), "unit": "instance-steps/s (both sampled rollouts counted)",
               "ms_per_step": ms / steps, "steps": steps,
               "workload": f"REINFORCE train step {kind.upper()}-{N}: sampled rollout + sampled baseline rollout + backward "
                           f"+ gradient all-reduce + Adam, {B} instances per GPU",
               "instances_per_gpu": B, "nodes": N, "steps_per_rollout": T, "loss": loss,
               "allreduce_ms_per_step": ar_ms, "allreduce": ("NCCL all-reduce of one flat f32 gradient bucket (1.15 M elements)"
                                                              if ctx.world > 1 else "single GPU: no collective"),
               "clocks": ctx.clocks.window(w0, w1), "gpu_launches": int(vrpx.launch_count() - l0),
               "peak_mem_gb": torch.cuda.max_memory_allocated() / 1e9,
               "roofline": {"bound": "tensor", "kernel": "encoder contractions of the step (2 forwards + backward), useful FLOPs",
                            "achieved": enc_flop / (ms / steps * 1e-3) / 1e12, "peak": tpeak, "unit": "TFLOP/s",
                            "frac": enc_flop / (ms / steps * 1e-3) / 1e12 / tpeak, "traffic": None,
                            "note": "whole-step time in the denominator (rollout decode loops and the decoder backward included)"}}
    del env, agent
    torch.cuda.empty_cache()
    return res


# ------------------------------------------------------------------------------------------------ GPU arm
def main():
    a = parse()
    if a.impl == "reference":
        return run_reference_arm(a)
    _use_product_paths()
    import vrpx  # noqa: F401  (fails loudly when libvrpx.so is missing: no CPU fallback)

    ctx = Ctx(a)
    B, N = a.batch, a.nodes
    dump = {} if (a.dump_outputs and ctx.rank == 0) else None
    if a.mode == "train":
        head = train_workload(a, ctx, a.kind, N, B, a.steps, a.warmup, dump=dump)
        metric = "train_instance_steps_per_sec"
    else:
        head = rollout_workload(a, ctx, a.kind, N, B, a.steps, a.warmup, with_e2e=True, dump=dump)
        metric = "instance_steps_per_sec"
    if dump is not None:
        write_outputs(a.dump_outputs, dump)
    extras = {}
    default_headline = (a.mode, a.kind, N, B) == ("rollout", "tsp", 50, 65536)
    if default_headline and not a.no_extras and not a.no_split:
        extras["vrp50_greedy_b65536"] = rollout_workload(a, ctx, "vrp", 50, 65536, a.steps, 3, with_e2e=False)
        extras["irp50_greedy_b65536"] = rollout_workload(a, ctx, "irp", 50, 65536, a.steps, 3, with_e2e=False)
        extras["c4_train_step_tsp50_b65536"] = train_workload(a, ctx, "tsp", 50, 65536, a.steps, 3)
        extras["c5_vrp100_greedy_b131072"] = rollout_workload(a, ctx, "vrp", 100, 131072, a.steps, 3, with_e2e=False)
    if ctx.rank == 0:
        line = {"metric": metric, "value": head["value"], "unit": "instance-steps/s", "n_gpus": ctx.world,
                "steps": a.steps, "warmup": max(a.warmup, 3), "ms_per_step": head["ms_per_step"], "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None,
                "dtype": ("f32 (tensor-core contractions on f16 hi/lo splits with f32 accumulation, ~fp32 accuracy; env "
                          "f64/bitmask)" if a.gemm_path == 0 else "f32"),
                "data": "synthetic",
                "config": {"workload": head["workload"], "instances_per_gpu": head["instances_per_gpu"], "nodes": head["nodes"],
                           "steps_per_rollout": head["steps_per_rollout"], "coupling_group": head.get("coupling_group"),
                           "decode_loop": ("persistent kernel, every step" if a.no_split else
                                           "split-step launches (glimpse / batched tcgen05 GEMM-B / pointer+env per step), "
                                           "chosen over the single persistent launch by measurement (DESIGN.md §3.3)"),
                           "l2": "inputs larger than L2 (embeddings %.2f GB per GPU re-streamed every decode step)"
                                 % (head["instances_per_gpu"] * head["nodes"] * 512 / 1e9)}}
        for key in ("rollouts_per_sec", "mean_cost", "breakdown_ms", "clocks", "e2e", "gpu_launches", "roofline", "loss",
                    "allreduce_ms_per_step", "allreduce", "peak_mem_gb"):
            if key in head:
                line[key] = head[key]
        if extras:
            line["workloads"] = extras
            line["gpu_launches"] += sum(int(w["gpu_launches"]) for w in extras.values())
        if not a.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_subprocess(a)
        ctx.clocks.close()
        print(json.dumps(line), flush=True)
    if ctx.dist is not None:
        ctx.dist.destroy_process_group()


if __name__ == "__main__":
    main()
