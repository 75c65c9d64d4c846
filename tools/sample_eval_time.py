#!/usr/bin/env python
"""Best-of-K sampling: the shared-embedding path (GraphDecoder.rollout_samples: encoder and score table over B base
instances, decode loop over K·B replicas) against the replicated path a user can build without it (a copy-major env of
K·B instances, the encoder over all of them, then rollout_episode with coupling = B and the same seed and offset).

    python tools/sample_eval_time.py [--nodes 50] [--batch 8192] [--samples 8] [--reps 5] [--big-samples 64] [--out F]

Per timed call (CUDA events on the current stream): encoder ms, rollout-call ms, the decode-loop bracket of
vrpx_debug_rollout_timing, tables_ms = rollout call minus decode loop (score table, weight transposes, env replication
of the shared path), whole-call ms, replica-steps/s and the peak of torch.cuda.max_memory_allocated.  The two paths
alternate in one process; the spread is min / median / max over the repetitions.  Both paths' tapes, costs and
log-probs at the timed size are compared bit for bit (and, if they differ, the K·B-row encoder output against K copies
of the B-row one).  The card's name and power limit are read in the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "vrp-gym_b200"), ROOT]
import torch  # noqa: E402

import vrpx  # noqa: E402
from agents import TSPAgent  # noqa: E402
from agents.graph_encoder import run_encoder  # noqa: E402
from gym_vrp.envs import TSPEnv  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


class Timer:
    def __init__(self):
        self.ev = {}

    def mark(self, name):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        self.ev[name] = e

    def ms(self, a, b):
        return self.ev[a].elapsed_time(self.ev[b])


def run_shared(model, env, K, seed):
    L = vrpx.lib()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    tm = Timer()
    tm.mark("0")
    h = run_encoder(model.encoder, env=env, gemm_path=model.encoder.gemm_path)
    tm.mark("enc")
    out = model.decoder.rollout_samples(env, h, K, seed=seed)   # ends in a synchronise (steps)
    tm.mark("end")
    torch.cuda.synchronize()
    dec = float(L.vrpx_debug_rollout_kernel_ms())
    r = {"encoder_ms": tm.ms("0", "enc"), "rollout_ms": tm.ms("enc", "end"), "decode_loop_ms": dec,
         "whole_ms": tm.ms("0", "end"), "steps": out["steps"], "peak_gib": torch.cuda.max_memory_allocated() / 2 ** 30}
    return r, out, h


def run_replicated(model, env_rep, B, seed):
    L = vrpx.lib()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    tm = Timer()
    tm.mark("0")
    env_rep.restart_episode()
    h = run_encoder(model.encoder, env=env_rep, gemm_path=model.encoder.gemm_path)
    tm.mark("enc")
    out = model.decoder.rollout_episode(env_rep, h, greedy=False, coupling=B, seed=seed, offset=0)
    tm.mark("end")
    torch.cuda.synchronize()
    dec = float(L.vrpx_debug_rollout_kernel_ms())
    r = {"encoder_ms": tm.ms("0", "enc"), "rollout_ms": tm.ms("enc", "end"), "decode_loop_ms": dec,
         "whole_ms": tm.ms("0", "end"), "steps": out["steps"], "peak_gib": torch.cuda.max_memory_allocated() / 2 ** 30}
    return r, out, h


def summary(rows, replicas):
    s = {}
    for key in ("encoder_ms", "rollout_ms", "decode_loop_ms", "whole_ms", "peak_gib"):
        v = [r[key] for r in rows]
        s[key] = {"median": statistics.median(v), "min": min(v), "max": max(v)}
    for r in rows:
        r["tables_ms"] = r["rollout_ms"] - r["decode_loop_ms"]
        r["replica_steps_per_s"] = replicas * r["steps"] / (r["whole_ms"] * 1e-3)
    for key in ("tables_ms", "replica_steps_per_s"):
        v = [r[key] for r in rows]
        s[key] = {"median": statistics.median(v), "min": min(v), "max": max(v)}
    return s


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nodes", type=int, default=50)
    ap.add_argument("--batch", type=int, default=8192)
    ap.add_argument("--samples", type=int, default=8)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--big-samples", type=int, default=64)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    N, B, K = a.nodes, a.batch, a.samples
    vrpx.require_device()
    vrpx.lib().vrpx_debug_rollout_timing(1)
    model = TSPAgent(seed=69).model
    model.eval()
    env = TSPEnv(N, B, 0, seed=69, instance_rng="philox")
    env_rep = TSPEnv(N, K * B, 0, seed=69, instance_rng="philox")
    env_rep._xy.copy_(env._xy.repeat(K, 1, 1))
    env_rep._depot.copy_(env._depot.repeat(K))
    env_rep._demand.copy_(env._demand.repeat(K, 1))
    env_rep.restart_episode()
    seed = 12345
    res = {"card": card(), "nodes": N, "batch": B, "samples": K, "replicas": K * B, "seed": seed,
           "timing": "CUDA events on the current stream; decode loop = vrpx_debug_rollout_timing bracket; "
                     "tables_ms = rollout call - decode loop"}
    with torch.no_grad():
        # warm-up of both shapes, then the bit-for-bit comparison at the timed size
        _, o_s, h_s = run_shared(model, env, K, seed)
        _, o_r, h_r = run_replicated(model, env_rep, B, seed)
        T = o_s["steps"]
        same = {"steps": T == o_r["steps"],
                "tape": torch.equal(o_s["tape"].reshape(T, K * B), o_r["tape"]),
                "cost": torch.equal(o_s["cost"].reshape(-1), o_r["cost"]),
                "logp": torch.equal(o_s["logp"].reshape(-1), o_r["logp"])}
        if not all(same.values()):
            same["embeddings_KB_rows_equal_K_copies"] = torch.equal(h_r, h_s.repeat(K, 1, 1))
        res["outputs_bit_identical"] = same
        del o_s, o_r, h_s, h_r
        shared, repl = [], []
        for _ in range(a.reps):
            shared.append(run_shared(model, env, K, seed)[0])
            repl.append(run_replicated(model, env_rep, B, seed)[0])
        res["shared"] = {"runs": shared, "summary": summary(shared, K * B)}
        res["replicated"] = {"runs": repl, "summary": summary(repl, K * B)}
        del env_rep
        torch.cuda.empty_cache()
        if a.big_samples:
            Kb = a.big_samples
            run_shared(model, env, Kb, seed)
            big = [run_shared(model, env, Kb, seed)[0] for _ in range(max(2, a.reps // 2))]
            res["shared_big_k"] = {"samples": Kb, "replicas": Kb * B, "runs": big, "summary": summary(big, Kb * B)}
    ws = lambda kind, Bb, K_: int(vrpx.lib().vrpx_rollout_samples_workspace_bytes(kind, Bb, K_, N))
    res["s1_gib_computed"] = {"shared": B * N * 8 * N * 4 / 2 ** 30, "replicated": K * B * N * 8 * N * 4 / 2 ** 30}
    res["workspace_gib_computed"] = {"shared": ws(vrpx.TSP, B, K) / 2 ** 30, "replicated": ws(vrpx.TSP, K * B, 1) / 2 ** 30}
    s, r = res["shared"]["summary"], res["replicated"]["summary"]
    res["verdict"] = {"whole_call_faster": s["whole_ms"]["max"] < r["whole_ms"]["min"],
                      "decode_loop_not_slower": s["decode_loop_ms"]["median"] <= r["decode_loop_ms"]["max"]}
    line = json.dumps(res, indent=1)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
