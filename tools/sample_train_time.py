#!/usr/bin/env python
"""Training on K sampled tours per instance: the K-sample train step (the phases of TSPModel.forward_samples and its
backward: train-mode encoder over B base instances, traced rollout_samples over K·B replicas, the baseline model's
rollout_samples, the decoder backward over the replicas, ONE encoder backward over the B instances, Adam) against the
route a user can build without it (today's train step on a copy-major env of K·B instances with coupling B: the
train-mode encoder, the decoder backward and the baseline over all K·B instances).

    python tools/sample_train_time.py [--nodes 50] [--batch 8192] [--samples 8] [--reps 5] [--big-batch 65536] [--out F]

Per step (CUDA events on the current stream): train encoder, sampled rollout, baseline rollout (encoder + rollout of the
target model), decoder backward (vrpx/backward.py decoder_backward incl. its per-episode epilogue and copy sum),
encoder backward, Adam, the whole step, and the peak of torch.cuda.max_memory_allocated.  The two paths alternate in one
process; the spread is min / median / max over the repetitions.  Before any Adam step, the replicated route is run
teacher-forced along the K-sample step's tapes with the same weights wts, and the largest gradient difference (per
tensor, relative to the tensor's largest element, for the tensors above 1e-3 of the model's largest element; the rest
are mathematically zero, e.g. the biases in front of a train-mode BatchNorm) is recorded.  Every step restarts the
episode on the same instances (TSPAgent.step draws fresh ones); the env restart and the baseline env copy are outside
the timed window on both paths.  The card's name and power limit are read in the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys
from copy import deepcopy

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "vrp-gym_b200"), ROOT]
import torch  # noqa: E402

import vrpx  # noqa: E402
from agents import TSPAgent  # noqa: E402
from agents.graph_encoder import run_encoder  # noqa: E402
from gym_vrp.envs import TSPEnv  # noqa: E402
from vrpx import backward as bw  # noqa: E402

PHASES = ("encoder", "rollout", "baseline", "decoder_bwd", "encoder_bwd", "adam")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


class Timer:
    def __init__(self):
        self.ev = []

    def mark(self, name):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        self.ev.append((name, e))

    def phases(self):
        torch.cuda.synchronize()
        r = {n: a.elapsed_time(b) for (_, a), (n, b) in zip(self.ev, self.ev[1:])}
        r["step"] = self.ev[0][1].elapsed_time(self.ev[-1][1])
        return r


def step_samples(agent, env, K, seed, adam=True):
    """One K-sample train step, phase by phase (TSPAgent.step / policy_gradient_step with samples=K)."""
    model, target = agent.model, agent.target_model
    model.train()
    env.restart_episode()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    tm = Timer()
    tm.mark("0")
    h, saved = run_encoder(model.encoder, env=env, gemm_path=model.encoder.gemm_path, save=True)
    tm.mark("encoder")
    out = model.decoder.rollout_samples(env, h, K, seed=seed, save_for_backward=True)
    tm.mark("rollout")
    with torch.no_grad():
        hb = run_encoder(target.encoder, env=env, gemm_path=target.encoder.gemm_path)
        base = target.decoder.rollout_samples(env, hb, K, seed=seed + 1)
    tm.mark("baseline")
    wts = ((base["cost"] - out["cost"]) * -1 / out["cost"].numel()).detach()   # advantage / (K·B), advantage = -(cost_m - cost_b)
    agent.opt.zero_grad()
    dH = bw.decoder_backward(model.decoder, env, h, out, wts.reshape(-1), gemm_path=model.encoder.gemm_path)
    tm.mark("decoder_bwd")
    bw.encoder_backward(model.encoder, env, None, saved, dH, gemm_path=model.encoder.gemm_path)
    tm.mark("encoder_bwd")
    if adam:
        agent.opt.step()
    tm.mark("adam")
    r = tm.phases()
    r["peak_gib"] = torch.cuda.max_memory_allocated() / 2 ** 30
    return r, out, wts


def step_replicated(agent, env_rep, B, seed, tape=None, wts=None, adam=True):
    """Today's train step on the replicated env with coupling B (optionally teacher-forced with given weights)."""
    model, target = agent.model, agent.target_model
    model.train()
    env_rep.restart_episode()
    env_b = deepcopy(env_rep)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    tm = Timer()
    tm.mark("0")
    h, saved = run_encoder(model.encoder, env=env_rep, gemm_path=model.encoder.gemm_path, save=True)
    tm.mark("encoder")
    out = model.decoder.rollout_episode(env_rep, h, greedy=False, tape_in=tape, coupling=B, seed=seed,
                                        save_for_backward=True)
    tm.mark("rollout")
    with torch.no_grad():
        hb = run_encoder(target.encoder, env=env_b, gemm_path=target.encoder.gemm_path)
        base = target.decoder.rollout_episode(env_b, hb, greedy=False, coupling=B, seed=seed + 1)
    tm.mark("baseline")
    if wts is None:
        wts = ((base["cost"] - out["cost"]) * -1 / out["cost"].numel()).detach()
    agent.opt.zero_grad()
    dH = bw.decoder_backward(model.decoder, env_rep, h, out, wts, gemm_path=model.encoder.gemm_path)
    tm.mark("decoder_bwd")
    bw.encoder_backward(model.encoder, env_rep, None, saved, dH, gemm_path=model.encoder.gemm_path)
    tm.mark("encoder_bwd")
    if adam:
        agent.opt.step()
    tm.mark("adam")
    r = tm.phases()
    r["peak_gib"] = torch.cuda.max_memory_allocated() / 2 ** 30
    return r, out


def summary(rows):
    return {k: {"median": statistics.median(r[k] for r in rows), "min": min(r[k] for r in rows),
                "max": max(r[k] for r in rows)} for k in PHASES + ("step", "peak_gib")}


def grads(model):
    return {n: p.grad.detach().clone() for n, p in model.named_parameters() if p.grad is not None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nodes", type=int, default=50)
    ap.add_argument("--batch", type=int, default=8192)
    ap.add_argument("--samples", type=int, default=8)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--big-batch", type=int, default=65536, help="K-sample path only at this base batch (0: skip)")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    N, B, K = a.nodes, a.batch, a.samples
    vrpx.require_device()
    agent = TSPAgent(seed=69)
    env = TSPEnv(N, B, 0, seed=69, instance_rng="philox")
    env_rep = TSPEnv(N, K * B, 0, seed=69, instance_rng="philox")
    env_rep._xy.copy_(env._xy.repeat(K, 1, 1))
    env_rep._depot.copy_(env._depot.repeat(K))
    env_rep._demand.copy_(env._demand.repeat(K, 1))
    env_rep.restart_episode()
    seed = 12345
    res = {"card": card(), "nodes": N, "batch": B, "samples": K, "replicas": K * B, "seed": seed,
           "timing": "CUDA events on the current stream around each phase of one train step; env reset and the "
                     "baseline env copy outside the window"}
    # the same update: the replicated route teacher-forced along the K-sample tapes with the same weights, no Adam step
    _, o_s, wts = step_samples(agent, env, K, seed, adam=False)
    g_s = grads(agent.model)
    T = o_s["steps"]
    tape = o_s["tape"].reshape(T, K * B).cpu().numpy()
    _, o_t = step_replicated(agent, env_rep, B, seed, tape=tape, wts=wts.reshape(-1), adam=False)
    g_r = grads(agent.model)
    gmax = max(float(g.abs().max()) for g in g_r.values())
    err = {n: float((g_s[n] - g_r[n]).abs().max()) for n in g_r}
    rel = {n: err[n] / float(g_r[n].abs().max()) for n in g_r if float(g_r[n].abs().max()) > 1e-3 * gmax}
    worst = max(rel, key=rel.get)
    res["gradient_difference"] = {
        "max_rel_to_tensor_max": rel[worst], "tensor": worst, "max_abs_rel_to_model_max": max(err.values()) / gmax,
        "tensors_compared": len(rel), "tensors_near_zero": len(err) - len(rel),
        "logp_max_abs_diff": float((o_t["logp"] - o_s["logp"].reshape(-1)).abs().max())}
    # sampled tapes of the two routes with the same seed (the encoders' BatchNorm sums differ in order only)
    _, o_r = step_replicated(agent, env_rep, B, seed, adam=False)
    res["sampled_tapes_bit_identical"] = bool(o_r["steps"] == T and torch.equal(o_r["tape"], o_s["tape"].reshape(T, K * B)))
    del o_s, o_r, o_t, g_s, g_r
    agent.opt.zero_grad()
    shared, repl = [], []
    for i in range(a.reps):
        shared.append(step_samples(agent, env, K, seed + 2 * i)[0])
        repl.append(step_replicated(agent, env_rep, B, seed + 2 * i)[0])
    res["samples_path"] = {"runs": shared, "summary": summary(shared)}
    res["replicated_path"] = {"runs": repl, "summary": summary(repl)}
    del env_rep
    torch.cuda.empty_cache()
    if a.big_batch:
        Bg = a.big_batch
        env_g = TSPEnv(N, Bg, 0, seed=70, instance_rng="philox")
        step_samples(agent, env_g, K, seed)
        big = [step_samples(agent, env_g, K, seed + i)[0] for i in range(max(2, a.reps // 2))]
        res["samples_path_big"] = {"batch": Bg, "samples": K, "tours": Bg * K, "runs": big, "summary": summary(big)}
        res["replicated_big_saved_gib_computed"] = int(vrpx.lib().vrpx_encoder_saved_bytes(K * Bg, N)) / 2 ** 30
    s, r = res["samples_path"]["summary"], res["replicated_path"]["summary"]
    res["verdict"] = {"step_faster": s["step"]["max"] < r["step"]["min"],
                      "decoder_bwd_ratio_median": s["decoder_bwd"]["median"] / r["decoder_bwd"]["median"]}
    line = json.dumps(res, indent=1)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
