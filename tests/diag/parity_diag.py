#!/usr/bin/env python
"""Diagnose logit parity at benchmark sizes: per-mode / per-step error against the oracle (runs on the GPU box)."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (os.path.join(ROOT, "vrp-gym_b200"), ROOT, os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
import numpy as np
import torch

import vrpx
from oracle import policy_oracle as po
from oracle.env_oracle import EnvOracle
from test_gpu_parity_sizes import MODES, _cls, _mask_history


def rel(a, b):
    return np.abs(a - b) / np.maximum(np.abs(b), 1.0)


def golden_case(kind, key, gemm_path, mode):
    z = np.load(os.path.join(ROOT, "tests", "golden", f"policy_{kind}_large.npz"))
    N, B, seed = (int(x) for x in key.split("_"))
    Env, Agent = _cls(kind)
    tables, split = MODES[mode]
    vrpx.lib().vrpx_debug_rollout_split(split)
    env = Env(N, B, 1, seed)
    agent = Agent(seed=seed)
    agent.model.eval()
    agent.model.encoder.gemm_path = gemm_path
    agent.model.decoder.score_tables = tables
    tape = z[key + "/greedy_actions"]
    with torch.no_grad():
        agent.model(env, rollout=True, tape=tape, want_logits=True)
    out = agent.model.last_rollout
    got, ref = out["logits"].cpu().numpy(), z[key + "/greedy_logits"]
    fin = np.isfinite(ref)
    e = np.where(fin, rel(got, np.where(fin, ref, 0)), 0)
    per_step = e.reshape(e.shape[0], -1).max(1)
    emb = rel(out["emb"].cpu().numpy(), z[key + "/emb_eval"]).max()
    worst = np.unravel_index(e.argmax(), e.shape)
    print(f"golden {kind} {key} path{gemm_path} {mode}: max {e.max():.2e} at (t,b,n)={worst} emb {emb:.2e} "
          f"steps>1e-5: {np.flatnonzero(per_step > 1e-5)[:12].tolist()} first3 {per_step[:3]}", flush=True)
    vrpx.lib().vrpx_debug_rollout_split(1)


def slice_case(kind, N, B, S, gemm_path=0, mode="tables_split", coupling=None, seed=3):
    Env, Agent = _cls(kind)
    tables, split = MODES[mode]
    vrpx.lib().vrpx_debug_rollout_split(split)
    env = Env(N, B, 0, seed=seed, instance_rng="philox")
    agent = Agent(seed=seed)
    agent.model.eval()
    agent.model.encoder.gemm_path = gemm_path
    agent.model.decoder.score_tables = tables
    agent.model.coupling = coupling
    G = B if coupling is None else coupling
    rs = np.random.RandomState(5)
    sel = np.unique(np.concatenate([[0, 1, B // 8 - 1, B // 8, B // 2, B - 2, B - 1], rs.choice(B, S, replace=False)]))[:S]
    sel_dev = torch.as_tensor(sel, device=env._device)
    with torch.no_grad():
        agent.model(env, rollout=True, want_logits=True)
    out = agent.model.last_rollout
    T = out["steps"]
    got = out["logits"][:, sel_dev].cpu().numpy()
    emb = out["emb"][sel_dev].cpu().numpy()
    tape = out["tape"].cpu().numpy()
    s = env.sampler
    xy, depot, demand = s.get_graph_positions(), s.get_depots()[:, 0], s.get_demands()[:, :, 0]
    g0 = (sel // G) * G
    partners = g0[:, None] + ((sel - g0)[:, None] * 8 + np.arange(8)[None, :]) % G
    rows = np.concatenate([sel, partners.reshape(-1)])
    masks, loads = _mask_history(kind, xy, depot, demand, tape, rows)
    own = masks[:, : len(sel)]
    glimpse = masks[:, len(sel):].reshape(T, len(sel), 8, N)
    sd = {k: v.float().cpu() for k, v in agent.model.state_dict().items()}
    st = torch.tensor(xy[sel], dtype=torch.float)
    doh = torch.zeros(len(sel), N, dtype=torch.bool)
    doh[torch.arange(len(sel)), torch.as_tensor(depot[sel])] = True
    if kind == "tsp":
        h = po.encoder_forward(sd, st, None, False)
    elif kind == "vrp":
        h = po.encoder_forward(sd, st, doh, False)
    else:
        h = po.encoder_forward(sd, torch.cat([st, torch.tensor(demand[sel], dtype=torch.float)[:, :, None]], -1), doh, False)
    eemb = rel(emb, h.numpy()).max()
    ref, _ = po.replay_subset_logits(sd, h, tape[:, sel].astype(np.int64), own, glimpse, loads[:, : len(sel)] if kind == "irp" else None)
    # same replay but with the GPU's embeddings: separates encoder error from decoder error
    ref2, _ = po.replay_subset_logits(sd, torch.tensor(emb), tape[:, sel].astype(np.int64), own, glimpse,
                                      loads[:, : len(sel)] if kind == "irp" else None)
    fin = np.isfinite(ref)
    okmask = np.array_equal(fin, np.isfinite(got))
    e = np.where(fin, rel(got, np.where(fin, ref, 0)), 0)
    e2 = np.where(fin, rel(got, np.where(fin, ref2, 0)), 0)
    per_step = e.reshape(T, -1).max(1)
    per_inst = e.max(axis=(0, 2))
    worst = np.unravel_index(e.argmax(), e.shape)
    print(f"slice {kind}-{N} B={B} G={G} path{gemm_path} {mode}: masks_equal={okmask} emb {eemb:.2e} max {e.max():.2e} "
          f"(with GPU emb {e2.max():.2e}) at (t,s,n)={worst} inst={sel[worst[1]]}; instances>1e-5: {(per_inst > 1e-5).sum()}/{len(sel)}; "
          f"steps>1e-5 {np.flatnonzero(per_step > 1e-5)[:10].tolist()} median step err {np.median(per_step):.1e}", flush=True)
    if e.max() > 1e-5:
        t, si, n = worst
        print("   worst row got", got[t, si][:8], "ref", ref[t, si][:8], "cands", int(fin[t, si].sum()), flush=True)
    vrpx.lib().vrpx_debug_rollout_split(1)


def ckpt_case(kind, tag, gemm_path, mode):
    """Trained checkpoint (tests/golden/ckpt_*): teacher-forced logits vs the reference's, vs the oracle in f32 and f64."""
    pt = os.path.join(ROOT, "tests", "golden", f"ckpt_{kind}_20_123.pt")
    z = np.load(os.path.join(ROOT, "tests", "golden", f"ckpt_{kind}_20_123_eval.npz"))
    Env, Agent = _cls(kind)
    tables, split = MODES[mode]
    vrpx.lib().vrpx_debug_rollout_split(split)
    n2, b2, s2 = (int(v) for v in z[f"{tag}/cfg"])
    env = Env(n2, b2, 3, seed=s2)
    agent = Agent(seed=s2)
    agent.model.load_state_dict(torch.load(pt, map_location=agent.device))
    agent.model.eval()
    agent.model.encoder.gemm_path = gemm_path
    agent.model.decoder.score_tables = tables
    tape, ref = z[f"{tag}/greedy_actions"], z[f"{tag}/greedy_logits"]
    with torch.no_grad():
        agent.model(env, rollout=True, tape=tape, want_logits=True)
    out = agent.model.last_rollout
    got = out["logits"].cpu().numpy()
    s = env.sampler
    xy, depot, demand = s.get_graph_positions(), s.get_depots()[:, 0], s.get_demands()[:, :, 0]
    sd = {k: v.float().cpu() for k, v in agent.model.state_dict().items()}
    sd64 = {k: (v.double() if v.is_floating_point() else v) for k, v in sd.items()}
    _, _, tr64 = po.rollout(sd64, EnvOracle(kind, xy, depot, demand), greedy=True, tape=tape, return_trace=True, dtype=torch.float64)
    fin = np.isfinite(ref)
    e_ref = np.where(fin, rel(got, np.where(fin, ref, 0)), 0)
    e_64 = np.where(fin, rel(got.astype(np.float64), np.where(fin, tr64["logits"], 0)), 0)
    r_64 = np.where(fin, rel(ref.astype(np.float64), np.where(fin, tr64["logits"], 0)), 0)
    emb64 = rel(out["emb"].cpu().numpy().astype(np.float64), tr64["emb"]).max()
    # decoder alone: oracle f64 replay on the GPU's embeddings
    B = b2
    rows = (np.arange(B)[:, None] * 8 + np.arange(8)[None, :]) % B
    masks, loads = _mask_history(kind, xy, depot, demand, tape, np.arange(B))
    ref2, _ = po.replay_subset_logits(sd64, out["emb"].cpu().double(), tape, masks, masks[:, rows], None)
    e_dec = np.where(fin, rel(got.astype(np.float64), np.where(fin, ref2, 0)), 0)
    per_step = e_64.reshape(e_64.shape[0], -1).max(1)
    print(f"ckpt {kind}/{tag} N={n2} path{gemm_path} {mode}: vs ref32 {e_ref.max():.2e} vs f64 {e_64.max():.2e} (ref32 vs f64 {r_64.max():.2e}) "
          f"emb vs f64 {emb64:.2e} |emb|max {np.abs(tr64['emb']).max():.1f} decoder-only vs f64 {e_dec.max():.2e} worst steps "
          f"{np.argsort(per_step)[-3:].tolist()} median step {np.median(per_step):.1e}", flush=True)
    vrpx.lib().vrpx_debug_rollout_split(1)


if __name__ == "__main__":
    what = sys.argv[1] if len(sys.argv) > 1 else "all"
    if what in ("all", "ckpt"):
        for kind in ("tsp", "vrp"):
            for tag in ("a", "b"):
                for gp, mode in ((0, "tables_split"), (1, "tables_split"), (0, "classic"), (1, "classic")):
                    ckpt_case(kind, tag, gp, mode)
    if what in ("all", "golden"):
        for mode in MODES:
            for gp in (0, 1):
                for key in ("40_8_30", "50_8_31", "100_8_32"):
                    golden_case("irp", key, gp, mode)
        golden_case("tsp", "50_8_31", 0, "tables_split")
        golden_case("vrp", "100_8_32", 0, "tables_split")
    if what in ("all", "slice"):
        for kind, N, B, S in (("tsp", 50, 65536, 256), ("tsp", 50, 4096, 256), ("tsp", 50, 256, 256)):
            for mode in ("tables_split", "classic"):
                for gp in (0, 1):
                    slice_case(kind, N, B, S, gp, mode)
        slice_case("tsp", 50, 65536, 256, 0, "tables_split", coupling=256)
        slice_case("irp", 40, 4096, 128, 0, "tables_split", seed=7)
        slice_case("irp", 40, 4096, 128, 1, "classic", seed=7)
        slice_case("vrp", 100, 131072, 48, 0, "tables_split")
