"""GPU parity of the encoder + fused rollout kernel through the reference-shaped surface (agents.*), against the
golden traces recorded from the unmodified reference and against the fp32 oracle.

Tolerances (north_star): logits / embeddings / costs 1e-5 relative (absolute floor 1e-5 for magnitudes below 1);
greedy tours identical except for documented near-ties (top-2 logit gap below 2e-5)."""
import json
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

CASES = [(4, 2, 69), (10, 8, 7), (20, 32, 1234)]


def _cls(kind):
    from agents import IRPAgent, TSPAgent, VRPAgent
    from gym_vrp.envs import IRPEnv, TSPEnv, VRPEnv

    return {"tsp": (TSPEnv, TSPAgent), "vrp": (VRPEnv, VRPAgent), "irp": (IRPEnv, IRPAgent)}[kind]


def _load(golden_dir, kind):
    return np.load(os.path.join(golden_dir, f"policy_{kind}.npz"))


def _rel(got, ref):
    return float((np.abs(got - ref) / np.maximum(np.abs(ref), 1.0)).max())


@pytest.mark.parametrize("score_tables", [True, False], ids=["tables", "classic"])
@pytest.mark.parametrize("gemm_path", [1, 0], ids=["simt", "tcgen05"])
@pytest.mark.parametrize("kind", ["tsp", "vrp", "irp"])
def test_teacher_forced_logits_and_embeddings(golden_dir, kind, gemm_path, score_tables):
    """Replay the reference's greedy tape: per-step masked pointer logits, embeddings and costs match — with the
    per-episode glimpse score tables (default) and with the classic per-step score pass."""
    z = _load(golden_dir, kind)
    Env, Agent = _cls(kind)
    for N, B, seed in CASES:
        key = f"{N}_{B}_{seed}"
        env = Env(N, B, 1, seed)
        agent = Agent(seed=seed)
        agent.model.eval()
        agent.model.encoder.gemm_path = gemm_path
        agent.model.decoder.score_tables = score_tables
        tape = z[key + "/greedy_actions"]
        with torch.no_grad():
            loss, logp = agent.model(env, rollout=True, tape=tape, want_logits=True)
        out = agent.model.last_rollout
        got, ref = out["logits"].cpu().numpy(), z[key + "/greedy_logits"]
        assert out["steps"] == tape.shape[0] == env.step_count
        fin = np.isfinite(ref)
        assert np.array_equal(fin, np.isfinite(got)), "mask pattern differs"
        assert _rel(got[fin], ref[fin]) < 1e-5, (kind, key, _rel(got[fin], ref[fin]))
        assert _rel(out["emb"][: min(B, 4)].cpu().numpy(), z[key + "/emb_eval"]) < 1e-5
        assert _rel(loss.cpu().numpy(), z[key + "/greedy_loss"]) < 1e-5


@pytest.mark.parametrize("kind", ["tsp", "vrp", "irp"])
def test_greedy_tours_identical(golden_dir, kind):
    """Free-running greedy evaluate(): same tours as the reference except for near-ties."""
    z = _load(golden_dir, kind)
    Env, Agent = _cls(kind)
    for N, B, seed in CASES:
        key = f"{N}_{B}_{seed}"
        env = Env(N, B, 1, seed)
        agent = Agent(seed=seed)
        loss = agent.evaluate(env)
        tape = agent.model.last_rollout["tape"].cpu().numpy()
        ref_tape, ref_logits = z[key + "/greedy_actions"], z[key + "/greedy_logits"]
        assert tape.shape == ref_tape.shape
        for b in range(B):
            diff = np.flatnonzero(tape[:, b] != ref_tape[:, b])
            if diff.size:  # must be a documented near-tie at the first divergence
                t = diff[0]
                top2 = np.sort(ref_logits[t, b][np.isfinite(ref_logits[t, b])])[-2:]
                assert top2[1] - top2[0] < 2e-5, (kind, key, b, t, top2)
            else:
                assert abs(loss[b].item() - z[key + "/greedy_loss"][b]) <= 1e-5 * max(1, abs(z[key + "/greedy_loss"][b]))
        assert loss.device.type == "cuda" and loss.dtype == torch.float32


def test_known_answer_means(golden_dir):
    """SURVEY App. C: Agent(seed=1234).evaluate(Env(20,256,3,seed=1234)) means and step counts."""
    ka = json.load(open(os.path.join(golden_dir, "known_answers.json")))
    for kind in ("tsp", "vrp", "irp"):
        Env, Agent = _cls(kind)
        env = Env(20, 256, 3, seed=1234)
        loss = Agent(seed=1234).evaluate(env)
        assert env.step_count == ka[f"{kind}_20_256_1234_steps"]
        # tolerance: mean tour cost within 0.1% (north_star); in practice ~1e-6
        assert abs(loss.mean().item() - ka[f"{kind}_20_256_1234_greedy_mean"]) <= 1e-3 * abs(ka[f"{kind}_20_256_1234_greedy_mean"])


def test_reference_agent_tests(golden_dir):
    """reference tests/test_agent.py:72-114 — agent.step(env, [True, True]) on B=2, N=4 with a model in train mode
    (batch-statistics BatchNorm)."""
    ka = json.load(open(os.path.join(golden_dir, "known_answers.json")))
    for kind in ("tsp", "vrp", "irp"):
        torch.manual_seed(69)
        np.random.seed(69)
        Env, Agent = _cls(kind)
        env = Env(num_nodes=4, batch_size=2, num_draw=1)
        agent = Agent()
        loss, loss_b, _ = agent.step(env, [True, True])
        assert np.isclose(loss.mean().item(), ka[f"test_{kind}_agent_mean"], rtol=1e-5), kind


@pytest.mark.parametrize("kind", ["tsp", "vrp", "irp"])
def test_teacher_forced_logprob_eval_and_train(golden_dir, kind):
    """Sampling mode, teacher-forced along a recorded tape: summed log-probs (eval- and train-mode BatchNorm)."""
    z = _load(golden_dir, kind)
    Env, Agent = _cls(kind)
    for N, B, seed in CASES:
        key = f"{N}_{B}_{seed}"
        tape = z[key + "/tf_tape"]
        agent = Agent(seed=seed)
        agent.model.eval()
        env = Env(N, B, 1, seed)
        with torch.no_grad():
            loss, logp = agent.model(env, rollout=False, tape=tape)
        assert _rel(loss.cpu().numpy(), z[key + "/tf_loss"]) < 1e-5
        assert np.allclose(logp.cpu().numpy(), z[key + "/tf_logp"], rtol=1e-5, atol=2e-5)
        agent.model.train()
        env = Env(N, B, 1, seed)
        with torch.no_grad():
            loss, logp = agent.model(env, rollout=False, tape=tape)
        assert np.allclose(agent.model.last_rollout["emb"][: min(B, 4)].cpu().numpy(), z[key + "/train_emb"], rtol=1e-4, atol=1e-4)
        assert np.allclose(logp.cpu().numpy(), z[key + "/train_logp"], rtol=1e-4, atol=1e-4)
        bn = agent.model.encoder.attention_layers[0].bn1.norm
        assert np.allclose(bn.running_mean.cpu().numpy(), z[key + "/bn_l0_running_mean"], rtol=1e-4, atol=1e-5)
        assert np.allclose(bn.running_var.cpu().numpy(), z[key + "/bn_l0_running_var"], rtol=1e-4, atol=1e-5)
        assert int(bn.num_batches_tracked) == 1


@pytest.mark.parametrize("kind", ["tsp", "vrp", "irp"])
def test_full_size_properties_vs_oracle(kind):
    """Size-independent properties at a large batch (B=8192, N=50) + oracle replay on a slice.
    * every customer is visited exactly once; TSP tours are N-1 steps;
    * the kernel's f32 cost equals the tour length recomputed from the action tape;
    * teacher-forcing the oracle with the kernel's tape reproduces the kernel's decisions."""
    from oracle import policy_oracle as po
    from oracle.env_oracle import EnvOracle

    Env, Agent = _cls(kind)
    B, N = 8192, 50
    env = Env(N, B, 0, seed=3, instance_rng="philox")
    agent = Agent(seed=3)
    agent.model.coupling = 256     # reference semantics at batch 256 for every group of 256 instances
    loss = agent.evaluate(env)
    out = agent.model.last_rollout
    tape = out["tape"].cpu().numpy().astype(np.int64)
    T = tape.shape[0]
    s = env.sampler
    xy, depot, demand = s.get_graph_positions(), s.get_depots()[:, 0], s.get_demands()[:, :, 0]
    if kind == "tsp":
        assert T == N - 1
    counts = np.zeros((B, N), dtype=np.int64)
    np.add.at(counts, (np.arange(B)[None, :].repeat(T, 0), tape), 1)
    cust = np.ones((B, N), dtype=bool)
    cust[np.arange(B), depot] = False
    assert np.all(counts[cust] == 1), "a customer was skipped or visited twice"
    # recompute tour length in f32 accumulation order
    cur = depot.copy()
    acc = np.zeros(B, dtype=np.float32)
    ar = np.arange(B)
    for t in range(T):
        d = xy[ar, cur] - xy[ar, tape[t]]
        acc = acc + np.sqrt(d[:, 0] ** 2 + d[:, 1] ** 2).astype(np.float32)
        cur = tape[t]
    assert np.allclose(-loss.cpu().numpy(), acc, rtol=1e-6, atol=1e-6)
    # oracle replay on the first coupling group (256 instances = one reference batch)
    G = 256
    sd = {k: v.float().cpu() for k, v in agent.model.state_dict().items()}
    orc = EnvOracle(kind, xy[:G], depot[:G], demand[:G])
    _, _, tr = po.rollout(sd, orc, greedy=True, tape=tape[:, :G], return_trace=True)
    lg = tr["logits"]
    agree = 0
    for t in range(T):
        for b in range(G):
            row = lg[t, b]
            a = tape[t, b]
            assert np.isfinite(row[a]), "kernel chose a masked node"
            assert row[a] >= row[np.isfinite(row)].max() - 2e-5, (t, b)  # greedy up to near-ties
            agree += 1
    assert agree == T * G


def test_sampling_distribution_and_determinism():
    """Philox sampling: same seed -> same tape; the empirical first-step distribution matches softmax(logits)."""
    from agents import TSPAgent
    from gym_vrp.envs import TSPEnv

    N, B = 10, 4096
    agent = TSPAgent(seed=1)
    agent.model.eval()
    agent.model.coupling = 0  # no cross-instance coupling: identical instances then have identical logits
    xy = np.random.RandomState(0).rand(1, N, 2).repeat(B, 0)
    depots = np.zeros(B, dtype=int)
    runs = []
    for rep in range(2):
        torch.manual_seed(77)
        env = TSPEnv.from_arrays(xy, depots)
        with torch.no_grad():
            loss, logp = agent.model(env, rollout=False, want_logits=True)
        runs.append(agent.model.last_rollout["tape"].cpu().numpy())
    assert np.array_equal(runs[0], runs[1])
    out = agent.model.last_rollout
    u = out["logits"][0, 0].cpu().double()
    p = torch.softmax(u, -1).numpy()
    emp = np.bincount(runs[0][0], minlength=N) / B
    chi2 = B * ((emp - p) ** 2 / np.maximum(p, 1e-12))[p > 0].sum()
    assert chi2 < 40, (chi2, emp, p)  # 8 dof; P(chi2 > 40) ~ 3e-6
    assert emp[0] == 0  # the depot is masked
    assert np.isfinite(logp.cpu().numpy()).all() and (logp <= 0).all()


@pytest.mark.parametrize("kind,N,B,greedy", [("irp", 40, 4096, False), ("tsp", 50, 65536, True), ("vrp", 100, 131072, True)],
                         ids=["C3_irp40_b4096_sampled", "C4_tsp50_b65536", "C5_vrp100_b131072_per_gpu"])
def test_baseline_config_sizes_properties(kind, N, B, greedy):
    """BASELINE.json configs[2..4] at their full (per-GPU) sizes, whole-batch mask coupling like the bench, checked through
    size-independent properties of the domain (the oracle cannot run these sizes in seconds):
    * every customer is visited exactly once, nothing is visited at a masked position, TSP tours take N-1 steps;
    * the f32 cost of every instance equals its tour length recomputed on the host from the action tape;
    * IRP: the vehicle load between two depot visits never exceeds 1 (the demand of every served customer fitted);
    * sampled rollouts: finite, non-positive log-probabilities."""
    Env, Agent = _cls(kind)
    env = Env(N, B, 0, seed=11, instance_rng="philox")
    agent = Agent(seed=11)
    agent.model.eval()
    with torch.no_grad():
        if greedy:
            loss = agent.evaluate(env)
            logp = None
        else:
            torch.manual_seed(5)
            loss, logp = agent.model(env, rollout=False)
    out = agent.model.last_rollout
    tape = out["tape"].cpu().numpy()
    T = tape.shape[0]
    s = env.sampler
    xy, depot, demand = s.get_graph_positions(), s.get_depots()[:, 0], s.get_demands()[:, :, 0]
    assert tape.max() < N
    if kind == "tsp":
        assert T == N - 1
    else:
        assert N - 1 <= T <= 2 * (N - 1)
    ar = np.arange(B)
    counts = np.zeros((B, N), dtype=np.int32)
    for t in range(T):
        np.add.at(counts, (ar, tape[t]), 1)
    cust = np.ones((B, N), dtype=bool)
    cust[ar, depot] = False
    assert np.all(counts[cust] == 1), "a customer was skipped or visited twice"
    if kind == "tsp":
        assert np.all(counts[~cust] == 0), "a TSP tour returned to its depot"
    cur = depot.copy()
    acc = np.zeros(B, dtype=np.float32)
    load = np.ones(B)
    for t in range(T):
        a = tape[t].astype(np.int64)
        d = xy[ar, cur] - xy[ar, a]
        acc = acc + np.sqrt(d[:, 0] ** 2 + d[:, 1] ** 2).astype(np.float32)
        if kind == "irp":
            load = load - demand[ar, a]
            assert load.min() > -1e-12, "an IRP vehicle served a customer it had no load for"
            load[a == depot] = 1.0
        cur = a
    assert np.allclose(-loss.cpu().numpy(), acc, rtol=2e-6, atol=2e-6)
    if logp is not None:
        lp = logp.cpu().numpy()
        assert np.isfinite(lp).all() and (lp <= 0).all()


# (kind, N, B, greedy).  vrp-20 x 4800 is more than 148 x 16 instances: the persistent kernel runs several 16-instance
# tiles per CTA, the setting of the glimpse-mask race of DESIGN §3.3.
DECODE_LOOP_CASES = [("tsp", 50, 777, True), ("vrp", 21, 300, True), ("irp", 100, 130, True), ("tsp", 128, 40, True),
                     ("tsp", 50, 1000, False), ("vrp", 30, 517, False), ("irp", 40, 300, False), ("vrp", 20, 4800, False)]


@pytest.mark.parametrize("kind,N,B,greedy", DECODE_LOOP_CASES,
                         ids=[f"{k}-{n}-{b}" + ("-greedy" if g else "") for k, n, b, g in DECODE_LOOP_CASES])
def test_split_step_launches_match_persistent_kernel(kind, N, B, greedy):
    """The two decode loops of a whole-episode rollout are two evaluation orders of the same scores: the classic loop in
    the persistent kernel (GEMM-A + score pass every step) and table mode (per-episode score tables, then glimpse /
    batched GEMM-B / pointer launches per step, csrc/rollout_steps.cu, the default).  The classic loop plays the episode
    (greedy or Philox-sampled); table mode is teacher-forced along its tape.  The step counts are equal (VRP / IRP
    episodes end early: the remaining launches must be no-ops), the masked logits and the costs agree to 1e-5, the
    sampled log-probs to 1e-4 sqrt(T)."""
    Env, Agent = _cls(kind)
    agent = Agent(seed=9)
    agent.model.eval()
    env = Env(N, B, 0, seed=21, instance_rng="philox")
    agent.model.decoder.score_tables = False
    torch.manual_seed(3)
    with torch.no_grad():
        loss0, logp0 = agent.model(env, rollout=greedy, want_logits=True)
    out0 = agent.model.last_rollout
    tape, ref, T0 = out0["tape"].cpu().numpy(), out0["logits"].cpu().numpy(), out0["steps"]
    env.restart_episode()
    agent.model.decoder.score_tables = True
    with torch.no_grad():
        loss1, logp1 = agent.model(env, rollout=greedy, tape=tape, want_logits=True)
    out1 = agent.model.last_rollout
    assert out1["steps"] == T0
    got = out1["logits"].cpu().numpy()
    fin = np.isfinite(ref)
    assert np.array_equal(fin, np.isfinite(got))
    assert _rel(got[fin], ref[fin]) < 1e-5
    assert _rel(loss1.cpu().numpy(), loss0.cpu().numpy()) < 1e-5
    if not greedy:
        assert np.abs(logp1.cpu().numpy() - logp0.cpu().numpy()).max() < 1e-4 * max(1.0, float(T0)) ** 0.5
