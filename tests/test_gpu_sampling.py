"""K sampled tours per instance from one encoder pass and one score table (GraphDecoder.rollout_samples,
vrpx_rollout_samples) and best-of-K evaluation (TSPModel.sample_best, TSPAgent.evaluate(env, samples=K)).

Copy k of the K copies must be bit-identical to the whole-episode sampled call on a fresh copy of the env with the Philox
offset shifted by k·B: tape rows before the copy's own step count, the depot in the rows after it (a finished VRP / IRP
copy idles on its depot while slower copies run), cost, log-prob and logits.  The cases cover the node edges of the
node-edge suite (N = 4, 33, 57, 105, 127, 128), ragged glimpse (10-warp) and pointer (8-warp) CTAs, coupling groups
smaller than the batch and 0, K = 1 and several waves of CTAs at K = 16."""
import ctypes as C
import os
from copy import deepcopy

import numpy as np
import pytest
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
NH = 8


def _cls(kind):
    from agents import IRPAgent, TSPAgent, VRPAgent
    from gym_vrp.envs import IRPEnv, TSPEnv, VRPEnv

    return {"tsp": (TSPEnv, TSPAgent), "vrp": (VRPEnv, VRPAgent), "irp": (IRPEnv, IRPAgent)}[kind]


def _setup(kind, N, B, seed):
    from agents.graph_encoder import run_encoder

    Env, Agent = _cls(kind)
    model = Agent(seed=seed).model
    model.eval()
    env = Env(N, B, 0, seed=seed, instance_rng="philox")
    with torch.no_grad():
        h = run_encoder(model.encoder, env=env, depot=env._depot if model._USES_DEPOT_EMBED else None,
                        gemm_path=model.encoder.gemm_path)
    return model, env, h


def _check_copy(model, env, h, out, k, seed, offset, G, logits=True):
    """Copy k of `out` against rollout_episode on a fresh copy of the env at Philox offset offset + k·B."""
    B = env.batch_size
    with torch.no_grad():
        ref = model.decoder.rollout_episode(deepcopy(env), h, greedy=False, want_logits=logits, coupling=G, seed=seed,
                                            offset=offset + k * B)
    Tk = ref["steps"]
    assert Tk <= out["steps"]
    assert torch.equal(out["tape"][:Tk, k], ref["tape"]), f"copy {k}: tape"
    depot = env._depot.to(torch.uint8)
    assert torch.equal(out["tape"][Tk:, k], depot.expand(out["steps"] - Tk, B)), f"copy {k}: idle rows are not the depot"
    assert torch.equal(out["cost"][k], ref["cost"]), f"copy {k}: cost"
    assert torch.equal(out["logp"][k], ref["logp"]), f"copy {k}: log-prob"
    if logits:
        assert torch.equal(out["logits"][:Tk, k], ref["logits"]), f"copy {k}: logits"
    return Tk


# (kind, N, B, K, coupling G (None: the base batch), copies to check (None: all))
CASES = [("tsp", 4, 1, 1, None, None), ("tsp", 33, 7, 3, None, None), ("tsp", 50, 37, 10, None, None),
         ("tsp", 128, 5, 8, None, None), ("vrp", 2, 3, 4, None, None), ("vrp", 57, 13, 5, None, None),
         ("vrp", 105, 9, 2, 3, None), ("irp", 24, 8, 8, 0, None), ("irp", 127, 4, 3, None, None),
         ("tsp", 50, 2003, 16, None, (0, 7, 15))]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,N,B,K,G,copies", CASES,
                         ids=[f"{k}{n}_b{b}_k{kk}" + ("" if g is None else f"_g{g}") for k, n, b, kk, g, _ in CASES])
def test_copies_equal_independent_rollouts(kind, N, B, K, G, copies):
    seed, offset = 4242 + N, 11
    model, env, h = _setup(kind, N, B, 1000 + N)
    step_before = env.step_count
    visited_before = env.visited.copy()
    out = model.decoder.rollout_samples(env, h, K, seed=seed, offset=offset, coupling=G, want_logits=True)
    assert out["cost"].shape == (K, B) and out["logp"].shape == (K, B)
    assert out["tape"].shape == (out["steps"], K, B) and out["logits"].shape == (out["steps"], K, B, N)
    steps = [_check_copy(model, env, h, out, k, seed, offset, G) for k in (range(K) if copies is None else copies)]
    if copies is None:
        assert out["steps"] == max(steps)
    # without logits the step kernels skip the glimpse of idle finished copies: the same results bit for bit
    prod = model.decoder.rollout_samples(env, h, K, seed=seed, offset=offset, coupling=G)
    assert prod["steps"] == out["steps"]
    for key in ("tape", "cost", "logp"):
        assert torch.equal(prod[key], out[key]), key
    assert env.step_count == step_before and np.array_equal(env.visited, visited_before), "the caller's env changed"
    print(f"\n[{kind}{N} B={B} K={K} G={G}] steps {out['steps']} per copy {sorted(set(steps))}")


def _replica_bytes(N, Tmax):
    """Device bytes per replica outside the rollout workspace: env state (xy, depot, demand, visited, mask, cur, load)
    and the outputs (tape, log-prob, cost)."""
    return 16 * N + 4 + 8 * N + 16 + 16 + 4 + 8 + Tmax + 4 + 4


@pytest.mark.gpu
def test_large_k_copies_and_peak_memory():
    import vrpx

    N, B, K = 50, 8192, 64
    seed, offset = 99, 0
    model, env, h = _setup("tsp", N, B, 7)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    out = model.decoder.rollout_samples(env, h, K, seed=seed, offset=offset)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    ws = int(vrpx.lib().vrpx_rollout_samples_workspace_bytes(vrpx.TSP, B, K, N))
    bound = ws + K * B * _replica_bytes(N, N - 1) + (64 << 20)   # 64 MiB: allocator rounding of the ~12 buffers
    print(f"\npeak {peak / 2**30:.2f} GiB (bound {bound / 2**30:.2f} GiB, embeddings {h.numel() * 4 / 2**30:.2f} GiB "
          f"outside it)")
    assert peak <= bound
    for k in (0, K - 1):
        _check_copy(model, env, h, out, k, seed, offset, None, logits=False)


def _tour_length_f32(xy, depot, tape):
    B = xy.shape[0]
    ar = np.arange(B)
    cur = depot.copy()
    acc = np.zeros(B, dtype=np.float32)
    for t in range(tape.shape[0]):
        a = tape[t].astype(np.int64)
        d = xy[ar, cur] - xy[ar, a]
        acc = acc + np.sqrt(d[:, 0] ** 2 + d[:, 1] ** 2).astype(np.float32)
        cur = a
    return acc


@pytest.mark.gpu
@pytest.mark.parametrize("N,B,K", [(5, 16, 64), (2, 5, 4), (3, 5, 6)], ids=["tsp5", "tsp2_fallback", "tsp3_fallback"])
def test_sample_best(N, B, K):
    from agents import TSPAgent
    from agents.graph_encoder import run_encoder
    from gym_vrp.envs import TSPEnv

    agent = TSPAgent(seed=3)
    model = agent.model
    model.eval()
    env = TSPEnv(N, B, 0, seed=5, instance_rng="philox")
    torch.manual_seed(17)
    best = model.sample_best(env, K)
    # the same draw of the Philox seed, then every copy's results
    torch.manual_seed(17)
    seed = int(torch.randint(0, 2 ** 62, (1,)).item())
    with torch.no_grad():
        h = run_encoder(model.encoder, env=env, gemm_path=model.encoder.gemm_path)
    full = model.decoder.rollout_samples(env, h, K, seed=seed)
    costs = full["cost"].cpu().numpy()
    assert np.array_equal(best["costs"].cpu().numpy(), costs)
    idx = best["index"].cpu().numpy()
    mn = costs.min(0)
    assert np.array_equal(idx, np.array([np.flatnonzero(costs[:, b] == mn[b])[0] for b in range(B)]))
    if N == 5:
        assert ((costs == mn).sum(0) > 1).any(), "no tie among the copies: the lowest-k rule is not exercised"
    ar = np.arange(B)
    assert np.array_equal(best["cost"].cpu().numpy(), mn)
    assert np.array_equal(best["logp"].cpu().numpy(), full["logp"].cpu().numpy()[idx, ar])
    tour = best["tour"].cpu().numpy()
    assert np.array_equal(tour, full["tape"].cpu().numpy()[:, idx, ar])
    s = env.sampler
    xy, depot = s.get_graph_positions(), s.get_depots()[:, 0]
    for b in range(B):
        assert sorted(tour[:, b].tolist() + [int(depot[b])]) == list(range(N)), f"instance {b}: not a permutation"
    assert np.allclose(mn, _tour_length_f32(xy, depot, tour), rtol=1e-6, atol=1e-6)

    step_before, visited_before = env.step_count, env.visited.copy()
    reward = agent.evaluate(env, samples=K)
    assert reward.shape == (B,)
    assert env.step_count == step_before and np.array_equal(env.visited, visited_before)


@pytest.mark.gpu
def test_best_of_16_beats_greedy_on_trained_checkpoint():
    from agents import TSPAgent
    from gym_vrp.envs import TSPEnv

    agent = TSPAgent(seed=123)
    agent.model.load_state_dict(torch.load(os.path.join(GOLDEN, "ckpt_tsp_20_123.pt"), map_location=agent.device))
    env = TSPEnv(20, 256, seed=1234)
    torch.manual_seed(0)
    sampled = -agent.evaluate(env, samples=16).mean().item()
    greedy = -agent.evaluate(env).mean().item()
    print(f"\nmean tour length: best of 16 {sampled:.4f}, greedy {greedy:.4f}")
    assert sampled < greedy, (sampled, greedy)


@pytest.mark.gpu
def test_argument_checks():
    import vrpx

    L = vrpx.lib()
    N, B, K = 10, 4, 3
    model, env, h = _setup("tsp", N, B, 1)
    dev = h.device
    R = B * K
    z = lambda *s, dt=torch.int32: torch.zeros(s, dtype=dt, device=dev)
    xy, depot, demand = env._xy.repeat(K, 1, 1), env._depot.repeat(K), env._demand.repeat(K, 1)
    visited, cur, load = z(R, 4), z(R), z(R, dt=torch.float64) + 1

    def view(rows):
        v = vrpx.EnvView()
        v.kind, v.N, v.B = vrpx.TSP, N, rows
        v.xy, v.depot, v.demand = xy.data_ptr(), depot.data_ptr(), demand.data_ptr()
        v.visited, v.mask, v.cur, v.load = visited.data_ptr(), visited.data_ptr(), cur.data_ptr(), load.data_ptr()
        return v

    w = model.decoder.packed(False, dev)
    tape, logp, cost, steps = z(N, R, dt=torch.uint8), z(R, dt=torch.float32), z(R, dt=torch.float32), z(1)
    nbytes = int(L.vrpx_rollout_samples_workspace_bytes(vrpx.TSP, B, K, N))
    ws = z(nbytes, dt=torch.uint8)

    def call(v=None, w_=w, Bb=B, K_=K, G=B, Tmax=N - 1, ws_bytes=nbytes):
        vv = view(R) if v is None else v
        L.vrpx_env_reset(C.byref(vv), vrpx.stream_ptr(dev))
        return L.vrpx_rollout_samples(C.byref(vv), C.byref(w_), vrpx.ptr(h), Bb, K_, G, C.c_uint64(1), C.c_uint64(0),
                                      vrpx.ptr(tape), Tmax, vrpx.ptr(logp), vrpx.ptr(cost), vrpx.ptr(steps), None,
                                      vrpx.ptr(ws), ws_bytes, vrpx.stream_ptr(dev))

    ERR_ARG, ERR_UNSUPPORTED = -1, -4
    no_qk = vrpx.DecoderWeights.from_buffer_copy(w)
    no_qk.qk_w = None
    assert call(K_=0) == ERR_ARG
    assert call(v=view(R - 1)) == ERR_ARG
    assert call(Bb=B + 1) == ERR_ARG
    assert call(G=3) == ERR_ARG                  # not a divisor of Bb
    assert call(G=R) == ERR_ARG                  # divides Bb·K but not Bb: partners would cross copies
    assert call(G=-1) == ERR_ARG
    assert call(w_=no_qk) == ERR_ARG
    assert call(ws_bytes=nbytes - 1) == ERR_ARG
    assert call(Tmax=2) == ERR_UNSUPPORTED
    for G in (B, 2, 1, 0):
        assert call(G=G) == 0, vrpx.lib().vrpx_last_error()
    torch.cuda.synchronize()
    assert int(steps.item()) == N - 1


@pytest.mark.parametrize("kind", [0, 1, 2])
@pytest.mark.parametrize("B,N", [(1, 2), (7, 33), (65536, 50), (9, 128)])
def test_samples_workspace_arithmetic(kind, B, N):
    """The samples workspace at K = 1 is the table workspace.  At K > 1 it is the table workspace of K·B instances with
    the K·B-row score table S1 replaced by the B-row one and the step flags of the copies added (up to the 256-byte
    alignment of the segments behind S1): every other per-instance segment is per replica, S1 does not grow with K."""
    import vrpx

    L = vrpx.lib()
    one = int(L.vrpx_rollout_samples_workspace_bytes(kind, B, 1, N))
    assert one == int(L.vrpx_rollout_table_workspace_bytes(kind, B, N))
    s1 = B * N * NH * N * 4
    for K in (2, 3, 64):
        ws = int(L.vrpx_rollout_samples_workspace_bytes(kind, B, K, N))
        replicated = int(L.vrpx_rollout_table_workspace_bytes(kind, K * B, N))
        # the same layout with the K·B-row S1 replaced by the B-row one, plus the step flags: [2N][K] int32 per copy and
        # one byte per replica
        flags = 2 * N * K * 4 + K * B
        assert abs(ws - (replicated - (K - 1) * s1) - flags) <= 3 * 256, (K, ws, replicated)
