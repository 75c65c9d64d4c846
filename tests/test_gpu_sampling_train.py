"""Training on K sampled tours per instance from one train-mode encoder pass (TSPModel.forward_samples, the K-sample
REINFORCE backward of vrpx/backward.py, vrpx_rollout_samples_traced and vrpx_decoder_backward_samples).

1. The trace of the copies: every copy's mask / load history, Q~g before and after the `first` fold equal those of the
   copy run alone bit for bit; after a copy's own end, up to the slowest copy's step count, its rows hold its terminal
   mask and load (the backward replays those steps); no row below the step count is left unwritten.
2. The decoder backward over the K·B replicas: copy k's per-replica dL/dh and per-episode sums equal
   vrpx_decoder_backward on copy k alone bit for bit; the step-weight gradients equal the sum over the lone copies up to
   the order of their red.add.
3. The whole train step against float64 autograd of the oracle: the encoder over the B base instances in train mode,
   the decoder teacher-forced over the K·B replicas on h[base], partners inside each copy.
4. The same update as today's train step on the copy-major K-fold replicated env (coupling B), teacher-forced along the
   same tapes, and running statistics equal to one train-mode encoder pass over the base batch.
5. TSPAgent.train(samples=K), the argument checks and a peak-memory bound at TSP-50 x 8,192, K = 8."""
import csv
import ctypes as C
from copy import deepcopy

import numpy as np
import pytest
import torch
from oracle_replay import check_logp as _check_logp
from oracle_replay import host_inputs as _host_inputs
from oracle_replay import partners as _partners
from test_gpu_backward_scale import TOL, _compare, _decoder_reference, _device_inputs, _kernel_gate
from test_gpu_sampling import _cls, _setup

pytestmark = pytest.mark.gpu

F64 = torch.float64


def _max_steps(kind, N):
    return (N - 1) if kind == "tsp" else 2 * (N - 1) + 1


def _replicas(env, K):
    """The copy-major replica env of K copies of env in its reset state: (vrpx_env view, arrays it points to)."""
    import vrpx

    B, N = env.batch_size, env.num_nodes
    R, dev = K * B, env._device
    env._sync_instances()
    a = {"xy": env._xy.repeat(K, 1, 1), "depot": env._depot.repeat(K), "demand": env._demand.repeat(K, 1),
         "visited": torch.zeros((R, 4), dtype=torch.int32, device=dev), "cur": torch.empty((R,), dtype=torch.int32, device=dev),
         "load": torch.ones((R,), dtype=torch.float64, device=dev)}
    a["mask"] = a["visited"] if env._KIND != vrpx.IRP else torch.zeros((R, 4), dtype=torch.int32, device=dev)
    v = vrpx.EnvView()
    v.kind, v.N, v.B = env._KIND, N, R
    for f in ("xy", "depot", "demand", "visited", "mask", "cur", "load"):
        setattr(v, f, a[f].data_ptr())
    vrpx.check(vrpx.lib().vrpx_env_reset(C.byref(v), vrpx.stream_ptr(dev)))
    return v, a


def _lone(model, env, h, G, seed, offset):
    """One copy alone: the whole-episode sampled call with its trace, and its env (terminal state)."""
    e = deepcopy(env)
    with torch.no_grad():
        out = model.decoder.rollout_episode(e, h, greedy=False, coupling=G, seed=seed, offset=offset, save_for_backward=True)
    return out, e


# ------------------------------------------------------------------------------------------------ 1. trace of the copies
TRACE_CASES = [("tsp", 33, 7, 3, None), ("vrp", 57, 13, 5, None), ("irp", 127, 4, 3, None), ("vrp", 105, 9, 2, 3),
               ("tsp", 128, 5, 8, None)]


@pytest.mark.parametrize("kind,N,B,K,G", TRACE_CASES,
                         ids=[f"{k}{n}_b{b}_k{kk}" + ("" if g is None else f"_g{g}") for k, n, b, kk, g in TRACE_CASES])
def test_trace_of_copies(kind, N, B, K, G):
    import vrpx

    L = vrpx.lib()
    seed, offset = 313 + N, 7
    model, env, h = _setup(kind, N, B, 3000 + N)
    dev = h.device
    R, Tmax, Gc = K * B, _max_steps(kind, N), (B if G is None else G)
    v, keep = _replicas(env, K)
    tape = torch.empty((Tmax, R), dtype=torch.uint8, device=dev)
    logp, cost = torch.empty(R, device=dev), torch.empty(R, device=dev)
    steps = torch.zeros(1, dtype=torch.int32, device=dev)
    # sentinels: an all-ones mask row (never a decoder-visible mask: some node is always open) and NaN
    mask_hist = torch.full((Tmax, R, 4), -1, dtype=torch.int32, device=dev)
    load_hist = torch.full((Tmax, R), float("nan"), device=dev)
    qg0 = torch.full((R, 1024), float("nan"), device=dev)
    trace = vrpx.RolloutTrace(mask_hist.data_ptr(), load_hist.data_ptr(), qg0.data_ptr())
    nbytes = int(L.vrpx_rollout_samples_workspace_bytes(env._KIND, B, K, N))
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
    w = model.decoder.packed(kind == "irp", dev)
    vrpx.check(L.vrpx_rollout_samples_traced(C.byref(v), C.byref(w), vrpx.ptr(h), B, K, Gc, C.c_uint64(seed),
                                             C.c_uint64(offset), vrpx.ptr(tape), Tmax, vrpx.ptr(logp), vrpx.ptr(cost),
                                             vrpx.ptr(steps), None, C.byref(trace), vrpx.ptr(ws), nbytes,
                                             vrpx.stream_ptr(dev)))
    T = int(steps.item())
    o = int(L.vrpx_rollout_workspace_qg_offset())
    qg = ws[o:o + R * 4096].view(torch.float32).view(R, 1024)
    # the trace changes nothing else
    plain = model.decoder.rollout_samples(env, h, K, seed=seed, offset=offset, coupling=G)
    assert plain["steps"] == T
    assert torch.equal(plain["tape"].reshape(T, R), tape[:T]) and torch.equal(plain["cost"].reshape(-1), cost)
    assert torch.equal(plain["logp"].reshape(-1), logp)
    lengths = []
    for k in range(K):
        ref, e = _lone(model, env, h, G, seed, offset + k * B)
        Tk, sv, r = ref["steps"], ref["saved"], slice(k * B, (k + 1) * B)
        lengths.append(Tk)
        assert torch.equal(mask_hist[:Tk, r], sv["mask_hist"][:Tk]), f"copy {k}: mask_hist"
        assert torch.equal(load_hist[:Tk, r], sv["load_hist"][:Tk]), f"copy {k}: load_hist"
        assert torch.equal(qg0[r], sv["qg0"]), f"copy {k}: qg0"
        assert torch.equal(qg[r], sv["qg"]), f"copy {k}: qg"
        # after the copy's own end: its terminal mask and load
        assert torch.equal(mask_hist[Tk:T, r], e._mask.expand(T - Tk, B, 4)), f"copy {k}: rows after its end"
        assert torch.equal(load_hist[Tk:T, r], e._load.float().expand(T - Tk, B)), f"copy {k}: loads after its end"
    assert max(lengths) == T
    assert not bool((mask_hist[:T] == -1).all(-1).any()), "sentinel mask row below the step count"
    assert not bool(load_hist[:T].isnan().any()) and not bool(qg0.isnan().any())
    if kind == "vrp" and G is None:
        assert len(set(lengths)) > 1, "the copies have one length: the rows after a copy's end are not exercised"
    print(f"\n[{kind}{N} B={B} K={K} G={G}] T={T}, per copy {lengths}")


# ------------------------------------------------------------------------------------------------ 2. decoder backward
def _decoder_backward_raw(model, view, h, Bb, K, roll, wts):
    """vrpx_decoder_backward(_samples) on zeroed gradient buffers; returns them (dH etc. per replica)."""
    import vrpx

    L = vrpx.lib()
    dev = h.device
    irp = view.kind == vrpx.IRP
    w = model.decoder.packed(irp, dev)
    tens = model.decoder._packed[irp].tensors
    R, N = view.B, view.N
    z = lambda *s: torch.zeros(s, dtype=torch.float32, device=dev)
    g = {"dH": z(R, N, 128), "D0": z(R, 1024), "D1": z(R, 1024), "Dl": z(R, 1024) if irp else None,
         "d_al_t": z(128, 1024), "d_m_t": z(1024, 128), "d_m_c": z(128)}
    gs = vrpx.DecoderGrads(*[None if g[k] is None else g[k].data_ptr() for k in ("dH", "D0", "D1", "Dl", "d_al_t", "d_m_t", "d_m_c")])
    m_n, al_n = tens["m_t"].t().contiguous(), tens["al_t"].t().contiguous()
    wb = vrpx.DecoderBwdWeights(m_n.data_ptr(), al_n.data_ptr())
    sv = roll["saved"]
    trace = vrpx.RolloutTrace(sv["mask_hist"].data_ptr(), sv["load_hist"].data_ptr(), sv["qg0"].data_ptr())
    T = roll["steps"]
    tape = roll["tape"].reshape(T, R).contiguous()
    nbytes = int(L.vrpx_decoder_backward_workspace_bytes(R, N))
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
    args = (vrpx.ptr(tape), T, int(roll["coupling"]), C.byref(trace), vrpx.ptr(sv["qg"]), vrpx.ptr(wts.contiguous()),
            C.byref(gs), vrpx.ptr(ws), nbytes, vrpx.stream_ptr(dev))
    if K is None:
        vrpx.check(L.vrpx_decoder_backward(C.byref(view), C.byref(w), C.byref(wb), vrpx.ptr(h), *args))
    else:
        vrpx.check(L.vrpx_decoder_backward_samples(C.byref(view), C.byref(w), C.byref(wb), vrpx.ptr(h), Bb, K, *args))
    return g


# d_al_t, d_m_t, d_m_c are sums over replicas and steps of per-tile partials (TF32 3-term mma.sync over the 32 instances
# of a tile, then red.add).  Copy k starts at replica k·B, which is a tile edge only when 32 divides B, so the partials
# group other instances than the lone copies' tiles do and round differently; relative to the largest element, measured
# on a B200 (1000 W): up to 3.6e-6 at TSP-20 x 1,185 (297 tiles on 148 CTAs), below 1e-6 at one tile per copy.
STEP_WEIGHT_TOL = 1e-5
BWD_CASES = [("tsp", 20, 1185, 8, None), ("tsp", 20, 1185, 8, 5), ("vrp", 57, 13, 5, None), ("irp", 127, 4, 3, None),
             ("vrp", 105, 9, 2, 3)]


@pytest.mark.parametrize("kind,N,B,K,G", BWD_CASES,
                         ids=[f"{k}{n}_b{b}_k{kk}" + ("" if g is None else f"_g{g}") for k, n, b, kk, g in BWD_CASES])
def test_decoder_backward_per_copy(kind, N, B, K, G):
    seed, offset = 919 + N, 3
    model, env, h = _setup(kind, N, B, 4000 + N)
    dev = h.device
    R = K * B
    with torch.no_grad():
        out = model.decoder.rollout_samples(env, h, K, seed=seed, offset=offset, coupling=G, save_for_backward=True)
    gen = torch.Generator(device=dev).manual_seed(N)
    wts = torch.randn(R, generator=gen, device=dev) * 1e-3
    got = _decoder_backward_raw(model, out["saved"]["replicas"], h, B, K, out, wts)
    acc = {n: torch.zeros_like(got[n]) for n in ("d_al_t", "d_m_t", "d_m_c")}
    for k in range(K):
        ref, e = _lone(model, env, h, G, seed, offset + k * B)
        r = slice(k * B, (k + 1) * B)
        one = _decoder_backward_raw(model, e._view(), h, B, None, ref, wts[r].clone())
        for n in ("dH", "D0", "D1", "Dl"):
            if one[n] is not None:
                assert torch.equal(got[n][r], one[n]), f"copy {k}: {n}"
        for n in acc:
            acc[n] += one[n]
    for n, a in acc.items():
        err, sc = (got[n] - a).abs().max().item(), a.abs().max().item()
        print(f"\n[{kind}{N} B={B} K={K} G={G}] {n}: max |samples - sum of lone copies| / max {err / sc:.3g}")
        assert err <= STEP_WEIGHT_TOL * sc, (n, err, sc)


# ------------------------------------------------------------------------------------------------ 3. vs float64
def _sample_train_step(kind, N, B, K, G, gemm_path, seed):
    """A K-sample train step of a seed-initialised model against K sampled copies of the same model in eval mode.
    Returns (model, env, wts = advantage / (K·B) as (K,B), float64 copy of the weights taken before the forward)."""
    Env, Agent = _cls(kind)
    model = Agent(seed=seed).model
    model.coupling = G
    model.encoder.gemm_path = gemm_path
    sd = {k: v.detach().to(F64).clone() for k, v in model.state_dict().items()}
    env = Env(N, B, 0, seed=seed, instance_rng="philox")
    model.eval()
    with torch.no_grad():
        loss_b, _ = model.forward_samples(env, K)
    model.train()
    torch.manual_seed(seed)
    loss_m, _ = model.forward_samples(env, K)
    wts = ((loss_m - loss_b) * -1 / (K * B)).detach()
    return model, env, wts, sd


def _replica_host_inputs(kind, env, tape_kb):
    """host_inputs of every copy's tape on the base instances, concatenated copy-major: masks (T,K·B,N), loads."""
    parts = [_host_inputs(kind, env, tape_kb[:, k]) for k in range(tape_kb.shape[1])]
    x, doh = parts[0][0], parts[0][1]
    return x, doh, np.concatenate([p[2] for p in parts], 1), np.concatenate([p[3] for p in parts], 1)


TRAIN_CASES = [("tsp", 20, 1185, 8, 31), ("vrp", 20, 517, 4, 32), ("irp", 20, 260, 3, 33), ("tsp", 50, 8200, 2, 34),
               ("tsp", 128, 40, 8, 35)]


@pytest.mark.parametrize("gemm_path", [0, 1], ids=["tcgen05", "simt"])
@pytest.mark.parametrize("kind,N,B,K,seed", TRAIN_CASES, ids=[f"{k}{n}_b{b}_k{kk}" for k, n, b, kk, _ in TRAIN_CASES])
def test_sample_train_step_vs_float64(kind, N, B, K, seed, gemm_path):
    """forward_samples(env, K) + backward(advantage / (K·B)): every element of every .grad against float64 autograd."""
    from oracle import policy_oracle as po

    model, env, wts, sd = _sample_train_step(kind, N, B, K, None, gemm_path, seed)
    ctx = model.last_rollout
    tape_kb = ctx["tape"].cpu().numpy()
    T = tape_kb.shape[0]
    logp_gpu = ctx["logp"].reshape(-1).detach().clone()
    saved = ctx["enc_saved"]
    model.zero_grad()
    model.backward(wts)
    dev = wts.device
    x, doh, masks, loads = _replica_host_inputs(kind, env, tape_kb)
    partners = torch.cat([_partners(B, B) + k * B for k in range(K)])
    x, doh, tape, masks, loads, partners = _device_inputs(x, doh, tape_kb.reshape(T, K * B), masks, loads, partners,
                                                          kind, dev)
    names = {n for n, _ in model.named_parameters()}
    for k in names:
        sd[k].requires_grad_(True)
    h = po.encoder_forward(sd, x, doh, train=True, relu=_kernel_gate(saved, B, N))
    del saved
    dh = torch.zeros((K * B,) + tuple(h.shape[1:]), dtype=F64, device=dev)
    logp = _decoder_reference(sd, h.detach().repeat(K, 1, 1), tape, masks, loads, partners, wts.reshape(-1),
                              lambda sl, g: dh[sl].copy_(g))
    h.backward(dh.view(K, B, *h.shape[1:]).sum(0))
    _check_logp(logp, logp_gpu, T)
    ref = {k: sd[k].grad for k in names if sd[k].grad is not None}
    gscale = max(g.abs().max().item() for g in ref.values())
    assert len(ref) >= 44
    _compare([(n, p.grad) for n, p in model.named_parameters()], ref, TOL, gscale,
             f"{kind}{N} B={B} K={K} path={gemm_path}")


# ------------------------------------------------------------------------------------------------ 4. vs replicated env
REP_CASES = [("tsp", 20, 517, 4, 41), ("vrp", 20, 260, 3, 42), ("irp", 20, 130, 3, 43)]


@pytest.mark.parametrize("kind,N,B,K,seed", REP_CASES, ids=[f"{k}{n}_b{b}_k{kk}" for k, n, b, kk, _ in REP_CASES])
def test_same_update_as_replicated_env(kind, N, B, K, seed):
    from agents.graph_encoder import run_encoder

    Env, Agent = _cls(kind)
    model = Agent(seed=seed).model
    model.train()
    twin, once = deepcopy(model), deepcopy(model)
    env = Env(N, B, 0, seed=seed, instance_rng="philox")
    torch.manual_seed(seed)
    _, logp = model.forward_samples(env, K)
    ctx = model.last_rollout
    T = ctx["steps"]
    tape = ctx["tape"].reshape(T, K * B).cpu().numpy()
    gen = torch.Generator(device=logp.device).manual_seed(seed)
    wts = torch.randn((K, B), generator=gen, device=logp.device) / (K * B)
    model.zero_grad()
    model.backward(wts)
    # today's train step on the copy-major replicated env, teacher-forced along the same tapes
    env_rep = Env(N, K * B, 0, seed=seed, instance_rng="philox")
    env_rep._xy.copy_(env._xy.repeat(K, 1, 1))
    env_rep._depot.copy_(env._depot.repeat(K))
    env_rep._demand.copy_(env._demand.repeat(K, 1))
    env_rep.restart_episode()
    twin.coupling = B
    _, logp_rep = twin(env_rep, rollout=False, tape=tape)
    assert twin.last_rollout["steps"] == T
    assert float((logp_rep - logp.reshape(-1)).abs().max()) <= 1e-4 * T
    twin.zero_grad()
    twin.backward(wts.reshape(-1))
    ref = {n: p.grad.to(F64) for n, p in twin.named_parameters() if p.grad is not None}
    gscale = max(g.abs().max().item() for g in ref.values())
    _compare([(n, p.grad) for n, p in model.named_parameters()], ref, TOL, gscale, f"{kind}{N} B={B} K={K} vs replicated")
    # running statistics: one train-mode encoder pass over the base batch
    run_encoder(once.encoder, env=env, depot=env._depot if once._USES_DEPOT_EMBED else None,
                gemm_path=once.encoder.gemm_path, save=True)
    got, want = dict(model.encoder.named_buffers()), dict(once.encoder.named_buffers())
    assert set(got) == set(want) and len(got) == 18
    for n in got:
        assert torch.equal(got[n], want[n]), n


# ------------------------------------------------------------------------------------------------ 5. agent, arguments, memory
def test_agent_train_with_samples(tmp_path):
    from agents import TSPAgent
    from gym_vrp.envs import TSPEnv

    agent = TSPAgent(seed=5, csv_path=str(tmp_path / "log.csv"))
    env = TSPEnv(12, 64, 0, seed=5, instance_rng="philox")
    bns = [m for m in agent.model.modules() if isinstance(m, torch.nn.BatchNorm1d)]
    before = [int(m.num_batches_tracked) for m in bns]
    w0 = agent.model.decoder._kp.weight.detach().clone()
    agent.train(env, epochs=2, samples=4, check_point_dir=str(tmp_path / "ck") + "/")
    with open(tmp_path / "log.csv") as f:
        rows = list(csv.reader(f))
    assert rows[0] == ["Epoch", "Loss", "Cost", "Advantage", "Time"] and len(rows) == 3
    assert all(np.isfinite(float(x)) for r in rows[1:] for x in r)
    assert [int(m.num_batches_tracked) for m in bns] == [b + 2 for b in before]
    assert not torch.equal(agent.model.decoder._kp.weight, w0), "no update"
    loss_m, loss_b, logp = agent.step(env, (False, True), samples=4)
    assert loss_m.shape == loss_b.shape == logp.shape == (4, 64)


def test_argument_checks():
    import vrpx
    from agents import TSPAgent
    from gym_vrp.envs import TSPEnv

    agent = TSPAgent(seed=1)
    model = agent.model
    env = TSPEnv(10, 12, 0, seed=1, instance_rng="philox")
    model.train()
    for K in (0, -1):
        with pytest.raises(ValueError, match="at least 1"):
            agent.train(env, epochs=1, samples=K)
        with pytest.raises(ValueError, match="at least 1"):
            model.forward_samples(env, K)
    model.coupling = 5   # does not divide B = 12
    with pytest.raises(ValueError, match="divisor"):
        model.forward_samples(env, 2)
    model.coupling = None
    with pytest.raises(ValueError, match="N <= 3"):
        agent.train(TSPEnv(3, 4, 0, seed=1, instance_rng="philox"), epochs=1, samples=2)
    with pytest.raises(ValueError, match="N <= 3"):
        model.forward_samples(TSPEnv(3, 4, 0, seed=1, instance_rng="philox"), 2)
    model.forward_samples(env, 3)
    for bad in (torch.zeros(12, device=env._device), torch.zeros(2, 12, device=env._device)):
        with pytest.raises(ValueError, match=r"\(K, B\)"):
            model.backward(bad)
    with pytest.raises(ValueError, match=r"\(K, B\)"):
        agent.policy_gradient_step(torch.zeros(36, device=env._device), torch.zeros(36, device=env._device), samples=3)
    # no trace: an eval-mode (or no-grad) rollout records nothing for the backward
    model.eval()
    model.forward_samples(env, 3)
    with pytest.raises(vrpx.VrpxError, match="no rollout recorded"):
        model.backward(torch.zeros(3, 12, device=env._device))
    # the C entry: a NULL trace, K < 1, a coupling that crosses copies, Bb·K != env->B
    model.train()
    with torch.no_grad():
        h = torch.zeros((12, 10, 128), device=env._device)
        out = model.decoder.rollout_samples(env, h, 3, seed=1, save_for_backward=True)
    L = vrpx.lib()
    view, dev = out["saved"]["replicas"], env._device
    irp = False
    w = model.decoder.packed(irp, dev)
    tens = model.decoder._packed[irp].tensors
    m_n, al_n = tens["m_t"].t().contiguous(), tens["al_t"].t().contiguous()
    wb = vrpx.DecoderBwdWeights(m_n.data_ptr(), al_n.data_ptr())
    z = lambda *s: torch.zeros(s, dtype=torch.float32, device=dev)
    g = [z(36, 10, 128), z(36, 1024), z(36, 1024), None, z(128, 1024), z(1024, 128), z(128)]
    gs = vrpx.DecoderGrads(*[None if t is None else t.data_ptr() for t in g])
    sv = out["saved"]
    trace = vrpx.RolloutTrace(sv["mask_hist"].data_ptr(), sv["load_hist"].data_ptr(), sv["qg0"].data_ptr())
    tape = out["tape"].reshape(out["steps"], 36).contiguous()
    wts = z(36)
    nbytes = int(L.vrpx_decoder_backward_workspace_bytes(36, 10))
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)

    def call(Bb=12, K=3, G=12, tr=trace):
        return L.vrpx_decoder_backward_samples(C.byref(view), C.byref(w), C.byref(wb), vrpx.ptr(h), Bb, K, vrpx.ptr(tape),
                                               out["steps"], G, C.byref(tr) if tr is not None else None, vrpx.ptr(sv["qg"]),
                                               vrpx.ptr(wts), C.byref(gs), vrpx.ptr(ws), nbytes, vrpx.stream_ptr(dev))

    ERR_ARG = -1
    assert call(tr=None) == ERR_ARG
    assert call(tr=vrpx.RolloutTrace(None, None, sv["qg0"].data_ptr())) == ERR_ARG
    assert call(K=0) == ERR_ARG
    assert call(Bb=13) == ERR_ARG
    assert call(G=36) == ERR_ARG   # divides Bb·K but not Bb: partners would cross copies
    assert call(G=5) == ERR_ARG
    assert call() == 0, L.vrpx_last_error()
    torch.cuda.synchronize()


# Peak allocated memory of one K-sample train step (forward_samples + backward) at TSP-50 x 8,192, K = 8, above what is
# allocated before it: 12.08 GiB measured on a B200 (1000 W); the bound leaves 10 % for allocator rounding and workspace
# changes.  The same step on the K-fold replicated env keeps 56 GiB of saved encoder activations alone.
PEAK_GIB_BOUND = 13.3


def test_peak_memory_tsp50_b8192_k8():
    from agents import TSPAgent
    from gym_vrp.envs import TSPEnv

    N, B, K = 50, 8192, 8
    model = TSPAgent(seed=9).model
    model.train()
    env = TSPEnv(N, B, 0, seed=9, instance_rng="philox")
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    torch.manual_seed(9)
    loss, logp = model.forward_samples(env, K)
    model.zero_grad()
    model.backward((loss - loss.mean()).detach() / (K * B))
    torch.cuda.synchronize()
    peak = (torch.cuda.max_memory_allocated() - base) / 2 ** 30
    print(f"\n[TSP-50 B={B} K={K}] peak {peak:.2f} GiB above {base / 2 ** 30:.2f} GiB (bound {PEAK_GIB_BOUND} GiB)")
    assert peak <= PEAK_GIB_BOUND
    assert all(bool(torch.isfinite(p.grad).all()) for p in model.parameters() if p.grad is not None)
