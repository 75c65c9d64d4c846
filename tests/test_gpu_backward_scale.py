"""The REINFORCE backward (csrc/decoder_bwd.cu, csrc/encoder_bwd.cu, vrpx/backward.py) against float64 torch autograd
at batch sizes that reach its large-batch code paths.  tests/test_gpu_backward.py and
test_full_gradient_tensors_vs_oracle_autograd run at B <= 32, where `k_decoder_bwd` is one CTA, every glimpse-mask
partner row lies in the instance's own 32-row tile and the weight gradients stay on the warp-level GEMMs.  Here:

* B = 9477 / 8200: 297 / 257 tiles of 32 instances on 148 CTAs (grid-stride tile loop, cross-CTA `red.global.add`
  of the step-weight gradients, a ragged last tile of 5 / 8 rows), partners (8b + h) mod G in far tiles, a coupling
  group G = 729 that is not a multiple of 32, and R = B*N >= 8192 rows, so the weight and bias gradients of the encoder
  and the per-episode ag_t / af_t products run on `k_gemm_tn_tc` (+ its `colsum_A` bias sums);
* C4 itself (TSP-50 x 65,536, the train step of bench.py): every element of dL/dh and of the decoder gradients, and
  the encoder gradients through directional derivatives (forward mode), at train-step gradient magnitudes.

The reference is the pinned oracle (oracle/policy_oracle.py) evaluated in float64 on the GPU with the model's f32
weights and f32-rounded observations, teacher-forced along the kernel's own sampled tape, with loss
sum_b wts_b * log p_b and wts = advantage / B against a greedy baseline.  Its masks and loads are rebuilt on the host
by stepping the env oracle along the tape (the kernel's saved mask history is not read).  The decoder loss is
separable over instances once h is fixed, so the reference runs it in instance chunks and sums the gradients."""
import math
import time

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

F64 = torch.float64
# Per-tensor bars relative to the tensor's largest element (the convention of test_full_gradient_tensors_vs_oracle_autograd);
# FLOOR * (the model's largest gradient element) covers the mathematically-zero gradients (encoder out_proj.bias and
# ff.2.bias in front of a train-mode BatchNorm, key biases): rounding noise on both sides.  Each bar is about 4-5 x the
# largest error measured on a B200 (1000 W), the same for both gemm_paths:
TOL = 5e-4        # whole train step, every parameter: measured 1.1e-4 (tcgen05) / 8.7e-5 (SIMT)
C4_DEC_TOL = 1e-3  # C4 decoder parameters: measured 2.3e-4 on both paths (the key-bias part of in_proj_bias)
DH_TOL = 5e-5     # C4 dL/dh, relative to its largest element: measured 1.0e-5 / 8.4e-6
DIR_TOL = 5e-4    # C4 encoder, |<g,v> - jvp| / |g|: measured 1.1e-4 / 2.6e-5
FLOOR = 3e-5
# reference chunk: instances x nodes x steps per float64 decoder chunk (about 8 GB of saved activations)
DEC_ROWS = 1 << 20
# ReLU pre-activations within GATE_BAND * max|pre| of zero take the kernel's gate (see _kernel_gate)
GATE_BAND = 1e-5


def _cls(kind):
    from agents import IRPAgent, TSPAgent, VRPAgent
    from gym_vrp.envs import IRPEnv, TSPEnv, VRPEnv

    return {"tsp": (TSPEnv, TSPAgent), "vrp": (VRPEnv, VRPAgent), "irp": (IRPEnv, IRPAgent)}[kind]


def _sampled_train_step(kind, N, B, G, gemm_path, seed):
    """A greedy baseline and a sampled train-mode rollout of a seed-initialised model on Philox instances.  Returns
    (model, env, wts = advantage / B, float64 copy of the weights taken before the forward)."""
    Env, Agent = _cls(kind)
    model = Agent(seed=seed).model
    model.coupling = G
    model.encoder.gemm_path = gemm_path
    sd = {k: v.detach().to(F64).clone() for k, v in model.state_dict().items()}
    model.eval()
    with torch.no_grad():
        loss_b, _ = model(Env(N, B, 0, seed=seed, instance_rng="philox"), rollout=True)
    model.train()
    env = Env(N, B, 0, seed=seed, instance_rng="philox")
    torch.manual_seed(seed)
    loss_m, _ = model(env, rollout=False)
    wts = ((loss_m - loss_b) * -1 / B).detach()
    return model, env, wts, sd


def _host_inputs(kind, env, tape):
    """Instances, the f32-rounded encoder features, the depot one-hot, and every instance's mask (T,B,N) uint8 and f32
    load (T,B) before every step of `tape`, from the env oracle replayed at the full batch."""
    from oracle.env_oracle import EnvOracle

    s = env.sampler
    xy, depot, demand = s.get_graph_positions(), s.get_depots()[:, 0], s.get_demands()[:, :, 0]
    B, N = xy.shape[:2]
    x = torch.tensor(xy, dtype=torch.float32)   # the encoder reads the f32 observation (graph_tsp_agent.py:72)
    if kind == "irp":
        x = torch.cat([x, torch.tensor(demand, dtype=torch.float32)[:, :, None]], -1)
    doh = None
    if kind != "tsp":
        doh = torch.zeros(B, N, dtype=torch.bool)
        doh[torch.arange(B), torch.as_tensor(depot)] = True
    orc = EnvOracle(kind, xy, depot, demand)
    T = tape.shape[0]
    masks = np.empty((T, B, N), dtype=np.uint8)
    loads = np.empty((T, B), dtype=np.float32)
    for t in range(T):
        masks[t] = orc.generate_mask()
        loads[t] = orc.load
        done = orc.step(tape[t].astype(np.int64)[:, None], observe=False)[2]
    assert done, "the kernel's tape does not finish the episode on the env oracle"
    return x, doh, masks, loads


def _partners(B, G):
    """(B, 8): the instance whose mask attention row (b, head) adds, g0 + ((b - g0) * 8 + head) mod G with g0 the first
    instance of b's coupling group (graph_decoder.py:93-94, `mask.repeat(H, 1)` within a group of G instances)."""
    b = torch.arange(B)[:, None]
    g0 = b // G * G
    return g0 + ((b - g0) * 8 + torch.arange(8)[None, :]) % G


def _teacher_forced_logp(sd, h, tape, masks, loads, partners, sl):
    """Sum over steps of log p(a_t) for the instances `sl` of the batch, as a function of their embeddings h (S,N,E)
    and the decoder weights in sd.  tape (T,B) long, masks (T,B,N) uint8, loads (T,B) or None, partners (B,8) long."""
    from oracle import policy_oracle as po

    S, N, E = h.shape
    first = sd["decoder._first_node"].reshape(1, E).repeat(S, 1)
    last = sd["decoder._last_node"].reshape(1, E).repeat(S, 1)
    ar = torch.arange(S, device=h.device)
    total = torch.zeros(S, dtype=h.dtype, device=h.device)
    for t in range(tape.shape[0]):
        mt = masks[t]
        u = po.decoder_logits(sd, h, mt[sl].to(h.dtype), first, last,
                              None if loads is None else loads[t, sl].to(h.dtype),
                              glimpse_mask=mt[partners[sl]].to(h.dtype))
        a = tape[t, sl]
        total = total + u.gather(1, a[:, None])[:, 0] - torch.logsumexp(u, dim=-1)
        last = h[ar, a]
        if t == 0:
            first = last
    return total


def _decoder_reference(sd, h, tape, masks, loads, partners, wts, visit):
    """Backward of sum_b wts_b log p_b through the decoder, chunk by chunk over instances.  visit(slice, dL/dh of the
    chunk) is called per chunk; the decoder parameter gradients accumulate in sd's .grad.  Returns log p (B,)."""
    B, N = h.shape[:2]
    chunk = max(64, DEC_ROWS // (N * tape.shape[0]))
    logp = torch.empty(B, dtype=F64, device=h.device)
    for i in range(0, B, chunk):
        sl = slice(i, min(B, i + chunk))
        hc = h[sl].detach().clone().requires_grad_(True)
        lp = _teacher_forced_logp(sd, hc, tape, masks, loads, partners, sl)
        (lp * wts[sl].to(F64)).sum().backward()
        logp[sl] = lp.detach()
        visit(sl, hc.grad)
    return logp


def _kernel_gate(saved, B, N):
    """relu hook for policy_oracle.encoder_forward: the float64 sign of the pre-activation decides the ReLU gate, except
    within GATE_BAND of zero, where the f32 kernel's own saved activation F (encoder_bwd.cu: per layer l at
    R*384 + l*R*1408 + R*768 of the saved block, [R][512]) decides.  There the sign is not determined by f32 inputs, and
    each disagreement moves a ReLU weight gradient by ~1/sqrt(R) of its largest element: 2e-3 ... 5e-3 for a handful of
    flips at R = 80,000 rows.  The band holds a few thousandths of a percent of the elements, so a wrong saved F stays
    visible through the gradients that use it (dW2 = dy2^T F and the backward's own gate)."""
    R = B * N

    def relu(pre, layer, first):
        b = pre.shape[0]
        o = R * 384 + layer * R * 1408 + R * 768 + first * N * 512
        on_kernel = saved[o:o + b * N * 512].view(b, N, 512) > 0
        x = pre.detach()
        on = torch.where(x.abs() <= GATE_BAND * x.abs().max(), on_kernel, x > 0)
        return pre * on.to(pre.dtype)

    return relu


def _device_inputs(x, doh, tape, masks, loads, partners, kind, dev):
    return (x.to(dev, F64), None if doh is None else doh.to(dev), torch.as_tensor(tape.astype(np.int64), device=dev),
            torch.from_numpy(masks).to(dev), torch.from_numpy(loads).to(dev) if kind == "irp" else None, partners.to(dev))


def _check_logp(logp_ref, logp_gpu, T):
    """The kernel's sampled log-probs are the teacher-forced ones of the reference: the mask history is the same."""
    d = (logp_ref - logp_gpu.to(F64)).abs()
    bar = 1e-5 * logp_ref.abs() + 1e-5 * T
    assert bool((d <= bar).all()), ("log-prob sums differ from the float64 replay", float(d.max()))


def _compare(named, ref, tol, gscale, what):
    """Every element of every gradient: |got - ref| <= tol * max|ref| + FLOOR * gscale.  Returns the largest error
    relative to its tensor's largest element over the tensors above the floor, and the largest error over gscale."""
    bad, rel, flo = [], (0.0, None), 0.0
    for name, got in named:
        g_ref = ref.get(name)
        if g_ref is None:
            assert got is None or got.abs().max().item() < 1e-6 * gscale, (what, name, "reference has no gradient")
            continue
        assert got is not None and got.shape == g_ref.shape, (what, name)
        err = (got.to(F64) - g_ref).abs().max().item()
        sc = g_ref.abs().max().item()
        if err > tol * sc + FLOOR * gscale:
            bad.append((name, err, sc))
        if tol * sc > FLOOR * gscale:   # the relative bar, not the floor, decides for this tensor
            rel = max(rel, (err / sc, name), key=lambda r: r[0])
        flo = max(flo, err / gscale)
    print(f"\n[{what}] max error / tensor max {rel[0]:.3g} ({rel[1]}), max error / model max {flo:.3g}")
    assert not bad, (what, gscale, bad)
    return rel[0]


# ------------------------------------------------------------------------------------------------ 1. whole train step
SCALE_CASES = [("tsp", 20, 9477, 9477, 11), ("tsp", 20, 9477, 729, 12), ("vrp", 20, 9477, 9477, 13),
               ("irp", 20, 9477, 9477, 14), ("tsp", 50, 8200, 8200, 15)]


@pytest.mark.parametrize("gemm_path", [0, 1], ids=["tcgen05", "simt"])
@pytest.mark.parametrize("kind,N,B,G,seed", SCALE_CASES, ids=[f"{k}{n}_b{b}_g{g}" for k, n, b, g, _ in SCALE_CASES])
def test_train_step_gradients_vs_float64(kind, N, B, G, seed, gemm_path):
    """model(env, rollout=False) + model.backward(advantage / B): every element of every parameter's .grad against
    torch autograd of the float64 teacher-forced loss (train-mode BatchNorm over the whole batch)."""
    from oracle import policy_oracle as po

    model, env, wts, sd = _sampled_train_step(kind, N, B, G, gemm_path, seed)
    ctx = model.last_rollout
    tape_np = ctx["tape"].cpu().numpy()
    logp_gpu = ctx["logp"].detach().clone()
    saved = ctx["enc_saved"]
    model.zero_grad()
    model.backward(wts)
    dev = wts.device
    x, doh, masks, loads = _host_inputs(kind, env, tape_np)
    x, doh, tape, masks, loads, partners = _device_inputs(x, doh, tape_np, masks, loads, _partners(B, G), kind, dev)
    names = {n for n, _ in model.named_parameters()}
    for k in names:
        sd[k].requires_grad_(True)
    h = po.encoder_forward(sd, x, doh, train=True, relu=_kernel_gate(saved, B, N))
    del saved
    dh = torch.zeros_like(h)
    logp = _decoder_reference(sd, h, tape, masks, loads, partners, wts, lambda sl, g: dh[sl].copy_(g))
    h.backward(dh)
    _check_logp(logp, logp_gpu, tape.shape[0])
    ref = {k: sd[k].grad for k in names if sd[k].grad is not None}
    gscale = max(g.abs().max().item() for g in ref.values())
    got = [(n, p.grad) for n, p in model.named_parameters()]
    assert len(ref) >= 44
    _compare(got, ref, TOL, gscale, f"{kind}{N} B={B} G={G} path={gemm_path}")


# ------------------------------------------------------------------------------------------------ 2./3. C4 shape
C4 = ("tsp", 50, 65536, 21)
ENC_CHUNK = 4096   # instances per attention / feed-forward chunk of the float64 encoder (BatchNorm spans the batch)


@pytest.fixture(scope="module")
def c4():
    """One C4 train-step forward (TSP-50 x 65,536, whole-batch coupling, production GEMM path), then the decoder
    backward and the encoder backward once per gemm_path on the same saved state.  Both encoder backwards start from a
    copy of the path-0 dL/dh (the call overwrites it), so one reference serves both.  The saved encoder activations
    (about 60 GB) are released before any reference work."""
    from vrpx import backward as bw

    kind, N, B, seed = C4
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    t0 = time.time()
    model, env, wts, sd = _sampled_train_step(kind, N, B, B, 0, seed)
    ctx = model.last_rollout
    model.last_rollout = None
    out = {"wts": wts, "sd": sd, "h": ctx["emb"], "logp": ctx["logp"].detach().clone(), "dH": {}, "dec": {}, "enc": {}}
    for path in (0, 1):
        model.zero_grad()
        out["dH"][path] = bw.decoder_backward(model.decoder, env, ctx["emb"], ctx, wts, gemm_path=path)
        out["dec"][path] = {"decoder." + n: p.grad for n, p in model.decoder.named_parameters()}
    for path in (0, 1):
        model.zero_grad()
        bw.encoder_backward(model.encoder, env, ctx["depot"], ctx["enc_saved"], out["dH"][0].clone(), gemm_path=path)
        out["enc"][path] = {"encoder." + n: p.grad for n, p in model.encoder.named_parameters()}
    torch.cuda.synchronize()
    print(f"\n[C4] train-step forward + 2 x (decoder + encoder backward): {time.time() - t0:.1f} s, peak "
          f"{torch.cuda.max_memory_allocated() / 2 ** 30:.1f} GiB")
    tape_np = ctx["tape"].cpu().numpy()
    del ctx, model
    torch.cuda.empty_cache()
    out["host"] = _host_inputs(kind, env, tape_np) + (tape_np,)
    yield out
    print(f"\n[C4] peak allocated over the module: {torch.cuda.max_memory_allocated() / 2 ** 30:.1f} GiB")


def test_c4_decoder_backward_vs_float64(c4):
    """C4: every element of dL/dh (65,536 x 50 x 128) and of every decoder parameter gradient, both gemm_paths."""
    kind, N, B, _ = C4
    x, doh, masks, loads, tape_np = c4["host"]
    dev = c4["h"].device
    _, _, tape, masks, loads, partners = _device_inputs(x, doh, tape_np, masks, loads, _partners(B, B), kind, dev)
    sd = {k: v.clone().requires_grad_(k.startswith("decoder.") and v.is_floating_point()) for k, v in c4["sd"].items()}
    h = c4["h"].to(F64)
    err = {0: 0.0, 1: 0.0}
    scale = [0.0]

    def visit(sl, g):
        scale[0] = max(scale[0], g.abs().max().item())
        for path in (0, 1):
            err[path] = max(err[path], (c4["dH"][path][sl].to(F64) - g).abs().max().item())

    logp = _decoder_reference(sd, h, tape, masks, loads, partners, c4["wts"], visit)
    _check_logp(logp, c4["logp"], tape.shape[0])
    print(f"\n[C4 dL/dh] max error / max element: path 0 {err[0] / scale[0]:.3g}, path 1 {err[1] / scale[0]:.3g}")
    for path in (0, 1):
        assert err[path] <= DH_TOL * scale[0], (path, err[path], scale[0])
    ref = {k: v.grad for k, v in sd.items() if v.grad is not None}
    gscale = max(g.abs().max().item() for g in ref.values())
    assert len(ref) >= 8
    for path in (0, 1):
        _compare(c4["dec"][path].items(), ref, C4_DEC_TOL, gscale, f"C4 decoder path={path}")


def test_c4_encoder_backward_directional_vs_float64(c4):
    """C4: for every encoder parameter tensor and three Gaussian directions v, <g, v> of the library's gradient equals
    the float64 forward-mode derivative (torch.func.jvp) of <dL/dh, encoder(theta)> along v, dL/dh being the library's
    own (fixed cotangent): |<g,v> - jvp| <= tol * |g| + FLOOR * max|g| * sqrt(numel) (the elementwise floor for the
    mathematically-zero gradients, as a norm)."""
    from oracle import policy_oracle as po

    x = c4["host"][0].to(c4["h"].device, F64)
    sd = c4["sd"]
    dH = c4["dH"][0].to(F64).reshape(-1)
    gen = torch.Generator(device=x.device).manual_seed(7)
    names = list(c4["enc"][0])
    gscale = {p: max(g.abs().max().item() for g in c4["enc"][p].values()) for p in (0, 1)}
    bad, worst = [], {0: (0.0, None), 1: (0.0, None)}
    t0 = time.time()
    for name in names:

        def loss(w, name=name):
            return torch.dot(po.encoder_forward({**sd, name: w}, x, None, train=True, chunk=ENC_CHUNK).reshape(-1), dH)

        for _ in range(3):
            v = torch.randn(sd[name].shape, generator=gen, dtype=F64, device=x.device)
            _, jv = torch.func.jvp(loss, (sd[name],), (v,))
            jv = jv.item()
            for path in (0, 1):
                g = c4["enc"][path][name].to(F64)
                gv = torch.dot(g.reshape(-1), v.reshape(-1)).item()
                gn = g.norm().item()
                err = abs(gv - jv)
                if err > DIR_TOL * gn + FLOOR * gscale[path] * math.sqrt(g.numel()):
                    bad.append((path, name, gv, jv, gn))
                if DIR_TOL * gn > FLOOR * gscale[path] * math.sqrt(g.numel()):
                    worst[path] = max(worst[path], (err / gn, name), key=lambda r: r[0])
    print(f"\n[C4 encoder] {len(names)} tensors x 3 directions in {time.time() - t0:.1f} s; max |<g,v> - jvp| / |g|: "
          f"path 0 {worst[0][0]:.3g} ({worst[0][1]}), path 1 {worst[1][0]:.3g} ({worst[1][1]})")
    assert not bad, bad
