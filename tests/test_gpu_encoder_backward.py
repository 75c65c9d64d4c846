"""The encoder backward (csrc/encoder_bwd.cu, csrc/attention_bwd.cu, the gemm_tn_accumulate weight gradients,
vrpx/backward.py::encoder_backward) against float64: stage by stage, end to end, and the attention backward at every
node count.

The test hook vrpx_debug_encoder_backward_stages runs the production launches and copies the eight gradients each layer
holds (dOUT, dY2, dPRE, dH1, dY1, dATT, dQKV, dX; include/vrpx.h) into a buffer.  One float64 layer-backward function,
`layer_backward64`, serves two modes:
* stage by stage: every stage from the kernel's own input to it, and every parameter gradient from the kernel's own stage
  gradients (dW2 = dY2^T F, dW1 = dPRE^T H1, dW_o = dY1^T ATT, dW_in = dQKV^T H[l], BatchNorm gamma / beta from dOUT / dH1
  and the saved statistics), so that each bar measures one kernel;
* end to end: the production route (no hook) against the same function chained in float64 from dL/dh.
Both are linearised at the kernel's saved activations: the ReLU gate is the saved F > 0 and the BatchNorm backward uses
the saved (mean, invstd).  That removes the forward's error and the gate flips that set the 5e-4 of the whole-train-step
tests, and checks every element of every encoder gradient.

Stage tensors are compared relative to the tensor's largest element.  Every parameter gradient is a sum over the R
rows, and each of its elements is compared against the sum of its terms' magnitudes: sum_r |dY_rc| |X_rk| for a weight
gradient dY^T X, sum_r |dY_rc| for a bias.  Two of the biases (ff.2.bias, out_proj.bias) and the key third of
in_proj_bias are zero in exact arithmetic, and at layer 0, whose inputs H[0] and ATT have nearly constant columns, the
out- and in-projection weight gradients cancel to about 1e-3 of their terms: against their own largest element the f32
sums there sat at 7.7e-4 on both gemm_paths (VRP-65 x 126), while against their terms they sit at 1e-5 like every other
weight gradient.

The upstream dL/dh is heavy-tailed (Gaussian x per-row 10^U(-4, 0) x 1e-6), so the power-of-two gain of
vrpx/backward.py::_grad_gain is far from 1; the float64 reference runs in the gained scale.  TSP-20 x 9477 also runs on
the real decoder dL/dh of a sampled rollout."""
import time

import pytest
import torch
from test_gpu_encoder_train import _attention64, _chunks, _encoder, saved_stages

pytestmark = pytest.mark.gpu

F64 = torch.float64
E, FF = 128, 512
STAGES = (("dout", 128), ("dy2", 128), ("dpre", 512), ("dh1", 128), ("dy1", 128), ("datt", 128), ("dqkv", 384),
          ("dx", 128))
STAGE_FLOATS = sum(w for _, w in STAGES)   # 1,664 per row and layer
ROWS = 1 << 18                             # rows per float64 chunk of the reference
# Bars, each 2-4 x the largest value measured over all cases and both gemm_paths on a B200 (1000 W power limit).
# Stage by stage, max |kernel - float64| relative to the (layer, stage) tensor's largest element:
STAGE_TOL = {"dy2": 4e-7,    # BN2 backward: measured 1.5e-7
             "dpre": 2e-6,   # ReLU-gate GEMM: 6.2e-7
             "dh1": 1.5e-6,  # residual GEMM, K = 512: 4.8e-7
             "dy1": 5e-7,    # BN1 backward: 1.6e-7
             "datt": 2e-6,   # out-projection data gradient: 6.2e-7
             "dqkv": 3e-5,   # attention backward: 1.1e-5 (mma.sync, TSP-128 x 64) / 3.1e-6 (fp32 SIMT)
             "dx": 3e-6}     # residual GEMM, K = 384: 9.8e-7
# parameter gradients from the kernel's own stage gradients, per element against the sum of its terms' magnitudes
PARAM_TOL = 3e-5   # measured 1.2e-5 (in_proj_weight on k_gemm_tn_mma, TSP-128 x 7); 1.7e-6 on k_gemm_tn_tc
# end to end (chained float64 from dL/dh): every element of every .grad, as above: measured 1.0e-5 from R = 8190 rows
# up (C4 2.1e-7).  Below 1024 rows a handful of heavy-tailed rows carry each element's sum of magnitudes, and the
# stage rounding of the other rows, about 1e-7 of the tensor's largest element, lands on top of it: measured 1.3e-3
# (TSP-8 x 2, R = 16), 8.7e-4 (TSP-64 x 3).
E2E_PARAM_TOL = 3e-5
E2E_PARAM_TOL_FEW_ROWS = 3e-3
# the returned dL/d(embedding output), relative to its largest element: measured 2.7e-6
E2E_DEMB_TOL = 8e-6
# a hook call against a plain call on the same inputs (float atomics in the weight-gradient flush), relative to the
# encoder's largest gradient element
HOOK_TOL = 5e-6   # measured 1.7e-6 (IRP-43 x 191, k_gemm_tn_tc); 0 at VRP-33 x 5
# attention backward, dQ / dK / dV each relative to its largest element
ATTN_TOL = 4e-5   # measured 1.4e-5 (sharp, fp32 SIMT, N = 120) / 7.0e-6 (sharp, mma.sync, N = 13); randn 2.1e-6


def backward_stages(buf, B, N, layers):
    """Named views of the buffer vrpx_debug_encoder_backward_stages fills, for R = B*N rows: the selected layers in
    ascending order, each eight stage-major blocks (STAGES).  Returns {layer: {stage: (R, width) view}}."""
    R = B * N
    out, o = {}, 0
    for l in sorted(layers):
        out[l] = {}
        for name, width in STAGES:
            out[l][name] = buf[o:o + R * width].view(R, width)
            o += R * width
    return out


def _layers_of(mask):
    return [l for l in range(3) if mask >> l & 1]


def _env(kind, N, B, seed):
    from gym_vrp.envs import IRPEnv, TSPEnv, VRPEnv

    return {"tsp": TSPEnv, "vrp": VRPEnv, "irp": IRPEnv}[kind](N, B, 0, seed=seed, instance_rng="philox")


def _features(env, f):
    """float64 copies of the f32 node features the encoder reads from the env (R, f), and the depot rows (R,) bool or
    None (TSP)."""
    B, N = env.batch_size, env.num_nodes
    x = env._xy.reshape(B * N, 2).float()
    if f == 3:
        x = torch.cat([x, env._demand.reshape(B * N, 1).float()], 1)
    if env._KIND == 0:
        return x.to(F64), None
    isdep = torch.zeros(B * N, dtype=torch.bool, device=x.device)
    isdep[torch.arange(B, device=x.device) * N + env._depot.long()] = True
    return x.to(F64), isdep


def _upstream(R, seed):
    """Heavy-tailed dL/dh (R, 128) f32: Gaussian x per-row 10^U(-4, 0) x 1e-6."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    d = torch.randn(R, E, generator=g, device="cuda", dtype=F64)
    d *= 10.0 ** (-4.0 * torch.rand(R, 1, generator=g, device="cuda", dtype=F64))
    return (d * 1e-6).float()


def _params64(enc):
    return {n: p.detach().to(F64) for n, p in enc.named_parameters()}


def _bn_backward64(dout, y, stat, gamma, name, take):
    """BatchNorm backward with the saved (mean, invstd): dy = gamma invstd (dout - mean(dout) - xhat mean(dout xhat)).
    Returns dy (R, 128) and {weight: dgamma, bias: dbeta} as (gradient, sum of its terms' magnitudes)."""
    R = dout.shape[0]
    mean, invstd = stat[0].to(F64), stat[1].to(F64)
    s1 = torch.zeros(E, dtype=F64, device=dout.device)
    s2, a1, a2 = torch.zeros_like(s1), torch.zeros_like(s1), torch.zeros_like(s1)
    for sl in _chunks(R, ROWS):
        xh = (y[sl].to(F64) - mean) * invstd
        s1 += dout[sl].sum(0)
        s2 += (dout[sl] * xh).sum(0)
        a1 += dout[sl].abs().sum(0)
        a2 += (dout[sl] * xh).abs().sum(0)
    dy = torch.empty_like(dout)
    for sl in _chunks(R, ROWS):
        xh = (y[sl].to(F64) - mean) * invstd
        dy[sl] = take(name, sl, gamma * invstd * (dout[sl] - s1 / R - xh * (s2 / R)))
    return dy, {"weight": (s2, a2), "bias": (s1, a1)}


def layer_backward64(S, hin, P, gout, N, take):
    """float64 backward of one encoder layer (graph_encoder.py:183-198, train-mode BatchNorm), linearised at the kernel's
    saved activations.  S: the layer's saved block (saved_stages), hin: its input H[l] (R, 128); P: the layer's float64
    parameters by name inside the layer; gout: dL/d(layer output) (R, 128) float64.
    Every stage gradient passes through take(stage, rows, ref), which returns what the next stage continues from: the
    float64 `ref` itself (chained) or the kernel's own value of that stage (stage by stage).  Returns dL/d(layer input)
    (R, 128) and {parameter: (gradient, sum over rows of its terms' magnitudes)}: |dY|^T |X| for dW = dY^T X,
    sum_r |dY_rc| for a bias."""
    R = gout.shape[0]
    dev = gout.device
    grads = {}
    dy2, bn2 = _bn_backward64(gout, S["y2"], S["bn2"], P["bn2.norm.weight"], "dy2", take)
    grads.update({"bn2.norm." + k: v for k, v in bn2.items()})
    acc = {k: 0 for k in ("ff.2.weight", "ff.2.wabs", "ff.2.bias", "ff.2.abs", "ff.0.weight", "ff.0.wabs", "ff.0.bias",
                          "ff.0.abs")}
    dh1 = torch.empty_like(gout)
    for sl in _chunks(R, ROWS):
        d = dy2[sl]
        f = S["f"][sl].to(F64)
        acc["ff.2.weight"] = acc["ff.2.weight"] + d.T @ f
        acc["ff.2.wabs"] = acc["ff.2.wabs"] + d.abs().T @ f
        acc["ff.2.bias"] = acc["ff.2.bias"] + d.sum(0)
        acc["ff.2.abs"] = acc["ff.2.abs"] + d.abs().sum(0)
        dpre = take("dpre", sl, (d @ P["ff.2.weight"]) * (f > 0))
        h1 = S["h1"][sl].to(F64)
        acc["ff.0.weight"] = acc["ff.0.weight"] + dpre.T @ h1
        acc["ff.0.wabs"] = acc["ff.0.wabs"] + dpre.abs().T @ h1.abs()
        acc["ff.0.bias"] = acc["ff.0.bias"] + dpre.sum(0)
        acc["ff.0.abs"] = acc["ff.0.abs"] + dpre.abs().sum(0)
        dh1[sl] = take("dh1", sl, d + dpre @ P["ff.0.weight"])
    for k in ("ff.2", "ff.0"):
        grads[k + ".weight"] = (acc[k + ".weight"], acc[k + ".wabs"])
        grads[k + ".bias"] = (acc[k + ".bias"], acc[k + ".abs"])
    del dy2
    dy1, bn1 = _bn_backward64(dh1, S["y1"], S["bn1"], P["bn1.norm.weight"], "dy1", take)
    grads.update({"bn1.norm." + k: v for k, v in bn1.items()})
    del dh1
    wo, wi = "attention_layer.out_proj.weight", "attention_layer.in_proj_weight"
    z = lambda *s: torch.zeros(s, dtype=F64, device=dev)
    acc = {"wo": z(E, E), "wao": z(E, E), "bo": z(E), "ao": z(E), "wi": z(3 * E, E), "wai": z(3 * E, E), "bi": z(3 * E),
           "ai": z(3 * E)}
    dx = torch.empty_like(gout)
    for ib in _chunks(R // N, max(1, ROWS // N)):
        sl = slice(ib.start * N, ib.stop * N)
        d = dy1[sl]
        att = S["att"][sl].to(F64)
        acc["wo"] += d.T @ att
        acc["wao"] += d.abs().T @ att.abs()
        acc["bo"] += d.sum(0)
        acc["ao"] += d.abs().sum(0)
        datt = take("datt", sl, d @ P[wo])
        with torch.enable_grad():
            qkv = S["qkv"][sl].to(F64).requires_grad_(True)
            (dq,) = torch.autograd.grad(_attention64(qkv.view(-1, N, 3 * E)), qkv, datt.view(-1, N, E))
        dqkv = take("dqkv", sl, dq)
        x = hin[sl].to(F64)
        acc["wi"] += dqkv.T @ x
        acc["wai"] += dqkv.abs().T @ x.abs()
        acc["bi"] += dqkv.sum(0)
        acc["ai"] += dqkv.abs().sum(0)
        dx[sl] = take("dx", sl, d + dqkv @ P[wi])
    grads[wo] = (acc["wo"], acc["wao"])
    grads["attention_layer.out_proj.bias"] = (acc["bo"], acc["ao"])
    grads[wi] = (acc["wi"], acc["wai"])
    grads["attention_layer.in_proj_bias"] = (acc["bi"], acc["ai"])
    return dx, grads


def embed_backward64(g, x, isdep, f):
    """Gradients of node_embed (rows that are not a depot) and depot_embed (depot rows, features x, y) from dL/d(embedding
    output) g (R, 128) float64; x (R, f) float64.  Same return convention as layer_backward64."""
    R = g.shape[0]
    z = lambda *s: torch.zeros(s, dtype=F64, device=g.device)
    a = {"nw": z(E, f), "nwa": z(E, f), "nb": z(E), "na": z(E), "dw": z(E, 2), "dwa": z(E, 2), "db": z(E), "da": z(E)}
    for sl in _chunks(R, ROWS):
        gn, gd = g[sl], None
        if isdep is not None:
            m = isdep[sl, None]
            gn, gd = torch.where(m, 0.0, g[sl]), torch.where(m, g[sl], 0.0)
        a["nw"] += gn.T @ x[sl]
        a["nwa"] += gn.abs().T @ x[sl].abs()
        a["nb"] += gn.sum(0)
        a["na"] += gn.abs().sum(0)
        if gd is not None:
            a["dw"] += gd.T @ x[sl, :2]
            a["dwa"] += gd.abs().T @ x[sl, :2].abs()
            a["db"] += gd.sum(0)
            a["da"] += gd.abs().sum(0)
    out = {"node_embed.weight": (a["nw"], a["nwa"]), "node_embed.bias": (a["nb"], a["na"])}
    if isdep is not None:
        out.update({"depot_embed.weight": (a["dw"], a["dwa"]), "depot_embed.bias": (a["db"], a["da"])})
    return out


def _param_errors(got, ref):
    """{name: max over elements of |got - ref| / the sum of the element's terms' magnitudes}."""
    return {name: ((got[name].to(F64) - r).abs() / mag.clamp_min(1e-300)).max().item() for name, (r, mag) in ref.items()}


def _seed(N, B):
    return 11 * N + B


def _backward(kind, N, B, gemm_path, upstream="heavy", mask=None, plain_too=False):
    """The train-mode forward on a Philox env (run_encoder, save=True) and the encoder backward through
    bw.encoder_backward, with the stage hook when `mask` is given.  upstream "heavy": _upstream; "decoder": dL/dh of the
    decoder backward of a sampled rollout of the agent's model with this encoder.  Returns a dict."""
    from agents import IRPAgent, TSPAgent, VRPAgent
    from agents.graph_encoder import run_encoder
    from vrpx import backward as bw

    seed = _seed(N, B)
    enc = _encoder(kind, seed, gemm_path)
    env = _env(kind, N, B, seed)
    depot = env._depot if kind != "tsp" else None
    R = B * N
    if upstream == "heavy":
        _, saved = run_encoder(enc, env=env, depot=depot, gemm_path=gemm_path, save=True)
        dH = _upstream(R, seed)
    else:
        model = {"tsp": TSPAgent, "vrp": VRPAgent, "irp": IRPAgent}[kind](seed=seed).model
        model.encoder = enc
        model.train()
        torch.manual_seed(seed)
        loss, _ = model(env, rollout=False)
        ctx = model.last_rollout
        model.last_rollout = None
        wts = ((loss - loss.mean()) / B).detach()
        dH = bw.decoder_backward(model.decoder, env, ctx["emb"], ctx, wts, gemm_path=gemm_path).reshape(R, E).contiguous()
        saved = ctx["enc_saved"]
        del ctx
    gain = bw._grad_gain(dH)
    out = {"enc": enc, "env": env, "saved": saved, "dH": dH, "gain": gain, "N": N, "B": B}
    stages = None
    if mask is not None:
        stages = torch.full((len(_layers_of(mask)) * R * STAGE_FLOATS,), float("nan"), device=dH.device)
    enc.zero_grad(set_to_none=True)
    g = dH.clone()
    ret = bw.encoder_backward(enc, env, depot, saved, g, gemm_path=gemm_path, stages=stages,
                              stage_layers=mask if mask is not None else 0b111)
    assert ret is g
    out.update(demb=g, stages=stages, grads={n: p.grad.detach().clone() for n, p in enc.named_parameters()})
    if plain_too:
        enc.zero_grad(set_to_none=True)
        g2 = dH.clone()
        bw.encoder_backward(enc, env, depot, saved, g2, gemm_path=gemm_path)
        out.update(demb_plain=g2, grads_plain={n: p.grad.detach().clone() for n, p in enc.named_parameters()})
    torch.cuda.synchronize()
    return out


class _StageAcc:
    """max |kernel - float64| and max |float64| per (layer, stage) over row chunks."""

    def __init__(self):
        self.acc = {}

    def put(self, key, got, ref):
        e, s = self.acc.get(key, (0.0, 0.0))
        self.acc[key] = (max(e, (got - ref).abs().max().item()), max(s, ref.abs().max().item()))

    def rel(self):
        return {k: e / s for k, (e, s) in self.acc.items()}


def _layer_inputs(run, l):
    B, N = run["B"], run["N"]
    H, layers = saved_stages(run["saved"], B, N)
    P = {k[len(f"attention_layers.{l}."):]: v for k, v in _params64(run["enc"]).items()
         if k.startswith(f"attention_layers.{l}.")}
    return layers[l], H[l], P


def _grad_key(l, name):
    return name if l is None else f"attention_layers.{l}.{name}"


# (kind, N, B): R = 6 / 16 (BatchNorm backward at tiny R); NJJ = 3 with NK8 = 5 / 6; NK8 = 8 / 9 (launch bounds 3 -> 1
# CTA per SM); NK8 = 11 / 12 (NJJ = 6); the top buckets; R = 8190 (k_gemm_tn_mma + k_colsum_atomic), R = 8192
# (k_gemm_tn_tc at the threshold), R = 8213 (k_gemm_tn_tc with a ragged last 64-row block and a ragged last 128-row tile
# of the gate GEMM); TSP-20 x 9477 (several register drains per CTA of k_gemm_tn_tc)
CASES = [("tsp", 2, 3), ("tsp", 8, 2), ("vrp", 33, 5), ("irp", 47, 7), ("tsp", 64, 3), ("vrp", 65, 11), ("irp", 88, 5),
         ("tsp", 96, 3), ("vrp", 113, 5), ("tsp", 128, 7), ("vrp", 65, 126), ("tsp", 128, 64), ("irp", 43, 191),
         ("tsp", 20, 9477)]
C4 = ("tsp", 50, 65536)
C4_STAGE_MASK = 0b001   # one layer of stages at C4 (22 GB)
PATH_CASES = [c + (p, "heavy") for c in CASES for p in (0, 1)] + [("tsp", 20, 9477, p, "decoder") for p in (0, 1)] \
    + [C4 + (0, "heavy")]
PATH_IDS = [f"{k}{n}_b{b}_path{p}" + ("_decoder_dh" if u == "decoder" else "") for k, n, b, p, u in PATH_CASES[:-1]] \
    + ["c4_tsp50_b65536_path0"]


def _is_c4(N, B):
    return (N, B) == C4[1:]


def _report(tag, items, t0):
    print(f"\n[{tag}] " + " ".join(f"{k} {v:.2g}" for k, v in items)
          + f"  ({time.time() - t0:.1f} s, peak {torch.cuda.max_memory_allocated() / 2 ** 30:.1f} GiB)")


@pytest.mark.parametrize("kind,N,B,gemm_path,upstream", PATH_CASES, ids=PATH_IDS)
def test_encoder_backward_stages_vs_float64(kind, N, B, gemm_path, upstream):
    """Through the stage hook: every stage gradient of every selected layer in float64 from the kernel's own input to
    that stage, every parameter gradient of those layers from the kernel's own stage gradients, and the embedding
    gradients from the kernel's final dL/d(embedding output)."""
    t0 = time.time()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    mask = C4_STAGE_MASK if _is_c4(N, B) else 0b111
    run = _backward(kind, N, B, gemm_path, upstream, mask=mask)
    gain = run["gain"]
    K = backward_stages(run["stages"], B, N, _layers_of(mask))
    acc = _StageAcc()
    perr = {}
    for l in sorted(K, reverse=True):
        S, hin, P = _layer_inputs(run, l)

        def take(name, sl, ref, l=l):
            got = K[l][name][sl].to(F64)
            acc.put((l, name), got, ref)
            return got

        dx, ref = layer_backward64(S, hin, P, K[l]["dout"].to(F64), N, take)
        got = {k: run["grads"][_grad_key(l, k)] * gain for k in ref}
        perr.update({(l, k): e for k, e in _param_errors(got, ref).items()})
        del dx
    f = run["enc"].node_embed.weight.shape[1]
    x, isdep = _features(run["env"], f)
    ref = embed_backward64(run["demb"].to(F64) * gain, x, isdep, f)
    perr.update({(None, k): e for k, e in _param_errors({k: run["grads"][k] * gain for k in ref}, ref).items()})
    serr = acc.rel()
    worst = {}
    for (l, s), e in serr.items():
        worst[s] = max(worst.get(s, 0.0), e)
    pw = max(perr.items(), key=lambda kv: kv[1])
    _report(f"{kind}{N} B={B} path={gemm_path} {upstream} gain 2^{int(torch.tensor(gain).log2())}",
            list(worst.items()) + [(f"params {pw[0]}", pw[1])], t0)
    bad = [(l, s, e) for (l, s), e in serr.items() if e > STAGE_TOL[s]]
    bad += [(l, k, e) for (l, k), e in perr.items() if e > PARAM_TOL]
    assert not bad, bad


@pytest.mark.parametrize("kind,N,B,gemm_path,upstream", PATH_CASES, ids=PATH_IDS)
def test_encoder_backward_end_to_end_vs_float64(kind, N, B, gemm_path, upstream):
    """The production route (bw.encoder_backward, no hook) against layer_backward64 chained in float64 from the gained
    dL/dh through the three layers and the embedding: every element of every encoder .grad and of the returned
    dL/d(embedding output)."""
    t0 = time.time()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    run = _backward(kind, N, B, gemm_path, upstream)
    gain = run["gain"]
    g = run["dH"].to(F64) * gain
    ref = {}
    chained = lambda name, sl, r: r
    for l in (2, 1, 0):
        S, hin, P = _layer_inputs(run, l)
        g, r = layer_backward64(S, hin, P, g, N, chained)
        ref.update({_grad_key(l, k): v for k, v in r.items()})
    f = run["enc"].node_embed.weight.shape[1]
    x, isdep = _features(run["env"], f)
    ref.update(embed_backward64(g, x, isdep, f))
    assert set(ref) == set(run["grads"]), set(ref) ^ set(run["grads"])
    perr = _param_errors({k: v * gain for k, v in run["grads"].items()}, ref)
    # the return value is dL/d(embedding output) in the scale of dL/dh
    e_demb = (run["demb"].to(F64) - g / gain).abs().max().item() / (g / gain).abs().max().item()
    pw = max(perr.items(), key=lambda kv: kv[1])
    _report(f"{kind}{N} B={B} path={gemm_path} {upstream} end to end",
            [(f"params {pw[0]}", pw[1]), ("dL/demb", e_demb)], t0)
    tol = E2E_PARAM_TOL if B * N >= 1024 else E2E_PARAM_TOL_FEW_ROWS
    bad = [(k, e) for k, e in perr.items() if e > tol]
    assert not bad, bad
    assert e_demb <= E2E_DEMB_TOL, e_demb


@pytest.mark.parametrize("gemm_path", [0, 1])
@pytest.mark.parametrize("kind,N,B", [("irp", 43, 191), ("vrp", 33, 5)], ids=["irp43_b191", "vrp33_b5"])
def test_stage_hook_matches_plain_call(kind, N, B, gemm_path):
    """A hook call (layers 0 and 2) and a plain call on the same inputs give the same parameter gradients and final
    dL/d(embedding output) within HOOK_TOL of each tensor's largest element (not bit-identical: k_gemm_tn_tc and the
    BatchNorm reductions flush with atomics).  The hook writes every element of the selected layers' blocks (NaN
    pre-fill), in the order the mask says: the first block is layer 0 (its dX is the final g), the second layer 2 (its
    dOUT is the gained dL/dh).  Masks outside 1..7 are refused."""
    import vrpx
    from vrpx import backward as bw

    run = _backward(kind, N, B, gemm_path, mask=0b101, plain_too=True)
    gain = run["gain"]
    assert not bool(run["stages"].isnan().any()), "stage element not written"
    K = backward_stages(run["stages"], B, N, [0, 2])
    assert torch.equal(K[2]["dout"], run["dH"] * gain)
    assert torch.equal(K[0]["dx"], run["demb"] * gain)
    gscale = max(p.abs().max().item() for p in run["grads_plain"].values())
    worst = 0.0
    for name, g in run["grads"].items():
        e = (g.to(F64) - run["grads_plain"][name].to(F64)).abs().max().item() / gscale
        worst = max(worst, e)
        assert e <= HOOK_TOL, (name, e)
    e = (run["demb"].to(F64) - run["demb_plain"].to(F64)).abs().max().item() / run["demb_plain"].abs().max().item()
    print(f"\n[{kind}{N} B={B} path={gemm_path}] hook vs plain: parameters {worst:.2g}, dL/demb {e:.2g}")
    assert e <= HOOK_TOL, e
    for bad_mask in (0, 8):
        with pytest.raises(vrpx.VrpxError):
            bw.encoder_backward(run["enc"], run["env"], run["env"]._depot, run["saved"], run["dH"].clone(),
                                gemm_path=gemm_path, stages=run["stages"], stage_layers=bad_mask)


def _attention_case(N, B, spread, seed):
    """qkv (B*N, 384) f32 with the q and k thirds scaled by `spread`, heavy-tailed datt, the float64 att and the float64
    autograd dqkv."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    qkv = torch.randn(B * N, 3 * E, generator=g, device="cuda")
    qkv[:, :2 * E] *= spread
    datt = torch.randn(B * N, E, generator=g, device="cuda", dtype=F64)
    datt *= 10.0 ** (-4.0 * torch.rand(B * N, 1, generator=g, device="cuda", dtype=F64))
    datt = (datt * 2.0 ** -6).float()
    x = qkv.to(F64).requires_grad_(True)
    with torch.enable_grad():
        att64 = _attention64(x.view(B, N, 3 * E))
        (ref,) = torch.autograd.grad(att64, x, datt.to(F64).view(B, N, E))
    return qkv, att64.detach().reshape(B * N, E), datt, ref


@pytest.mark.parametrize("path", [0, 1], ids=["mma", "simt"])
@pytest.mark.parametrize("spread", [1.0, 4.0], ids=["randn", "sharp"])
def test_attention_backward_every_node_count(spread, path):
    """vrpx_debug_attention_backward at every N = 1 ... 128 (all sixteen NK8 = ceil(N / 8) instantiations of
    k_enc_attention_bwd_mma, path 0; the fp32 SIMT kernel, path 1) with an odd instance count, against float64 autograd:
    dQ, dK and dV each relative to its own largest element.  Scores from randn qkv, and sharp ones (q, k x 4: scores of
    standard deviation 16) where most softmax rows are nearly one-hot.  att is the float64 forward rounded to f32; datt is
    heavy-tailed in the gained scale of the encoder backward.  dqkv starts as NaN: every element must be written."""
    import vrpx

    L = vrpx.lib()
    dev = vrpx.require_device()
    worst = {"dq": (0.0, 0), "dk": (0.0, 0), "dv": (0.0, 0)}
    onehot = []
    bad = []
    for N in range(1, 129):
        B = 3 + 2 * (N % 3)
        qkv, att64, datt, ref = _attention_case(N, B, spread, 1000 * N + int(spread))
        if spread > 1.0 and N >= 8:
            q, k = (qkv.to(F64).view(B, N, 3, 8, 16)[:, :, i].transpose(1, 2) for i in range(2))
            onehot.append((torch.softmax(q @ k.transpose(-1, -2) / 4.0, -1).amax(-1) > 0.9).double().mean().item())
        att = att64.float().contiguous()
        dqkv = torch.full((B * N, 3 * E), float("nan"), device=dev)
        vrpx.check(L.vrpx_debug_attention_backward(vrpx.ptr(qkv), vrpx.ptr(att), vrpx.ptr(datt), vrpx.ptr(dqkv), B, N,
                                                   path, vrpx.stream_ptr(dev)))
        torch.cuda.synchronize()
        assert not bool(dqkv.isnan().any()), (N, "element not written")
        for i, name in enumerate(("dq", "dk", "dv")):
            r = ref[:, i * E:(i + 1) * E]   # at N = 1, dQ = dK = 0 exactly: relative to dV there
            e = (dqkv[:, i * E:(i + 1) * E].to(F64) - r).abs().max().item() / (r.abs().max().item() or ref.abs().max().item())
            worst[name] = max(worst[name], (e, N))
            if e > ATTN_TOL:
                bad.append((N, name, e))
    if onehot:
        print(f"\n[attention backward spread {spread} path {path}] rows with max p > 0.9: "
              f"{min(onehot):.2f} ... {max(onehot):.2f}")
        assert min(onehot) > 0.5
    print(f"\n[attention backward spread {spread} path {path}] "
          + " ".join(f"{k} {e:.2g}@N={n}" for k, (e, n) in worst.items()))
    assert not bad, bad
