"""REINFORCE backward on libvrpx: loss = mean_b(advantage_b * sum_t log p(a_{b,t}))
(reference agents/graph_tsp_agent.py:179-186 `loss.backward()` through the whole rollout).

No autograd graph is recorded during the fused rollout.  Instead the forward keeps (a) the action tape and the
per-step masks/loads, (b) the encoder activations; the backward then runs
  1. vrpx_decoder_backward  — recompute-based backward of every decode step (csrc/decoder_bwd.cu) -> dL/dh and the
     gradients of the packed decoder arrays,
  2. the per-episode decoder terms (graph mean, first node, biases) with small GEMM / reduction kernels,
  3. one torch.autograd pull-back of the packed-array gradients through vrpx.packing.fold_decoder (a handful of
     128..1024-sized matrix products, float64) to the decoder's own parameters,
  4. vrpx_encoder_backward — BatchNorm(batch stats) / FF / attention / embedding backward (csrc/encoder_bwd.cu),
and accumulates into `param.grad` exactly where torch would have put it.
"""
from __future__ import annotations

import ctypes as C
import math

import torch

import vrpx
from vrpx import packing


def _acc_grad(p, g):
    g = g.to(p.dtype)
    if p.grad is None:
        p.grad = g.clone()
    else:
        p.grad.add_(g)


def _gemm_nt(X, W, residual=None, path=0):
    """Y = X · W^T (+ residual) through the library GEMM (W in [NOUT][K] layout)."""
    R, K = X.shape
    NOUT = W.shape[0]
    Y = torch.empty((R, NOUT), dtype=torch.float32, device=X.device)
    vrpx.check(vrpx.lib().vrpx_debug_gemm(vrpx.ptr(X), R, K, vrpx.ptr(W), NOUT, None, 0,
                                          vrpx.ptr(residual) if residual is not None else None, None, None,
                                          vrpx.ptr(Y), path, vrpx.stream_ptr(X.device)))
    return Y


# The f16 hi/lo split of the tensor-core GEMMs (f16split.cuh) scales its operands by 2^8: values below ~1e-4 leave their lo
# halves in the f16 subnormals and values above 255 overflow.  Per-row gradients of a mean loss shrink with the batch
# (1e-5 ... 1e-7 at 65,536 instances: 0.3 % ... 24 % error in the encoder gradients, tools/grad_scale_probe.py), so the
# encoder backward runs on dH * 2^k with max|dH| * 2^k = 2^-6 — every op of the backward is linear in dH, a power of two
# is exact, and the 2^14 of headroom covers what BatchNorm and the projections can amplify — and the parameter
# gradients are scaled back before they are accumulated.
_GRAD_TARGET_LOG2 = -6
_GRAD_TARGET_ENV = None   # tools/grad_scale_probe.py overrides the target for its sweep


def _grad_gain(dH, target_log2=None):
    amax = float(dH.abs().amax())
    if not (amax > 0.0) or amax == float("inf") or amax != amax:
        return 1.0
    if target_log2 is None:
        target_log2 = _GRAD_TARGET_LOG2 if _GRAD_TARGET_ENV is None else _GRAD_TARGET_ENV
    k = target_log2 - math.frexp(amax)[1]          # amax = m * 2^e with 0.5 <= m < 1: amax * 2^k in [2^-7, 2^-6)
    return 2.0 ** max(-60, min(60, k))


def decoder_backward(dec, env, h, roll, wts, gemm_path=0):
    """Back-propagate wts[b] = dL/d(logp_b) through the rollout `roll` (dict from GraphDecoder.rollout_episode with
    save_for_backward=True).  Accumulates the decoder parameters' .grad and returns dL/dh (B,N,128)."""
    L = vrpx.lib()
    dev = h.device
    st = vrpx.stream_ptr(dev)
    B, N = env.batch_size, env.num_nodes
    irp = env._KIND == vrpx.IRP
    w = dec.packed(irp, dev)
    tens = dec._packed[irp].tensors
    sv = roll["saved"]
    tape = roll["tape"].contiguous()
    T = int(tape.shape[0])
    z = lambda *s: torch.zeros(s, dtype=torch.float32, device=dev)
    g = {"dH": z(B, N, 128), "D0": z(B, 1024), "D1": z(B, 1024), "Dl": z(B, 1024) if irp else None,
         "d_al_t": z(128, 1024), "d_m_t": z(1024, 128), "d_m_c": z(128)}
    gs = vrpx.DecoderGrads(*[None if g[k] is None else g[k].data_ptr() for k in ("dH", "D0", "D1", "Dl", "d_al_t", "d_m_t", "d_m_c")])
    m_n = tens["m_t"].t().contiguous()
    al_n = tens["al_t"].t().contiguous()
    wb = vrpx.DecoderBwdWeights(m_n.data_ptr(), al_n.data_ptr())
    trace = vrpx.RolloutTrace(sv["mask_hist"].data_ptr(), sv["load_hist"].data_ptr(), sv["qg0"].data_ptr())
    nbytes = int(L.vrpx_decoder_backward_workspace_bytes(B, N))
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
    wts = wts.detach().to(dev, torch.float32).contiguous()
    vrpx.check(L.vrpx_decoder_backward(C.byref(env._view()), C.byref(w), C.byref(wb), vrpx.ptr(h), vrpx.ptr(tape), T,
                                       int(roll["coupling"]), C.byref(trace), vrpx.ptr(sv["qg"]), vrpx.ptr(wts),
                                       C.byref(gs), vrpx.ptr(ws), nbytes, st))
    # ---- per-episode terms: q~ also contains A_g·g + a_c (every step), A_f·h[first] (steps >= 1), a_q0 (step 0)
    # the per-episode sums D are gradients too: the products below run on the f16-split tensor-core kernels (the weight
    # gradients ag_t / af_t at B >= 8192 on either gemm_path), so they get them scaled to 2^-2 (see _grad_gain; the sums
    # are final, nothing amplifies them further) and are scaled back
    Dsum = g["D0"] + g["D1"]
    gs_, g1_ = _grad_gain(Dsum, -2), _grad_gain(g["D1"], -2)
    DsumS = Dsum * gs_ if gs_ != 1.0 else Dsum
    D1S = g["D1"] * g1_ if g1_ != 1.0 else g["D1"]
    G = torch.empty((B, 128), dtype=torch.float32, device=dev)
    Xf = None if irp else torch.empty((B, 128), dtype=torch.float32, device=dev)
    tape0 = tape[0].contiguous()
    vrpx.check(L.vrpx_episode_gather(vrpx.ptr(h), vrpx.ptr(tape0), B, N, vrpx.ptr(G), vrpx.ptr(Xf) if Xf is not None else None, st))
    dG = _gemm_nt(DsumS, tens["ag_t"], path=gemm_path)                      # (B,128) = Dsum · A_g
    dXf = None if irp else _gemm_nt(D1S, tens["af_t"], path=gemm_path)       # (B,128) = D1 · A_f
    if gs_ != 1.0:
        dG.mul_(1.0 / gs_)
    if dXf is not None and g1_ != 1.0:
        dXf.mul_(1.0 / g1_)
    vrpx.check(L.vrpx_episode_scatter(vrpx.ptr(g["dH"]), vrpx.ptr(tape0), B, N, vrpx.ptr(dG),
                                      vrpx.ptr(dXf) if dXf is not None else None, st))
    grads = {"al_t": g["d_al_t"], "m_t": g["d_m_t"], "m_c": g["d_m_c"], "ag_t": z(128, 1024), "a_c": z(1024), "a_q0": z(1024)}
    vrpx.check(L.vrpx_gemm_tn_accumulate(vrpx.ptr(G), vrpx.ptr(DsumS), vrpx.ptr(grads["ag_t"]), B, 128, 1024, st))
    if gs_ != 1.0:
        grads["ag_t"].mul_(1.0 / gs_)
    vrpx.check(L.vrpx_colsum_accumulate(vrpx.ptr(Dsum), B, 1024, vrpx.ptr(grads["a_c"]), st))
    vrpx.check(L.vrpx_colsum_accumulate(vrpx.ptr(g["D0"]), B, 1024, vrpx.ptr(grads["a_q0"]), st))
    if irp:
        grads["a_load"] = z(1024)
        vrpx.check(L.vrpx_colsum_accumulate(vrpx.ptr(g["Dl"]), B, 1024, vrpx.ptr(grads["a_load"]), st))
    else:
        grads["af_t"] = z(128, 1024)
        vrpx.check(L.vrpx_gemm_tn_accumulate(vrpx.ptr(Xf), vrpx.ptr(D1S), vrpx.ptr(grads["af_t"]), B, 128, 1024, st))
        if g1_ != 1.0:
            grads["af_t"].mul_(1.0 / g1_)
    # ---- pull the packed-array gradients back to the module parameters (tiny weight-only products)
    params = [p for p in dec.parameters() if p.requires_grad]
    with torch.enable_grad():
        folded = packing.fold_decoder(dec, irp)
        outs, gouts = [], []
        for k, gv in grads.items():
            if folded.get(k) is not None:
                outs.append(folded[k])
                gouts.append(gv.double())
        pg = torch.autograd.grad(outs, params, gouts, allow_unused=True)
    for p, gp in zip(params, pg):
        if gp is not None:
            _acc_grad(p, gp)
    return g["dH"]


def encoder_backward(enc, env, depot, saved, dH, gemm_path=0):
    """Back-propagate dL/dh (overwritten) through the train-mode encoder; accumulates the parameters' .grad."""
    L = vrpx.lib()
    dev = dH.device
    B, N = env.batch_size, env.num_nodes
    w = packing.encoder_struct(enc, dev)
    keep = []
    wt = vrpx.EncoderWeightsT()
    gr = vrpx.EncoderGrads()
    # gemm_path = 1 runs the data-gradient GEMMs and the attention backward in fp32, but the weight gradients go through
    # the f16-split k_gemm_tn_tc on both paths once B*N >= 8192 rows, so both need the gain
    gain = _grad_gain(dH)
    if gain != 1.0:
        dH.mul_(gain)
    # the kernels accumulate into a zeroed flat buffer (one view per parameter); it is scaled back and added to .grad below
    dep = getattr(enc, "depot_embed", None)
    plist = [enc.node_embed.weight, enc.node_embed.bias] + ([dep.weight, dep.bias] if dep is not None else [])
    for layer in enc.attention_layers:
        a = layer.attention_layer
        plist += [a.in_proj_weight, a.in_proj_bias, a.out_proj.weight, a.out_proj.bias, layer.bn1.norm.weight,
                  layer.bn1.norm.bias, layer.ff[0].weight, layer.ff[0].bias, layer.ff[2].weight, layer.ff[2].bias,
                  layer.bn2.norm.weight, layer.bn2.norm.bias]
    offs, total = [], 0
    for p in plist:
        offs.append(total)
        total += (p.numel() + 3) // 4 * 4                 # 16-byte aligned views
    flat = torch.zeros((total,), dtype=torch.float32, device=dev)
    view = {id(p): flat[o:o + p.numel()] for p, o in zip(plist, offs)}
    vp_ = lambda p: view[id(p)].data_ptr()

    gr.node_w, gr.node_b = vp_(enc.node_embed.weight), vp_(enc.node_embed.bias)
    gr.depot_w = vp_(dep.weight) if dep is not None else None
    gr.depot_b = vp_(dep.bias) if dep is not None else None
    for i, layer in enumerate(enc.attention_layers):
        a = layer.attention_layer
        tr = [a.in_proj_weight.detach().t().contiguous(), a.out_proj.weight.detach().t().contiguous(),
              layer.ff[0].weight.detach().t().contiguous(), layer.ff[2].weight.detach().t().contiguous()]
        keep.extend(tr)
        T_ = wt.layer[i]
        T_.in_proj_wT, T_.out_proj_wT, T_.ff0_wT, T_.ff2_wT = [t.data_ptr() for t in tr]
        G_ = gr.layer[i]
        G_.in_proj_w, G_.in_proj_b = vp_(a.in_proj_weight), vp_(a.in_proj_bias)
        G_.out_proj_w, G_.out_proj_b = vp_(a.out_proj.weight), vp_(a.out_proj.bias)
        G_.bn1_w, G_.bn1_b = vp_(layer.bn1.norm.weight), vp_(layer.bn1.norm.bias)
        G_.ff0_w, G_.ff0_b = vp_(layer.ff[0].weight), vp_(layer.ff[0].bias)
        G_.ff2_w, G_.ff2_b = vp_(layer.ff[2].weight), vp_(layer.ff[2].bias)
        G_.bn2_w, G_.bn2_b = vp_(layer.bn2.norm.weight), vp_(layer.bn2.norm.bias)
    nbytes = int(L.vrpx_encoder_backward_workspace_bytes(B, N))
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
    vrpx.check(L.vrpx_encoder_backward(C.byref(w), C.byref(wt), C.byref(env._view()), None,
                                       vrpx.ptr(depot) if depot is not None else None, B, N, vrpx.ptr(saved),
                                       vrpx.ptr(dH), C.byref(gr), vrpx.ptr(ws), nbytes, gemm_path, vrpx.stream_ptr(dev)))
    if gain != 1.0:
        flat.mul_(1.0 / gain)
    if not bool(torch.isfinite(flat.sum())):
        raise vrpx.VrpxError("encoder backward: non-finite gradient (an operand of the f16-split GEMMs left the f16 range; "
                             "gain %g)" % gain)
    for p in plist:
        _acc_grad(p, view[id(p)].view_as(p))
    return dH
