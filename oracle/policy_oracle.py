"""Plain-op fp32 restatement of the reference attention policy (encoder, decoder
step, rollout loop, REINFORCE loss).

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).  Works from a reference-format
`state_dict` (SURVEY App. A.5) with explicit matmuls — no nn.MultiheadAttention,
no nn.BatchNorm1d — so that it documents the arithmetic the CUDA kernels follow.

Parity: PINNED against embeddings / logits / greedy tapes recorded from the
unmodified reference (tests/golden/policy_*.npz) and reference tests' means.
"""
from __future__ import annotations

import math

import numpy as np
import torch

from .env_oracle import IRP, TSP, VRP, EnvOracle

H = 8  # heads everywhere (graph_tsp_agent.py:55, graph_encoder.py:13)


def _bn(x2d, sd, prefix, train, eps=1e-5):
    """BatchNorm1d over flattened (B*N, E) rows — graph_encoder.py:141-154."""
    w, b = sd[prefix + ".norm.weight"], sd[prefix + ".norm.bias"]
    if train:
        mean = x2d.mean(0)
        var = x2d.var(0, unbiased=False)
    else:
        mean, var = sd[prefix + ".norm.running_mean"], sd[prefix + ".norm.running_var"]
    return (x2d - mean) / torch.sqrt(var + eps) * w + b


def encoder_forward(sd, x, depot_onehot=None, train=False, num_layers=3, chunk=None, relu=None):
    """graph_encoder.py:41-58 (GraphEncoder) / :95-138 (GraphDemandEncoder) /
    :183-198 (MultiHeadAttentionLayer).  x (B,N,f) f32; depot_onehot (B,N) bool or None.

    chunk (optional): run attention and feed-forward on `chunk` instances at a time, so that a large batch (or its
    float64 / forward-mode evaluation) fits in memory.  BatchNorm statistics still span all B*N rows; the arithmetic
    is the same as with chunk=None.

    relu (optional): relu(pre, layer, first) replaces torch.relu in the feed-forward of `layer`, pre (b,N,512) being
    the pre-activations of instances first .. first + b - 1.  Lets a float64 evaluation follow the ReLU gate of an
    fp32 computation where a pre-activation lies within rounding of zero."""
    B, N, f = x.shape
    E = sd["encoder.node_embed.weight"].shape[0]
    h = x @ sd["encoder.node_embed.weight"].T + sd["encoder.node_embed.bias"]
    if depot_onehot is not None:
        # depot rows use depot_embed on the first 2 features (:110-132)
        hd = x[:, :, :2] @ sd["encoder.depot_embed.weight"].T + sd["encoder.depot_embed.bias"]
        h = torch.where(depot_onehot[:, :, None], hd, h)
    dh = E // H

    def per_chunk(fn, h):
        if chunk is None or chunk >= B:
            return fn(h, 0)
        return torch.cat([fn(h[i:i + chunk], i) for i in range(0, B, chunk)])

    for l in range(num_layers):
        p = f"encoder.attention_layers.{l}."
        Wi, bi = sd[p + "attention_layer.in_proj_weight"], sd[p + "attention_layer.in_proj_bias"]
        Wo, bo = sd[p + "attention_layer.out_proj.weight"], sd[p + "attention_layer.out_proj.bias"]

        def attention(h, first):
            b = h.shape[0]
            qkv = h @ Wi.T + bi  # rows ordered [q;k;v]
            q, k, v = qkv.split(E, dim=-1)
            q = q.view(b, N, H, dh).transpose(1, 2)
            k = k.view(b, N, H, dh).transpose(1, 2)
            v = v.view(b, N, H, dh).transpose(1, 2)
            s = (q @ k.transpose(-1, -2)) / math.sqrt(dh)
            a = torch.softmax(s, dim=-1) @ v  # (b,H,N,dh)
            a = a.transpose(1, 2).reshape(b, N, E)
            o = a @ Wo.T + bo
            return h + o

        def feed_forward(h, first):
            ff = h @ sd[p + "ff.0.weight"].T + sd[p + "ff.0.bias"]
            ff = torch.relu(ff) if relu is None else relu(ff, l, first)
            ff = ff @ sd[p + "ff.2.weight"].T + sd[p + "ff.2.bias"]
            return h + ff

        h = _bn(per_chunk(attention, h).reshape(B * N, E), sd, p + "bn1", train).view(B, N, E)
        h = _bn(per_chunk(feed_forward, h).reshape(B * N, E), sd, p + "bn2", train).view(B, N, E)
    return h


def decoder_logits(sd, h, mask, first, last, load=None, C=10.0, glimpse_mask=None):
    """One decode step up to the masked pointer logits — graph_decoder.py:75-98.

    h (B,N,E); mask (B,N) f32 0/1; first/last (B,E).  Returns u (B,N) with -inf on
    masked nodes.  Includes the additive, head-scrambled glimpse mask (:93-94):
    attention row (b,h) adds mask[(b*H+h) mod B].

    glimpse_mask (B,H,N), optional: the rows `mask.repeat(H,1)` would deliver, given
    explicitly — lets a test evaluate a SUBSET of a large batch (the rows of the
    partner instances (b*H+h) mod B_full are looked up by the caller).
    """
    B, N, E = h.shape
    D = 3 * E
    g = h.mean(dim=1)  # :75-77
    kk = h @ sd["decoder._kp.weight"].T  # :83
    if load is None:
        ctx = torch.cat([g, first, last], -1)  # :88
    else:
        ctx = torch.cat([g, last, load[:, None]], -1) @ sd["decoder._context_proj.weight"].T  # :90-91
    bq, bk, bv = sd["decoder.attention.in_proj_bias"].split(D)
    q = ctx @ sd["decoder.attention.q_proj_weight"].T + bq
    K = h @ sd["decoder.attention.k_proj_weight"].T + bk
    V = h @ sd["decoder.attention.v_proj_weight"].T + bv
    dh = D // H
    q = q.view(B, H, dh)
    K = K.view(B, N, H, dh).permute(0, 2, 1, 3)
    V = V.view(B, N, H, dh).permute(0, 2, 1, 3)
    s = torch.einsum("bhd,bhnd->bhn", q, K) / math.sqrt(dh)
    if glimpse_mask is None:
        rows = (torch.arange(B)[:, None] * H + torch.arange(H)[None, :]) % B  # mask.repeat(H,1) quirk
        glimpse_mask = mask[rows]
    s = s + glimpse_mask  # float mask is ADDED (:93-94)
    p = torch.softmax(s, dim=-1)
    a = torch.einsum("bhn,bhnd->bhd", p, V).reshape(B, D)
    o = a @ sd["decoder.attention.out_proj.weight"].T + sd["decoder.attention.out_proj.bias"]
    qq = o @ sd["decoder._att_output.weight"].T  # :95
    u = torch.tanh(torch.einsum("be,bne->bn", qq, kk) / math.sqrt(E)) * C  # :97
    return u.masked_fill(mask.bool(), float("-inf"))  # :98


def rollout(sd, env: EnvOracle, greedy=True, train=False, tape=None, return_trace=False, dtype=torch.float32):
    """The rollout loop — graph_tsp_agent.py:61-92 / graph_vrp_agent.py:52-83 /
    graph_irp_agent.py:54-105.

    `tape` (T,B) int: teacher-forced actions (replayed instead of argmax / sampling).
    `dtype`: float32 = the reference's arithmetic.  float64 (with a float64 `sd`) evaluates the SAME f32 weights on the
    SAME f32-rounded observations (graph_tsp_agent.py:72 casts the state to f32) without rounding in between — the
    yardstick that measures how far the reference's own fp32 result is from its exact value.
    Returns (acc_loss (B,), acc_log_prob (B,)[, trace dict]).
    """
    kind = env.kind
    st = env.get_state()
    load = None
    if kind == IRP:
        st, load_np = st
        load = torch.tensor(load_np, dtype=torch.float).to(dtype)
    st = torch.tensor(st, dtype=torch.float).to(dtype)
    B, N = st.shape[:2]
    if kind == TSP:
        h = encoder_forward(sd, st[:, :, :2], None, train)
    elif kind == VRP:
        # depot mask taken from state col 3 (= initial mask) — graph_vrp_agent.py:67
        h = encoder_forward(sd, st[:, :, :2], st[:, :, 3].bool(), train)
    else:
        h = encoder_forward(sd, st[:, :, :3], st[:, :, 3].bool(), train)  # graph_irp_agent.py:77-79
    E = h.shape[-1]
    first = sd["decoder._first_node"].reshape(1, E).repeat(B, 1)
    last = sd["decoder._last_node"].reshape(1, E).repeat(B, 1)
    acc_loss = torch.zeros(B)
    acc_logp = torch.zeros(B, dtype=dtype)
    trace = {"actions": [], "logits": [], "logp": [], "reward": []}
    done, t = False, 0
    while not done:
        mask = st[:, :, -1]
        u = decoder_logits(sd, h, mask, first, last, load if kind == IRP else None)
        if tape is not None:
            a = torch.as_tensor(tape[t], dtype=torch.long)
        elif greedy:
            a = u.argmax(-1)  # graph_decoder.py:103
        else:
            a = torch.distributions.Categorical(logits=u).sample()  # :105-106
        if greedy and tape is None:
            logp = torch.zeros(B, dtype=dtype)  # :100
        else:
            logp = u.gather(1, a[:, None])[:, 0] - torch.logsumexp(u, dim=-1)  # :107
        if not greedy:
            acc_logp = acc_logp + logp
        last = h[torch.arange(B), a]  # :108-109
        if t == 0:
            first = last  # :111-113
        s2, r, done, _ = env.step(a.numpy()[:, None])
        acc_loss = acc_loss + torch.tensor(r, dtype=torch.float)  # f32 accumulate (:85)
        if kind == IRP:
            s2, load_np = s2
            load = torch.tensor(load_np, dtype=torch.float).to(dtype)
        st = torch.tensor(s2, dtype=torch.float).to(dtype)
        if return_trace:
            trace["actions"].append(a.numpy().copy())
            trace["logits"].append(u.detach().numpy().copy())
            trace["logp"].append(logp.detach().numpy().copy())
            trace["reward"].append(np.asarray(r).copy())
        t += 1
    if return_trace:
        trace = {k: np.stack(v) for k, v in trace.items()}
        trace["emb"] = h.detach().numpy()
        return acc_loss, acc_logp, trace
    return acc_loss, acc_logp


def replay_subset_logits(sd, h, tape, own_masks, glimpse_masks, loads=None):
    """Teacher-forced per-step pointer logits of a SUBSET of a (possibly huge) batch — graph_decoder.py:75-115 looped as
    in graph_tsp_agent.py:78-88.

    h (S,N,E) embeddings of the subset; tape (T,S) the subset's actions; own_masks (T,S,N) each instance's mask before
    step t; glimpse_masks (T,S,H,N) the masks of its partner rows (b*H+h) mod B_full before step t; loads (T,S) f32
    (IRP) or None.  Returns logits (T,S,N) and per-step log-probs (T,S)."""
    S, N, E = h.shape
    first = sd["decoder._first_node"].reshape(1, E).repeat(S, 1)
    last = sd["decoder._last_node"].reshape(1, E).repeat(S, 1)
    out, lps = [], []
    ar = torch.arange(S)
    for t in range(tape.shape[0]):
        u = decoder_logits(sd, h, torch.as_tensor(own_masks[t], dtype=torch.float), first, last,
                           None if loads is None else torch.as_tensor(loads[t], dtype=torch.float),
                           glimpse_mask=torch.as_tensor(glimpse_masks[t], dtype=torch.float))
        a = torch.as_tensor(tape[t], dtype=torch.long)
        lps.append((u.gather(1, a[:, None])[:, 0] - torch.logsumexp(u, dim=-1)).numpy())
        last = h[ar, a]
        if t == 0:
            first = last
        out.append(u.numpy())
    return np.stack(out), np.stack(lps)


def reinforce_loss(cost_model, cost_baseline, logp):
    """graph_tsp_agent.py:179-180 with loss_* = -cost: advantage = cost_m - cost_b."""
    adv = cost_model - cost_baseline
    return (adv * logp).mean()


def reinforce_gradients(kind, sd, xy, depot, demand, tape, baseline):
    """torch autograd through the oracle's train-mode teacher-forced rollout: loss = mean((cost_m - cost_b) * log_prob)
    (graph_tsp_agent.py:179-186).  Returns {parameter name: gradient} for every parameter with a gradient."""
    sd = {k: v.detach().clone() for k, v in sd.items()}
    for k, v in sd.items():
        if v.dtype == torch.float32 and "running_" not in k:
            v.requires_grad_(True)
    loss_m, logp = rollout(sd, EnvOracle(kind, xy, depot, demand), greedy=False, train=True, tape=tape)
    adv = (loss_m.detach() - torch.as_tensor(baseline)) * -1
    loss = (adv * logp).mean()
    loss.backward()
    return {k: v.grad for k, v in sd.items() if v.requires_grad and v.grad is not None}, float(loss.item())
