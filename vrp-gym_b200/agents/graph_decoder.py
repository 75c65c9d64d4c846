"""GraphDecoder — parameters of the attention decoder + a single-step entry point on libvrpx.

Parameter names/shapes/construction order follow the reference (agents/graph_decoder.py:13-48) so that
state dicts interchange:  _first_node, _last_node, attention.{q,k,v}_proj_weight, attention.in_proj_bias,
attention.out_proj.{weight,bias}, _kp.weight, _att_output.weight, _context_proj.weight.

The decode step itself (context -> glimpse attention with the reference's additive, head-scrambled mask ->
tanh-clipped pointer logits -> masked argmax / sampling, graph_decoder.py:51-115) lives in the persistent
CUDA rollout kernel (csrc/rollout.cu).  Models call it for whole episodes (`rollout_episode`); calling this
module directly decodes ONE step through the same kernel (resumable launch), keeping `first_/last_` state
between calls exactly like the reference module does.
"""
from __future__ import annotations

import ctypes as C
import logging
from copy import deepcopy

import numpy as np
import torch
import torch.nn as nn

import vrpx
from vrpx import packing


class GraphDecoder(nn.Module):
    def __init__(self, emb_dim: int = 128, num_heads: int = 8, v_dim: int = 128, k_dim: int = 128):
        super().__init__()
        assert (emb_dim, num_heads, v_dim, k_dim) == (128, 8, 128, 128), \
            "libvrpx kernels are specialised for E=128, H=8 (the reference's only configuration)"
        self._first_node = nn.Parameter(torch.rand(1, 1, emb_dim))
        self._last_node = nn.Parameter(torch.rand(1, 1, emb_dim))
        self.attention = nn.MultiheadAttention(embed_dim=3 * emb_dim, num_heads=num_heads, kdim=k_dim, vdim=v_dim,
                                               batch_first=True)
        self._kp = nn.Linear(emb_dim, emb_dim, bias=False)
        self._att_output = nn.Linear(emb_dim * 3, emb_dim, bias=False)
        self._context_proj = nn.Linear(emb_dim * 2 + 1, emb_dim * 3, bias=False)

        self.first_ = None
        self.last_ = None
        self.first_step = True
        self.num_heads = num_heads
        self._packed = {False: packing.PackedDecoder(), True: packing.PackedDecoder()}
        self._ep = None  # single-step decoding state
        self.score_tables = True  # whole-episode rollouts precompute the glimpse score tables (False: classic kernel path)

    # ------------------------------------------------------------------ whole-episode entry (used by the models)
    def packed(self, irp: bool, device) -> "vrpx.DecoderWeights":
        return self._packed[irp].get(self, irp, device)

    def rollout_episode(self, env, h: torch.Tensor, *, greedy: bool, tape_in=None, want_logits: bool = False,
                        coupling=None, seed: int = 0, offset: int = 0, save_for_backward: bool = False):
        """Run every decode step + environment transition of one episode in one persistent launch.

        env: device-resident TSPEnv/VRPEnv/IRPEnv in its reset state.  h: (B,N,128) f32 CUDA embeddings.
        Returns dict(cost (B,) f32, logp (B,) f32, steps int, tape (steps,B) uint8[, logits (steps,B,N)])."""
        dev = env._device
        B, N = env.batch_size, env.num_nodes
        irp = env._KIND == vrpx.IRP
        w = self.packed(irp, dev)
        Tmax = (N - 1) if env._KIND == vrpx.TSP else 2 * (N - 1) + 1
        if tape_in is not None:
            mode = vrpx.TEACHER
            tape = torch.as_tensor(np.ascontiguousarray(tape_in, dtype=np.uint8)).to(dev)
            Tmax = int(tape.shape[0])
        else:
            mode = vrpx.GREEDY if greedy else vrpx.SAMPLE
            tape = torch.empty((Tmax, B), dtype=torch.uint8, device=dev)
        logp = torch.empty((B,), dtype=torch.float32, device=dev)
        cost = torch.empty((B,), dtype=torch.float32, device=dev)
        steps = torch.zeros((1,), dtype=torch.int32, device=dev)
        logits = torch.empty((Tmax, B, N), dtype=torch.float32, device=dev) if want_logits else None
        L = vrpx.lib()
        nbytes = int(L.vrpx_rollout_workspace_bytes(B, N))
        ws = None
        if self.score_tables and Tmax >= 3:
            # table mode (include/vrpx.h, qk_w): per-episode glimpse score tables in a larger workspace
            tbytes = int(L.vrpx_rollout_table_workspace_bytes(env._KIND, B, N))
            try:
                ws, nbytes = torch.empty((tbytes,), dtype=torch.uint8, device=dev), tbytes
            except torch.cuda.OutOfMemoryError:
                # not silent: the classic per-step score pass is the same arithmetic but ~2x slower
                logging.getLogger(__name__).warning(
                    "vrpx: %.1f GiB score-table workspace does not fit on %s; this rollout runs the classic decode "
                    "loop (set decoder.score_tables = False to choose it explicitly)", tbytes / 2 ** 30, dev)
                ws = None
        if ws is None:
            ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
        G = _coupling_group(coupling, B)
        trace, saved = None, None
        if save_for_backward:
            saved = {"mask_hist": torch.empty((Tmax, B, 4), dtype=torch.int32, device=dev),
                     "load_hist": torch.empty((Tmax, B), dtype=torch.float32, device=dev),
                     "qg0": torch.empty((B, 1024), dtype=torch.float32, device=dev)}
            trace = vrpx.RolloutTrace(saved["mask_hist"].data_ptr(), saved["load_hist"].data_ptr(), saved["qg0"].data_ptr())
        env._sync_instances()
        vrpx.check(L.vrpx_rollout(C.byref(env._view()), C.byref(w), vrpx.ptr(h), mode, G, C.c_uint64(seed),
                                  C.c_uint64(offset), vrpx.ptr(tape), 0, Tmax, vrpx.ptr(logp), vrpx.ptr(cost),
                                  vrpx.ptr(steps), vrpx.ptr(logits) if logits is not None else None,
                                  C.byref(trace) if trace is not None else None,
                                  vrpx.ptr(ws), nbytes, vrpx.stream_ptr(dev)))
        T = int(steps.item())
        env.step_count += T
        env._host_cur = None
        out = {"cost": cost, "logp": logp, "steps": T, "tape": tape[:T], "coupling": G}
        if saved is not None:
            o = int(L.vrpx_rollout_workspace_qg_offset())
            saved["qg"] = ws[o:o + B * 4096].view(torch.float32).view(B, 1024)  # Q~g incl. the `first` fold
            saved["ws"] = ws
            out["saved"] = saved
        if logits is not None:
            out["logits"] = logits[:T]
        return out

    def rollout_samples(self, env, h: torch.Tensor, num_samples: int, *, seed: int, offset: int = 0, coupling=None,
                        want_logits: bool = False, save_for_backward: bool = False):
        """K = num_samples sampled episodes of every instance from one set of embeddings (vrpx_rollout_samples_traced).

        env: device-resident TSPEnv/VRPEnv/IRPEnv of B instances in its reset state; it is left untouched (the K copies
        run on a private copy-major replica, replica k·B + b = copy k of instance b).  h: (B,N,128) f32 CUDA embeddings.
        Copy k is bit-identical to rollout_episode(copy of env, h, greedy=False, seed=seed, offset=offset + k·B,
        coupling=coupling).  All copies run until the slowest is done; a finished VRP/IRP copy idles on its depot.
        Returns dict(cost (K,B) f32, logp (K,B) f32, steps int = max over copies, tape (steps,K,B) uint8, samples K
        [, logits (steps,K,B,N)]).  save_for_backward=True adds `saved`: the per-replica trace (mask_hist (Tmax,K·B,4),
        load_hist (Tmax,K·B), qg0 (K·B,1024)), qg (K·B,1024) and the workspace holding it, and `replicas`, the vrpx_env
        view of the replica env (with `replica_arrays` keeping its arrays alive) — what vrpx/backward.py replays."""
        K, G = check_samples(env, num_samples, coupling, train=save_for_backward)
        dev = env._device
        B, N, kind = env.batch_size, env.num_nodes, env._KIND
        Tmax = _max_steps(kind, N)
        if Tmax < 3:
            # TSP with N <= 3 has no table-mode decode loop: the definition itself, K episodes on copies of the env
            runs = [self.rollout_episode(deepcopy(env), h, greedy=False, want_logits=want_logits, coupling=G, seed=seed,
                                         offset=offset + k * B) for k in range(K)]
            T = max(r["steps"] for r in runs)
            tape = env._depot.to(torch.uint8).repeat(T, K, 1)
            for k, r in enumerate(runs):
                tape[:r["steps"], k] = r["tape"]
            out = {"cost": torch.stack([r["cost"] for r in runs]), "logp": torch.stack([r["logp"] for r in runs]),
                   "steps": T, "tape": tape, "coupling": G}
            if want_logits:
                logits = torch.full((T, K, B, N), float("nan"), dtype=torch.float32, device=dev)
                for k, r in enumerate(runs):
                    logits[:r["steps"], k] = r["logits"]
                out["logits"] = logits
            return out
        if tuple(h.shape) != (B, N, vrpx.EMB) or h.dtype != torch.float32:
            raise ValueError(f"h must be ({B}, {N}, {vrpx.EMB}) float32, got {tuple(h.shape)} {h.dtype}")
        h = h.contiguous()
        R = K * B
        env._sync_instances()
        # the replicated env: instances repeated copy-major, fresh episode state
        xy, depot, demand = env._xy.repeat(K, 1, 1), env._depot.repeat(K), env._demand.repeat(K, 1)
        visited = torch.zeros((R, 4), dtype=torch.int32, device=dev)
        mask = visited if kind != vrpx.IRP else torch.zeros((R, 4), dtype=torch.int32, device=dev)
        cur = torch.empty((R,), dtype=torch.int32, device=dev)
        load = torch.ones((R,), dtype=torch.float64, device=dev)
        v = vrpx.EnvView()
        v.kind, v.N, v.B = kind, N, R
        v.xy, v.depot, v.demand = xy.data_ptr(), depot.data_ptr(), demand.data_ptr()
        v.visited, v.mask, v.cur, v.load = visited.data_ptr(), mask.data_ptr(), cur.data_ptr(), load.data_ptr()
        L = vrpx.lib()
        st = vrpx.stream_ptr(dev)
        vrpx.check(L.vrpx_env_reset(C.byref(v), st))
        w = self.packed(kind == vrpx.IRP, dev)
        tape = torch.empty((Tmax, R), dtype=torch.uint8, device=dev)
        logp = torch.empty((R,), dtype=torch.float32, device=dev)
        cost = torch.empty((R,), dtype=torch.float32, device=dev)
        steps = torch.zeros((1,), dtype=torch.int32, device=dev)
        logits = torch.empty((Tmax, R, N), dtype=torch.float32, device=dev) if want_logits else None
        nbytes = int(L.vrpx_rollout_samples_workspace_bytes(kind, B, K, N))
        ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
        trace, saved = None, None
        if save_for_backward:
            saved = {"mask_hist": torch.empty((Tmax, R, 4), dtype=torch.int32, device=dev),
                     "load_hist": torch.empty((Tmax, R), dtype=torch.float32, device=dev),
                     "qg0": torch.empty((R, 1024), dtype=torch.float32, device=dev)}
            trace = vrpx.RolloutTrace(saved["mask_hist"].data_ptr(), saved["load_hist"].data_ptr(), saved["qg0"].data_ptr())
        vrpx.check(L.vrpx_rollout_samples_traced(C.byref(v), C.byref(w), vrpx.ptr(h), B, K, G, C.c_uint64(seed),
                                                 C.c_uint64(offset), vrpx.ptr(tape), Tmax, vrpx.ptr(logp), vrpx.ptr(cost),
                                                 vrpx.ptr(steps), vrpx.ptr(logits),
                                                 C.byref(trace) if trace is not None else None, vrpx.ptr(ws), nbytes, st))
        T = int(steps.item())
        out = {"cost": cost.view(K, B), "logp": logp.view(K, B), "steps": T, "tape": tape[:T].view(T, K, B),
               "coupling": G, "samples": K}
        if saved is not None:
            o = int(L.vrpx_rollout_workspace_qg_offset())
            saved["qg"] = ws[o:o + R * 4096].view(torch.float32).view(R, 1024)  # Q~g incl. the `first` fold, per replica
            saved["ws"] = ws
            saved["replicas"] = v
            saved["replica_arrays"] = (xy, depot, demand, visited, mask, cur, load)
            out["saved"] = saved
        if logits is not None:
            out["logits"] = logits[:T].view(T, K, B, N)
        return out

    # ------------------------------------------------------------------ single-step entry (reference call style)
    def forward(self, node_embs: torch.Tensor, mask: torch.Tensor = None, load: torch.Tensor = None, C_: int = 10,
                rollout: bool = False, **kw):
        """One decode step: node_embs (B,N,128), mask (B,N) 0/1, load (B,) or None -> (next node (B,1) long,
        log-prob).  Greedy (`rollout=True`) returns zeros for the log-prob like the reference (:100)."""
        C_ = kw.pop("C", C_)
        assert C_ == 10, "the tanh clip is fixed at C=10 in the kernel (the reference never uses another value)"
        src = node_embs.device
        dev = vrpx.require_device(None if src.type != "cuda" else src)
        if next(self.parameters()).device != dev:
            self.to(dev)
        B, N, _ = node_embs.shape
        irp = load is not None
        ep = self._ep
        if ep is None:
            h = node_embs.detach().to(dev, torch.float32).contiguous()
            z = lambda *s, dt=torch.float64: torch.zeros(s, dtype=dt, device=dev)
            ep = {"t": 0, "h": h, "xy": z(B, N, 2), "depot": z(B, dt=torch.int32), "demand": z(B, N),
                  "visited": z(B, 4, dt=torch.int32), "cur": z(B, dt=torch.int32), "load": z(B) + 1,
                  "logp": z(B, dt=torch.float32), "cost": z(B, dt=torch.float32), "steps": z(1, dt=torch.int32),
                  "tape": z(1, B, dt=torch.uint8)}
            ep["mask"] = z(B, 4, dt=torch.int32) if irp else ep["visited"]
            nbytes = int(vrpx.lib().vrpx_rollout_workspace_bytes(B, N))
            ep["ws"], ep["ws_bytes"] = torch.empty((nbytes,), dtype=torch.uint8, device=dev), nbytes
            self._ep = ep
        v = vrpx.EnvView()
        v.kind, v.N, v.B = (vrpx.IRP if irp else vrpx.TSP), N, B
        v.xy, v.depot, v.demand = ep["xy"].data_ptr(), ep["depot"].data_ptr(), ep["demand"].data_ptr()
        v.visited, v.mask = ep["visited"].data_ptr(), ep["mask"].data_ptr()
        v.cur, v.load = ep["cur"].data_ptr(), ep["load"].data_ptr()
        L = vrpx.lib()
        st = vrpx.stream_ptr(dev)
        if irp:
            ep["load"].copy_(load.detach().to(dev, torch.float64).reshape(B))
        m = mask.detach().to(dev, torch.float64).contiguous()
        vrpx.check(L.vrpx_env_set_visited(C.byref(v), vrpx.ptr(m), st))
        w = self.packed(irp, dev)
        seed = int(torch.randint(0, 2 ** 62, (1,)).item()) if not rollout else 0
        prev_logp = ep["logp"].clone()
        vrpx.check(L.vrpx_rollout(C.byref(v), C.byref(w), vrpx.ptr(ep["h"]), vrpx.GREEDY if rollout else vrpx.SAMPLE,
                                  B, C.c_uint64(seed), C.c_uint64(0), vrpx.ptr(ep["tape"]), ep["t"], 1,
                                  vrpx.ptr(ep["logp"]), vrpx.ptr(ep["cost"]), vrpx.ptr(ep["steps"]), None, None,
                                  vrpx.ptr(ep["ws"]), ep["ws_bytes"], st))
        nn_idx = ep["tape"][0].to(torch.long)
        ep["cur"].copy_(nn_idx.to(torch.int32))
        step_logp = ep["logp"] - (prev_logp if ep["t"] > 0 else 0)
        ep["t"] += 1
        # reference bookkeeping (graph_decoder.py:108-113)
        self.last_ = ep["h"][torch.arange(B, device=dev), nn_idx][:, None, :].to(src)
        if self.first_step:
            self.first_ = self.last_
            self.first_step = False
        if rollout:
            return nn_idx[:, None].to(src), torch.zeros(size=(B,))
        return nn_idx[:, None].to(src), step_logp[:, None].to(src)

    def reset(self):
        """Forget the episode state; must be called before a new game (reference :117-124)."""
        self.first_ = None
        self.last_ = None
        self.first_step = True
        self._ep = None


def _max_steps(kind: int, N: int) -> int:
    """Rows of an episode's tape: a TSP tour visits N - 1 nodes, a VRP / IRP episode takes at most 2 (N - 1) + 1 steps."""
    return (N - 1) if kind == vrpx.TSP else 2 * (N - 1) + 1


def check_samples(env, num_samples, coupling=None, train: bool = False):
    """Arguments of a K-sample rollout of env, checked before any work is done: returns (K, coupling group G).  train:
    the rollout is recorded for the backward, which replays the table-mode decode loop (vrpx_rollout_samples_traced)."""
    K = int(num_samples)
    if K < 1:
        raise ValueError(f"num_samples must be at least 1, got {num_samples}")
    G = _coupling_group(coupling, env.batch_size)
    if train and _max_steps(env._KIND, env.num_nodes) < 3:
        raise ValueError(f"training on K sampled tours needs the table-mode decode loop, which TSP with N <= 3 does not "
                         f"have (N = {env.num_nodes}); train on the K-fold replicated env instead")
    return K, G


def _coupling_group(coupling, B: int) -> int:
    G = B if coupling is None else int(coupling)
    if G < 0 or (G != 0 and (G > B or B % G != 0)):
        raise ValueError(f"coupling group {G} must be 0 or a divisor of the batch size {B}: attention row (b, head) "
                         "reads the mask of instance (8b + head) mod G of its group (graph_decoder.py:93)")
    return G
