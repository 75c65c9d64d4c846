"""Graph encoders — parameter containers whose forward pass runs on libvrpx (sm_100a CUDA).

State-dict layout and construction order equal the reference (agents/graph_encoder.py:6-198) so that
checkpoints interchange and `torch.manual_seed(s)` yields the same initial weights:
    encoder.node_embed, [encoder.depot_embed], encoder.attention_layers.{0,1,2}.{attention_layer, bn1.norm,
    bn2.norm, ff.0, ff.2}.
The arithmetic (embedding, 3 x {MHA + skip + BatchNorm, FF + skip + BatchNorm}) is `vrpx_encoder_forward`:
tcgen05 tensor-core GEMMs (kind::f16 on f16 hi/lo operand halves, ~fp32 accuracy) for the dense layers, a fused per-instance attention kernel, BatchNorm in
eval (running statistics) or train (batch statistics over all B*N rows) mode.
"""
from __future__ import annotations

import ctypes as C

import torch
import torch.nn as nn

import vrpx
from vrpx import packing


class BatchNorm(nn.Module):
    """Holds the BatchNorm1d parameters/buffers applied over flattened (B*N, E) rows (reference :141-154)."""

    def __init__(self, feature_dim: int):
        super().__init__()
        self.norm = nn.BatchNorm1d(feature_dim)


class MultiHeadAttentionLayer(nn.Module):
    """Parameters of one encoder layer: self-attention, two BatchNorms, feed-forward (reference :157-198)."""

    def __init__(self, embedding_dim: int, hidden_dim: int, num_heads: int):
        super().__init__()
        self.attention_layer = nn.MultiheadAttention(embed_dim=embedding_dim, num_heads=num_heads, batch_first=True)
        self.bn1 = BatchNorm(embedding_dim)
        self.bn2 = BatchNorm(embedding_dim)
        self.ff = nn.Sequential(nn.Linear(embedding_dim, hidden_dim), nn.ReLU(), nn.Linear(hidden_dim, embedding_dim))


def run_encoder(enc: "GraphEncoder", *, env=None, x=None, depot=None, gemm_path: int = 0, save: bool = False):
    """Launch vrpx_encoder_forward.  Features come from a device-resident env or from x (B,N,f) f32 CUDA;
    depot (B,) int32 CUDA or None.  Returns h (B,N,128) f32 on the device; with save=True (train mode only) returns
    (h, saved) where `saved` holds the activations vrpx_encoder_backward needs."""
    dev = vrpx.require_device(env._device if env is not None else x.device)
    if next(enc.parameters()).device != dev:
        enc.to(dev)
    w = packing.encoder_struct(enc, dev)
    if env is not None:
        B, N = env.batch_size, env.num_nodes
    else:
        B, N = int(x.shape[0]), int(x.shape[1])
    h = torch.empty((B, N, vrpx.EMB), dtype=torch.float32, device=dev)
    L = vrpx.lib()
    train = 1 if enc.training else 0
    need = int(L.vrpx_encoder_workspace_bytes(B, N))
    if not train:  # eval mode is per-instance: cap the scratch and let the library chunk the batch
        need = min(need, max(int(L.vrpx_encoder_workspace_bytes(1, N)), 8 << 30))
    ws = torch.empty((need,), dtype=torch.uint8, device=dev)
    saved = None
    if save:
        assert train, "activations are only saved in train mode"
        saved = torch.empty((int(L.vrpx_encoder_saved_bytes(B, N)) // 4,), dtype=torch.float32, device=dev)
    view = env._view() if env is not None else None
    vrpx.check(L.vrpx_encoder_forward(C.byref(w), C.byref(view) if view is not None else None,
                                      vrpx.ptr(x) if x is not None else None,
                                      vrpx.ptr(depot) if depot is not None else None,
                                      B, N, train, vrpx.ptr(h), vrpx.ptr(ws), need, gemm_path,
                                      vrpx.ptr(saved) if saved is not None else None, vrpx.stream_ptr(dev)))
    if train:
        for layer in enc.attention_layers:  # BatchNorm1d bookkeeping the kernel does not touch
            layer.bn1.norm.num_batches_tracked += 1
            layer.bn2.norm.num_batches_tracked += 1
    return (h, saved) if save else h


class GraphEncoder(nn.Module):
    def __init__(self, node_input_dim: int, embedding_dim: int = 128, hidden_dim: int = 512,
                 num_attention_layers: int = 3, num_heads: int = 8):
        super().__init__()
        assert (embedding_dim, hidden_dim, num_attention_layers, num_heads) == (128, 512, 3, 8), \
            "libvrpx kernels are specialised for E=128, F=512, L=3, H=8 (the reference's only configuration)"
        self.node_embed = nn.Linear(node_input_dim, embedding_dim)
        self.attention_layers = nn.ModuleList(
            [MultiHeadAttentionLayer(embedding_dim=embedding_dim, hidden_dim=hidden_dim, num_heads=num_heads)
             for _ in range(num_attention_layers)])
        # 0: tcgen05 f16-split (production), 1: fp32 SIMT GEMMs (cross-check); the backward's weight gradients run on
        # tcgen05 on both paths once B*N >= 8192 rows (vrpx/backward.py)
        self.gemm_path = 0

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """x (num_graphs, num_nodes, f) -> embeddings (num_graphs, num_nodes, 128), on x's device."""
        src = x.device
        dev = vrpx.require_device(None if src.type != "cuda" else src)
        xd = x.detach().to(dev, torch.float32).contiguous()
        h = run_encoder(self, x=xd, gemm_path=self.gemm_path)
        return h.to(src)


class GraphDemandEncoder(GraphEncoder):
    def __init__(self, depot_input_dim: int, node_input_dim: int, embedding_dim: int = 128, hidden_dim: int = 512,
                 num_attention_layers: int = 3, num_heads: int = 8):
        super().__init__(node_input_dim=node_input_dim, embedding_dim=embedding_dim, hidden_dim=hidden_dim,
                         num_attention_layers=num_attention_layers, num_heads=num_heads)
        assert depot_input_dim == 2, "depot rows are embedded from their (x, y) coordinates"
        self.node_f_dim = node_input_dim
        self.depot_f_dim = depot_input_dim
        self.emb_dim = embedding_dim
        self.depot_embed = nn.Linear(depot_input_dim, embedding_dim)

    def forward(self, x: torch.Tensor, depot_mask: torch.Tensor) -> torch.Tensor:
        """x (B,N,f); depot_mask (B,N) bool with one depot per graph (reference :95-138: the depot row goes
        through depot_embed, every other row through node_embed — a per-row select in the kernel)."""
        src = x.device
        dev = vrpx.require_device(None if src.type != "cuda" else src)
        xd = x.detach().to(dev, torch.float32).contiguous()
        depot = depot_mask.to(dev).to(torch.uint8).argmax(dim=1).to(torch.int32).contiguous()
        h = run_encoder(self, x=xd, depot=depot, gemm_path=self.gemm_path)
        return h.to(src)
