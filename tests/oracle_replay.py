"""Replay of a kernel's action tape on the env oracle, for the float64 reference tests (test_gpu_backward_scale.py,
test_gpu_node_edges.py).  Test helper only: the masks and loads every step saw, the glimpse-mask partner rows, and the
bar on summed log-probs."""
import numpy as np
import torch

F64 = torch.float64


def host_inputs(kind, env, tape):
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


def partners(B, G):
    """(B, 8): the instance whose mask attention row (b, head) adds, g0 + ((b - g0) * 8 + head) mod G with g0 the first
    instance of b's coupling group (graph_decoder.py:93-94, `mask.repeat(H, 1)` within a group of G instances)."""
    b = torch.arange(B)[:, None]
    g0 = b // G * G
    return g0 + ((b - g0) * 8 + torch.arange(8)[None, :]) % G


def check_logp(logp_ref, logp_gpu, T):
    """The kernel's sampled log-probs are the teacher-forced ones of the reference: the mask history is the same.
    Returns the largest difference."""
    d = (logp_ref - logp_gpu.to(F64)).abs()
    bar = 1e-5 * logp_ref.abs() + 1e-5 * T
    assert bool((d <= bar).all()), ("log-prob sums differ from the float64 replay", float(d.max()))
    return float(d.max())
