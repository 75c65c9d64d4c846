"""CPU-only checks: the C-ABI library loads and exports every symbol include/vrpx.h declares (no compute calls),
the product refuses to run without a GPU (no CPU fallback), and the host-side instance store mirrors the
reference's VRPGraph / VRPNetwork behaviour (reference tests/test_graph.py)."""
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "vrpx.h")).read()
    return sorted(set(re.findall(r"VRPX_API\s+[\w\s\*]+?\b(vrpx_\w+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    import vrpx

    L = vrpx.lib()
    names = _declared_symbols()
    assert len(names) >= 14, names
    for n in names:
        assert hasattr(L, n), f"libvrpx.so does not export {n}"
    assert L.vrpx_abi_version() == vrpx.ABI_VERSION
    header = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'include', 'vrpx.h')).read()
    assert f'#define VRPX_ABI_VERSION {vrpx.ABI_VERSION}' in header
    assert L.vrpx_launch_count() == 0


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_no_cpu_fallback():
    import vrpx
    from gym_vrp.envs import TSPEnv

    assert vrpx.lib().vrpx_device_check(0) < 0
    assert b"no CUDA device" in vrpx.lib().vrpx_last_error() or b"device" in vrpx.lib().vrpx_last_error()
    with pytest.raises(vrpx.VrpxError):
        vrpx.require_device()
    with pytest.raises(RuntimeError):
        TSPEnv(num_nodes=5, batch_size=2, num_draw=1)
    from agents import GraphEncoder

    with pytest.raises(RuntimeError):
        GraphEncoder(node_input_dim=2)(torch.zeros(2, 5, 2))


# ---- reference tests/test_graph.py on the SoA-backed host classes
def test_vrp_graph_init():
    from gym_vrp.graph.vrp_graph import VRPGraph
    import networkx as nx

    np.random.seed(69)
    graph = VRPGraph(10, 5)
    depots = list(nx.get_node_attributes(graph.graph, "depot").values())
    assert len(graph.nodes) == 10
    assert depots.count(1) == 5


def test_vrp_euclid_dist_write_through():
    from gym_vrp.graph.vrp_graph import VRPGraph
    import networkx as nx

    np.random.seed(69)
    graph = VRPGraph(2, 1)
    nx.set_node_attributes(graph, {0: np.array([2, -1]), 1: np.array([-2, 2])}, "coordinates")
    assert graph.euclid_distance(0, 1) == 5


def test_vrp_network_init_and_stream_order():
    from gym_vrp.graph.vrp_network import VRPNetwork
    from oracle.env_oracle import draw_instances

    np.random.seed(69)
    net = VRPNetwork(num_graphs=10, num_nodes=10, num_depots=2)
    assert len(net.graphs) == 10
    depots = net.get_depots()
    assert depots.shape == (10, 2) and np.unique(depots, axis=0).shape[0] > 1
    # single-depot stream equals the oracle's restatement of the reference order
    np.random.seed(5)
    net = VRPNetwork(7, 13, 1)
    np.random.seed(5)
    xy, depot, demand = draw_instances(7, 13)
    assert np.array_equal(net.get_graph_positions(), xy)
    assert np.array_equal(net.get_depots()[:, 0], depot)
    assert np.array_equal(net.get_demands()[:, :, 0], demand)
    v0 = net.version
    net.graphs[3].nodes[2]["coordinates"] = np.array([0.25, 0.75])
    assert net.version == v0 + 1 and np.array_equal(net.get_graph_positions()[3, 2], [0.25, 0.75])
    assert net.get_demands().shape == (7, 13, 1)
    with pytest.raises(AssertionError):
        VRPNetwork(2, 3, 4)


def test_state_dict_layout_matches_reference_keys():
    """SURVEY App. A.5: 67 tensors (TSP) / 69 (VRP, IRP) with the reference's names and shapes."""
    from agents import IRPAgent, TSPAgent, VRPAgent

    sd = TSPAgent(seed=1).model.state_dict()
    assert len(sd) == 67
    assert sd["encoder.attention_layers.2.attention_layer.in_proj_weight"].shape == (384, 128)
    assert sd["encoder.attention_layers.0.ff.0.weight"].shape == (512, 128)
    assert sd["encoder.attention_layers.1.bn2.norm.running_var"].shape == (128,)
    assert sd["decoder._first_node"].shape == (1, 1, 128)
    assert sd["decoder.attention.q_proj_weight"].shape == (384, 384)
    assert sd["decoder.attention.k_proj_weight"].shape == (384, 128)
    assert sd["decoder.attention.in_proj_bias"].shape == (1152,)
    assert sd["decoder._context_proj.weight"].shape == (384, 257)
    assert sd["decoder._att_output.weight"].shape == (128, 384)
    for A, f in ((VRPAgent, 2), (IRPAgent, 3)):
        sd = A(seed=1).model.state_dict()
        assert len(sd) == 69
        assert sd["encoder.node_embed.weight"].shape == (128, f)
        assert sd["encoder.depot_embed.weight"].shape == (128, 2)


# ---- sizes of the rollout workspace (pure arithmetic entry points: callable without a GPU)
def test_rollout_workspace_layout_is_consistent():
    import vrpx

    L = vrpx.lib()
    off = int(L.vrpx_rollout_workspace_qg_offset())
    assert off % 256 == 0 and off >= 4096 + 512 * 1024      # header + pre-split m_t in front of the Q~g table
    for kind in (vrpx.TSP, vrpx.VRP, vrpx.IRP):
        prev_plain = prev_table = 0
        for B, N in [(1, 4), (64, 20), (4096, 40), (65536, 50), (131072, 100)]:
            plain = int(L.vrpx_rollout_workspace_bytes(B, N))
            table = int(L.vrpx_rollout_table_workspace_bytes(kind, B, N))
            # Q~g [B][1024] f32 right behind the header, then the two glimpse-mask snapshots [2][B][4] u32
            assert plain == off + B * 1024 * 4 + 2 * B * 16
            # the table workspace also holds S0 (, SL), S1 [B][N][8][N], c [B][1024], q^ [B][128], m_t^T
            floor = plain + B * 8 * N * 4 + B * N * 8 * N * 4 + B * 1024 * 4 + B * 128 * 4 + 1024 * 128 * 4
            assert table >= floor, (kind, B, N, table, floor)
            assert table % 256 == 0
            assert plain > prev_plain and table > prev_table
            prev_plain, prev_table = plain, table
        if kind == vrpx.IRP:                                  # IRP carries the extra load table SL [B][8][N]
            assert int(L.vrpx_rollout_table_workspace_bytes(vrpx.IRP, 4096, 40)) > int(
                L.vrpx_rollout_table_workspace_bytes(vrpx.TSP, 4096, 40))


# ---- precision policy of the tensor-core contractions (csrc/f16split.cuh), restated in numpy
def _split_f16(x, scale):
    hi = x.astype(np.float16)
    lo = ((x - hi.astype(np.float32)) * np.float32(scale)).astype(np.float16)
    return hi, lo


@pytest.mark.parametrize("scale", [1.0, 2048.0], ids=["unscaled_lo", "scaled_lo"])
def test_f16_hi_lo_split_keeps_fp32_accuracy(scale):
    """x = hi + lo / scale with hi = f16(x), lo = f16((x - hi) * scale) carries ~22 significant bits, and the three-term
    product hi·hi + (lo·hi + hi·lo) / scale reproduces an fp32 dot product to ~1e-6 of its scale (the kernels accumulate
    in fp32 on the tensor cores; here float64 sums isolate the operand error)."""
    rs = np.random.RandomState(0)
    x = (rs.randn(256, 512) * 2.0).astype(np.float32)          # activations after BatchNorm: O(1)
    w = (rs.randn(512, 64) / np.sqrt(512)).astype(np.float32)  # weights: O(1/sqrt(K))
    if scale == 1.0:
        w = w * np.float32(256.0)                              # the GEMM scales W by 2^8 before the unscaled split
    xh, xl = _split_f16(x, scale)
    wh, wl = _split_f16(w, scale)
    rec = xh.astype(np.float64) + xl.astype(np.float64) / scale
    big = np.abs(x) >= 0.25                                    # below, an unscaled lo is a subnormal f16: absolute 2^-25
    assert np.max(np.abs(rec - x)[big] / np.abs(x)[big]) < 2.0 ** -21
    assert np.max(np.abs(rec - x)) < 2.0 ** -20 * np.abs(x).max()
    f = lambda a: a.astype(np.float64)
    got = f(xh) @ f(wh) + (f(xl) @ f(wh) + f(xh) @ f(wl)) / scale
    ref = f(x) @ f(w)
    assert np.max(np.abs(got - ref)) < 2e-6 * np.abs(ref).max()
    # a single f16 (or TF32) pass would miss the bar by three orders of magnitude
    assert np.max(np.abs(f(xh) @ f(wh) - ref)) > 1e-4 * np.abs(ref).max()


def test_gradient_gain_is_an_exact_power_of_two_in_range():
    """vrpx/backward.py::_grad_gain: the gain that brings a gradient tensor into the range of the f16-split GEMMs is a
    power of two (exact to apply and to undo), puts the largest element in [2^(t-1), 2^t), and is 1 for empty / zero /
    non-finite inputs; the numpy restatement of the split shows what it buys: a 1e-6-sized operand keeps ~13 bits
    unscaled (2^8 only) and ~21 bits with the gain."""
    import math
    import sys

    sys.path.insert(0, os.path.join(ROOT, "vrp-gym_b200"))
    from vrpx import backward as vb

    rs = np.random.RandomState(1)
    for mag in (1e-9, 3e-6, 0.02, 1.0, 77.0, 5e4):
        t = torch.from_numpy((rs.randn(64, 128) * mag).astype(np.float32))
        for target in (-6, -2):
            g = vb._grad_gain(t, target)
            assert math.frexp(g)[0] == 0.5                                        # a power of two
            top = float(t.abs().max()) * g
            assert 2.0 ** (target - 1) <= top < 2.0 ** target, (mag, target, top)
    assert vb._grad_gain(torch.zeros(4, 4)) == 1.0
    assert vb._grad_gain(torch.tensor([float("nan"), 1.0])) == 1.0
    assert vb._grad_gain(torch.tensor([float("inf"), 1.0])) == 1.0
    # what the gain buys, on the numpy restatement of the operand split (scale 2^8, unscaled lo half)
    x = (rs.randn(4096) * 1e-6).astype(np.float32)

    def rel_err(v):
        s = v * np.float32(256.0)
        hi, lo = _split_f16(s, 1.0)
        rec = hi.astype(np.float64) + lo.astype(np.float64)
        big = np.abs(v) > 0.1 * np.abs(v).max()
        return np.max(np.abs(rec - s)[big] / np.abs(s)[big])

    g = vb._grad_gain(torch.from_numpy(x))
    assert rel_err(x) > 2.0 ** -15                       # ~13 bits: the lo half is a subnormal
    assert rel_err(x * np.float32(g)) < 2.0 ** -17       # the gain moves it back into the normal range
