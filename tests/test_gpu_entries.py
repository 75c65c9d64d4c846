"""GPU tests of the module-level entry points the reference's own tests call directly (tests/test_agent.py:24-54):
`GraphEncoder(node_input_dim)(x)`, `GraphDemandEncoder(...)(x, depot_mask)` and the SINGLE-STEP
`GraphDecoder(v_dim, k_dim)(embs, mask[, load])` — the resumable `vrpx_rollout` launch (t_begin > 0) fed through
`vrpx_env_set_visited` — each compared with the oracle over a whole episode, plus the multi-device / bad-coupling
argument handling of the C ABI."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _rel(got, ref):
    return float((np.abs(got - ref) / np.maximum(np.abs(ref), 1.0)).max())


def _sd(module, prefix):
    return {prefix + k: v.detach().float().cpu() for k, v in module.state_dict().items()}


@pytest.mark.parametrize("train", [True, False], ids=["train_bn", "eval_bn"])
def test_graph_encoder_entry(train):
    """reference tests/test_agent.py:24-31 (shape) + values: a freshly built module is in train mode there."""
    from agents import GraphEncoder
    from gym_vrp.envs import VRPEnv
    from oracle import policy_oracle as po

    torch.manual_seed(69)
    np.random.seed(69)
    env = VRPEnv(num_nodes=8, batch_size=2, num_draw=1)
    state = torch.from_numpy(env.reset()).float()
    encoder = GraphEncoder(node_input_dim=2)
    encoder.train(train)
    emb = encoder(state[:, :, :2])
    assert emb.shape == (2, 8, 128) and emb.device.type == "cpu"     # result follows the input's device
    ref = po.encoder_forward(_sd(encoder, "encoder."), state[:, :, :2], None, train)
    assert _rel(emb.numpy(), ref.numpy()) < (1e-4 if train else 1e-5)
    # larger, CUDA input stays on the device
    x = torch.rand(64, 50, 2, device="cuda")
    encoder.eval()
    h = encoder(x)
    assert h.is_cuda
    ref = po.encoder_forward(_sd(encoder, "encoder."), x.cpu(), None, False)
    assert _rel(h.cpu().numpy(), ref.numpy()) < 1e-5


def test_graph_demand_encoder_entry():
    """GraphDemandEncoder.forward(x, depot_mask) (graph_encoder.py:95-138): depot rows through depot_embed."""
    from agents import GraphDemandEncoder
    from oracle import policy_oracle as po

    torch.manual_seed(3)
    for f, B, N in ((2, 5, 20), (3, 33, 40)):
        enc = GraphDemandEncoder(depot_input_dim=2, node_input_dim=f)
        enc.eval()
        x = torch.rand(B, N, f)
        depot = torch.randint(0, N, (B,))
        mask = torch.zeros(B, N, dtype=torch.bool)
        mask[torch.arange(B), depot] = True
        h = enc(x, mask)
        ref = po.encoder_forward(_sd(enc, "encoder."), x, mask, False)
        assert h.shape == (B, N, 128)
        assert _rel(h.numpy(), ref.numpy()) < 1e-5


@pytest.mark.parametrize("kind,N,B", [("tsp", 8, 2), ("vrp", 20, 16), ("irp", 30, 9), ("tsp", 128, 3), ("vrp", 65, 5),
                                      ("irp", 97, 4)])
def test_single_step_decoder_episode_vs_oracle(kind, N, B):
    """Drive a whole episode the way the reference's model loop does (graph_tsp_agent.py:78-88): per step
    `decoder(emb, mask[, load], rollout=True)` -> env step on the host (env oracle) -> next mask.  Every greedy action is
    the oracle's argmax (up to near-ties) and `first_/last_` follow the reference bookkeeping (graph_decoder.py:108-113).
    A second pass in sampling mode checks the per-step log-prob of the sampled node against the oracle's."""
    from agents import GraphDecoder
    from oracle import policy_oracle as po
    from oracle.env_oracle import EnvOracle, draw_instances

    torch.manual_seed(11)
    np.random.seed(11)
    xy, depot, demand = draw_instances(B, N)
    decoder = GraphDecoder(v_dim=128, k_dim=128)
    emb = torch.randn(B, N, 128) * 0.7
    sd = _sd(decoder, "decoder.")
    E = 128
    for greedy in (True, False):
        env = EnvOracle(kind, xy, depot, demand)
        st = env.get_state()
        first = sd["decoder._first_node"].reshape(1, E).repeat(B, 1)
        last = sd["decoder._last_node"].reshape(1, E).repeat(B, 1)
        done, t = False, 0
        while not done:
            load = None
            if kind == "irp":
                st, load_np = st
                load = torch.tensor(load_np, dtype=torch.float)
            mask = torch.tensor(st[:, :, -1], dtype=torch.float)
            if kind == "irp":
                nxt, logp = decoder(emb, mask, load=load, rollout=greedy)
            else:
                nxt, logp = decoder(emb, mask, rollout=greedy)
            assert nxt.shape == (B, 1) and nxt.dtype == torch.long
            u = po.decoder_logits(sd, emb, mask, first, last, load)
            a = nxt[:, 0]
            chosen = u[torch.arange(B), a]
            assert torch.isfinite(chosen).all(), "a masked node was chosen"
            if greedy:
                assert (chosen >= u.max(dim=1).values - 2e-5).all(), (kind, t)
                assert float(torch.as_tensor(logp).abs().max()) == 0.0      # graph_decoder.py:100
            else:
                ref_lp = chosen - torch.logsumexp(u, dim=-1)
                assert np.allclose(logp.reshape(B).numpy(), ref_lp.numpy(), rtol=1e-5, atol=2e-5), (kind, t)
            last = emb[torch.arange(B), a]
            if t == 0:
                first = last
            assert torch.equal(decoder.last_[:, 0].cpu(), last)
            assert torch.equal(decoder.first_[:, 0].cpu(), first)
            st, _, done, _ = env.step(a.numpy()[:, None])
            t += 1
        assert t >= N - 1
        decoder.reset()
        assert decoder.first_ is None and decoder.first_step


def test_reference_test_decoder_call_shape():
    """reference tests/test_agent.py:34-54 call pattern (the asserted sample [[5],[7]] depends on torch.multinomial's
    CPU stream and no longer reproduces in the reference itself, SURVEY §4): shapes / dtypes / feasibility."""
    from agents import GraphDecoder, GraphEncoder
    from gym_vrp.envs import VRPEnv

    torch.manual_seed(69)
    np.random.seed(69)
    env = VRPEnv(num_nodes=8, batch_size=2, num_draw=1)
    state = torch.from_numpy(env.reset()).float()
    encoder = GraphEncoder(node_input_dim=2)
    decoder = GraphDecoder(v_dim=128, k_dim=128)
    embs = encoder(state[:, :, :2])
    mask = torch.zeros(size=(2, 8))
    next_node, logp = decoder(embs, mask)
    assert next_node.shape == (2, 1) and next_node.dtype == torch.long
    assert ((next_node >= 0) & (next_node < 8)).all() and (logp <= 0).all()


def test_bad_coupling_is_an_argument_error():
    """ADVICE r1: a coupling group that does not divide the batch would index masks outside the batch."""
    from agents import TSPAgent
    from gym_vrp.envs import TSPEnv

    agent = TSPAgent(seed=1)
    for bad in (1000, 7, 100000):
        env = TSPEnv(10, 2500 if bad == 1000 else 64, 0, seed=1, instance_rng="philox")
        agent.model.coupling = bad
        with pytest.raises(ValueError):
            agent.evaluate(env)
    env = TSPEnv(10, 64, 0, seed=1, instance_rng="philox")
    agent.model.coupling = 16
    assert torch.isfinite(agent.evaluate(env)).all()


def test_env_edit_reaches_encoder_and_irp_mask():
    """ADVICE r1: host-side write-through edits are uploaded before the encoder runs, and an IRP demand edit refreshes
    the `demand - load > 0` mask of the current state."""
    from agents import IRPAgent
    from gym_vrp.envs import IRPEnv

    env = IRPEnv(6, 4, 1, seed=5)
    agent = IRPAgent(seed=5)
    base = agent.evaluate(env).cpu().numpy()
    env2 = IRPEnv(6, 4, 1, seed=5)
    n = int((env2.depots[0, 0] + 1) % 6)
    env2.sampler.graphs[0].nodes[n]["coordinates"] = np.array([0.123, 0.987])
    env2.sampler.graphs[1].nodes[int((env2.depots[1, 0] + 1) % 6)]["demand"] = np.array([5.0])   # exceeds any load
    m = env2.generate_mask()
    assert m[1, int((env2.depots[1, 0] + 1) % 6)] == 1.0, "IRP mask not refreshed after a demand edit"
    with torch.no_grad():
        agent.model.eval()
        agent.model(env2, rollout=True)
    emb = agent.model.last_rollout["emb"]
    env3 = IRPEnv.from_arrays(env2.sampler.get_graph_positions(), env2.sampler.get_depots()[:, 0], env2.sampler.get_demands()[:, :, 0])
    from agents.graph_encoder import run_encoder

    ref = run_encoder(agent.model.encoder, env=env3, depot=env3._depot)
    assert torch.equal(emb, ref), "the encoder read stale device coordinates"
    assert base.shape == (4,)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_non_current_device():
    """ADVICE r1: buffers on cuda:1 while cuda:0 is current — the library runs on the owner of the buffers."""
    from agents import TSPAgent
    from gym_vrp.envs import TSPEnv

    torch.cuda.set_device(0)
    env0 = TSPEnv(20, 64, 0, seed=2, device="cuda:0", instance_rng="numpy")
    env1 = TSPEnv(20, 64, 0, seed=2, device="cuda:1", instance_rng="numpy")
    a0, a1 = TSPAgent(seed=2), TSPAgent(seed=2)
    l0 = a0.evaluate(env0)
    l1 = a1.evaluate(env1)
    assert l1.device.index == 1 and torch.equal(l0.cpu(), l1.cpu())
