"""GPU parity of the hand-written REINFORCE backward (csrc/decoder_bwd.cu, csrc/encoder_bwd.cu, vrpx/backward.py)
against (a) torch autograd on the fp32 oracle for dL/dh and the decoder parameters, and (b) the gradients the
UNMODIFIED reference produced for the same teacher-forced tape (tests/golden/policy_*.npz: per-parameter gradient
norms and leading elements; train-mode BatchNorm, loss = mean(advantage * log_prob), graph_tsp_agent.py:179-186).

These run at B <= 32 (N 4 ... 20): `k_decoder_bwd` is a single CTA, glimpse-mask partners stay in the instance's own
tile and the weight gradients stay on the warp-level GEMMs.  The large-batch paths of the same backward (multi-CTA tile
loop, far partners, coupling groups, `k_gemm_tn_tc`, train-step gradient magnitudes, the C4 shape) are checked against
float64 in tests/test_gpu_backward_scale.py."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

CASES = [(4, 2, 69), (10, 8, 7), (20, 32, 1234)]


def _cls(kind):
    from agents import IRPAgent, TSPAgent, VRPAgent
    from gym_vrp.envs import IRPEnv, TSPEnv, VRPEnv

    return {"tsp": (TSPEnv, TSPAgent), "vrp": (VRPEnv, VRPAgent), "irp": (IRPEnv, IRPAgent)}[kind]


def _oracle_logp_from_h(sd, kind, xy, depot, demand, h, tape):
    """Teacher-forced sum of log-probs as a differentiable function of h (oracle decoder + oracle env)."""
    from oracle import policy_oracle as po
    from oracle.env_oracle import EnvOracle

    env = EnvOracle(kind, xy, depot, demand)
    st = env.get_state()
    load = None
    if kind == "irp":
        st, load = st
    B, N = st.shape[:2]
    E = h.shape[-1]
    first = sd["decoder._first_node"].reshape(1, E).repeat(B, 1)
    last = sd["decoder._last_node"].reshape(1, E).repeat(B, 1)
    total = torch.zeros(B)
    for t in range(tape.shape[0]):
        mask = torch.tensor(st[:, :, -1], dtype=torch.float)
        ld = torch.tensor(load, dtype=torch.float) if kind == "irp" else None
        u = po.decoder_logits(sd, h, mask, first, last, ld)
        a = torch.as_tensor(tape[t], dtype=torch.long)
        total = total + u.gather(1, a[:, None])[:, 0] - torch.logsumexp(u, dim=-1)
        last = h[torch.arange(B), a]
        if t == 0:
            first = last
        st = env.step(tape[t][:, None])[0]
        if kind == "irp":
            st, load = st
    return total


@pytest.mark.parametrize("kind", ["tsp", "vrp", "irp"])
def test_decoder_backward_vs_oracle_autograd(golden_dir, kind):
    from vrpx import backward as bw

    z = np.load(os.path.join(golden_dir, f"policy_{kind}.npz"))
    Env, Agent = _cls(kind)
    for N, B, seed in CASES[1:]:
        key = f"{N}_{B}_{seed}"
        tape = z[key + "/tf_tape"]
        agent = Agent(seed=seed)
        model = agent.model
        model.train()
        env = Env(N, B, 1, seed)
        s = env.sampler
        xy, depot, demand = s.get_graph_positions(), s.get_depots()[:, 0], s.get_demands()[:, :, 0]
        loss, logp = model(env, rollout=False, tape=tape)
        ctx = model.last_rollout
        h = ctx["emb"]
        wts = torch.linspace(-1.0, 1.0, B)
        model.zero_grad()
        dH = bw.decoder_backward(model.decoder, env, h, ctx, wts, gemm_path=1).cpu()
        # oracle: same h, autograd
        sd = {k: v.detach().float().cpu().clone() for k, v in model.state_dict().items()}
        dec_keys = [k for k in sd if k.startswith("decoder.")]
        for k in dec_keys:
            sd[k].requires_grad_(True)
        h_ref = h.detach().cpu().clone().requires_grad_(True)
        total = _oracle_logp_from_h(sd, kind, xy, depot, demand, h_ref, tape)
        assert np.allclose(total.detach().numpy(), logp.detach().cpu().numpy(), rtol=1e-4, atol=1e-4)
        (total * wts).sum().backward()
        ref = h_ref.grad
        scale = ref.abs().max().item()
        assert (dH - ref).abs().max().item() <= 2e-4 * scale + 1e-7, (kind, key, (dH - ref).abs().max().item(), scale)
        for name, p in model.decoder.named_parameters():
            g_ref = sd["decoder." + name].grad
            if g_ref is None or g_ref.abs().max() == 0:
                assert p.grad is None or p.grad.abs().max().item() < 1e-6, name
                continue
            got = p.grad.cpu()
            sc = g_ref.abs().max().item()
            assert (got - g_ref).abs().max().item() <= 1e-3 * sc + 1e-7, (kind, key, name, (got - g_ref).abs().max().item(), sc)


@pytest.mark.parametrize("gemm_path", [1, 0], ids=["simt", "tcgen05"])
@pytest.mark.parametrize("kind", ["tsp", "vrp", "irp"])
def test_full_backward_matches_reference_gradients(golden_dir, kind, gemm_path):
    z = np.load(os.path.join(golden_dir, f"policy_{kind}.npz"))
    Env, Agent = _cls(kind)
    for N, B, seed in CASES:
        key = f"{N}_{B}_{seed}"
        tape = z[key + "/tf_tape"]
        agent = Agent(seed=seed)
        model = agent.model
        model.train()
        model.encoder.gemm_path = gemm_path
        env = Env(N, B, 1, seed)
        loss_m, logp = model(env, rollout=False, tape=tape)
        baseline = torch.tensor(z[key + "/greedy_loss"], device=loss_m.device)
        adv = (loss_m - baseline) * -1
        loss = (adv * logp).mean()
        assert np.isclose(loss.item(), float(z[key + "/train_loss"]), rtol=2e-3, atol=1e-5)
        model.zero_grad()
        model.backward(adv / B)
        tol = 3e-3 if gemm_path == 1 else 1e-2
        # Parameters that feed a train-mode BatchNorm only through a constant shift (out_proj.bias, ff.2.bias) or a
        # softmax-invariant shift (key biases) have a mathematically ZERO gradient: the reference's values there are
        # rounding noise (~1e-6 of the largest gradient).  They are compared against an absolute floor instead.
        gscale = max(float(z[k]) for k in z.files if k.startswith(f"{key}/grad_norm/"))
        floor = 3e-5 * gscale
        checked, bad = 0, []
        for name, p in model.named_parameters():
            kn, kh = f"{key}/grad_norm/{name}", f"{key}/grad_head/{name}"
            if kn not in z.files:
                assert p.grad is None or p.grad.abs().max().item() < 1e-6, f"{name}: reference has no gradient"
                continue
            ref_norm, ref_head = float(z[kn]), z[kh]
            got = p.grad.detach().reshape(-1).cpu()
            if abs(got.double().norm().item() - ref_norm) > tol * ref_norm + floor:
                bad.append((name, "norm", got.double().norm().item(), ref_norm))
            head_scale = max(np.abs(ref_head).max(), ref_norm / max(got.numel(), 1) ** 0.5)
            if np.abs(got[:16].numpy() - ref_head).max() > tol * head_scale + floor:
                bad.append((name, "head", float(np.abs(got[:16].numpy() - ref_head).max()), float(head_scale)))
            checked += 1
        assert not bad, (kind, key, gscale, bad)
        assert checked >= 44


def test_train_epoch_runs_and_improves():
    """A few REINFORCE epochs of the public train() on TSP-10: finite loss, weights move, baseline logic runs."""
    import tempfile

    from agents import TSPAgent
    from gym_vrp.envs import TSPEnv

    env = TSPEnv(num_nodes=10, batch_size=256, num_draw=1, seed=3)
    agent = TSPAgent(seed=3, lr=1e-3, csv_path=os.path.join(tempfile.mkdtemp(), "log.csv"))
    before = {k: v.clone() for k, v in agent.model.state_dict().items()}
    agent.train(env, epochs=3, eval_epochs=1, check_point_dir=tempfile.mkdtemp() + "/")
    moved = sum(float((v - before[k]).abs().sum()) for k, v in agent.model.state_dict().items() if v.dtype == torch.float32)
    assert moved > 0 and all(torch.isfinite(v).all() for v in agent.model.state_dict().values())
    rows = open(agent.csv_path).read().strip().splitlines()
    assert rows[0] == "Epoch,Loss,Cost,Advantage,Time" and len(rows) == 4


def test_encoder_gradients_do_not_depend_on_gradient_magnitude(golden_dir):
    """The REINFORCE gradient is linear in the advantage: grad(s * adv) / s must equal grad(adv).  Per-row gradients of a
    mean loss at a 65,536 batch are ~1e-5 of this 8-instance fixture's; without the power-of-two gain of
    vrpx/backward.py::encoder_backward the f16-split GEMMs of the encoder backward lost 0.3 % at s = 1e-5 and 24 % at
    s = 1e-7 (tools/grad_scale_probe.py)."""
    TSPEnv, TSPAgent = _cls("tsp")
    z = np.load(os.path.join(golden_dir, "policy_tsp_large.npz"))
    key, N, B, seed = "50_8_31", 50, 8, 31
    tape = z[key + "/tf_tape"]

    def grads(scale):
        model = TSPAgent(seed=seed).model
        model.train()
        env = TSPEnv(N, B, 1, seed)
        loss_m, _ = model(env, rollout=False, tape=tape)
        adv = (loss_m - torch.tensor(z[key + "/greedy_loss"], device=loss_m.device)) * -1
        model.zero_grad()
        model.backward(adv / B * scale)
        return {n: p.grad.detach().double().cpu() / scale for n, p in model.named_parameters() if p.grad is not None}

    ref = grads(1.0)
    gmax = max(g.abs().max().item() for g in ref.values())
    for s in (1e-5, 1e-7):
        got = grads(s)
        for n, g in ref.items():
            dev = (got[n] - g).abs().max().item() / max(g.abs().max().item(), 1e-3 * gmax)
            assert dev < 1e-2, (s, n, dev)
