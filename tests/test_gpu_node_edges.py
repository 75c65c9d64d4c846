"""The decode loop, the score tables and the Philox sampler against float64 at the node counts where the kernels change
shape, up to N = 128.

The decode kernels branch on N in several places, and the golden fixtures cover N = 4 .. 100 only:
* softmax, P store and value contraction (glimpse_mma.cuh): node = lane + 32 i over four strides, boundaries at
  N = 32 / 33, 64 / 65, 96 / 97, the last stride full at N = 128;
* the pointer phase (rollout.cuh, rollout_steps.cu k_step_pointer): node = 4 lane + i, the candidate list built from four
  mask words with `(1u << rem) - 1` word ranges and prefix counts, the same ranges in `instance_idle`;
* k_step_glimpse: 8-row cp.async slices, the last one partly zeroed when N % 8 != 0, fewer slices than ring stages at
  N <= 8; glimpse CTAs of 10 warps and pointer CTAs of 8, so B mod 10 and B mod 8 leave ragged CTAs;
* the score-table kernel's template buckets (switching at N = 24 / 25, 56 / 57, 104 / 105), odd and even N;
* the glimpse coupling (8b + h) mod G at B = 1 and small odd B, where the partner index wraps several times.

Every case runs in both whole-episode decode loops: table mode (the default: score tables + split-step launches, used
whenever the episode has at least 3 steps) and the classic loop of the persistent kernel.  The reference is the pinned
oracle (oracle/policy_oracle.py) in float64 on the GPU with the model's f32 weights, teacher-forced along the kernel's
own tape from the kernel's own embeddings (promoted to float64), so the logit bar measures the decoder alone; the
embeddings are checked on their own against the float64 encoder.  Masks and loads come from the env oracle stepped along
the tape at the full batch, and each attention row reads the mask of its partner instance (8b + h) mod G.

The sampler test draws one step of 8,192 identical instances through the single-step entry (coupling = B, so every row
has the same logits) with masks that open and close nodes at word and lane edges, and compares the histogram of the
sampled node with the float64 softmax by chi-squared.  A biased sampler would still pass every teacher-forced log-prob
test: the log-prob it reports is the exact one of the node it took."""
import numpy as np
import pytest
import torch
from oracle_replay import check_logp, host_inputs, partners

pytestmark = pytest.mark.gpu

F64 = torch.float64
# Bars: the suite's 1e-5, which is 2.4 x / 4.3 x the largest value measured on a B200 (1000 W power limit)
LOGIT_TOL = 1e-5   # |got - ref64| / max(1, |ref64|), masked pointer logits: measured 4.2e-6 (IRP-127, table mode)
EMB_TOL = 1e-5     # the same for the embeddings: measured 2.3e-6
TIE = 2e-5         # greedy actions are the float64 argmax up to near-ties

# (kind, N, B, coupling group G (None: the whole batch), greedy)
CASES = [("tsp", 3, 1, None, True), ("tsp", 9, 7, None, False), ("tsp", 32, 9, None, True), ("tsp", 33, 37, None, False),
         ("tsp", 64, 11, None, True), ("tsp", 65, 20, 5, False), ("tsp", 96, 7, None, True), ("tsp", 97, 10, None, True),
         ("tsp", 128, 21, None, True), ("tsp", 128, 21, None, False),
         ("vrp", 2, 3, None, True), ("vrp", 25, 16, None, True), ("vrp", 57, 13, None, False), ("vrp", 105, 9, None, True),
         ("vrp", 128, 5, None, False),
         ("irp", 24, 8, None, True), ("irp", 56, 12, None, False), ("irp", 104, 6, None, True), ("irp", 127, 4, None, False)]


def _cls(kind):
    from agents import IRPAgent, TSPAgent, VRPAgent
    from gym_vrp.envs import IRPEnv, TSPEnv, VRPEnv

    return {"tsp": (TSPEnv, TSPAgent), "vrp": (VRPEnv, VRPAgent), "irp": (IRPEnv, IRPAgent)}[kind]


def _rel(got, ref):
    return ((got.to(F64) - ref).abs() / ref.abs().clamp_min(1.0)).max().item()


def _reference_logits(sd, h, tape, masks, loads, part):
    """(T, B, N) float64 masked pointer logits teacher-forced along tape (T, B) long; masks (T, B, N) uint8, loads (T, B)
    or None, part (B, 8) long partner instances, all on h's device."""
    from oracle import policy_oracle as po

    B, N, E = h.shape
    first = sd["decoder._first_node"].reshape(1, E).repeat(B, 1)
    last = sd["decoder._last_node"].reshape(1, E).repeat(B, 1)
    ar = torch.arange(B, device=h.device)
    out = torch.empty((tape.shape[0], B, N), dtype=F64, device=h.device)
    for t in range(tape.shape[0]):
        mt = masks[t]
        out[t] = po.decoder_logits(sd, h, mt.to(F64), first, last, None if loads is None else loads[t].to(F64),
                                   glimpse_mask=mt[part].to(F64))
        last = h[ar, tape[t]]
        if t == 0:
            first = last
    return out


def _tour_length_f32(xy, depot, tape):
    """The tour length of every instance accumulated in f32 in step order, as the kernel accumulates its rewards."""
    B = xy.shape[0]
    ar = np.arange(B)
    cur = depot.copy()
    acc = np.zeros(B, dtype=np.float32)
    for t in range(tape.shape[0]):
        a = tape[t].astype(np.int64)
        d = xy[ar, cur] - xy[ar, a]
        acc = acc + np.sqrt(d[:, 0] ** 2 + d[:, 1] ** 2).astype(np.float32)
        cur = a
    return acc


@pytest.mark.parametrize("loop", ["tables", "classic"])
@pytest.mark.parametrize("kind,N,B,G,greedy", CASES,
                         ids=[f"{k}{n}_b{b}" + (f"_g{g}" if g else "") + ("_greedy" if gr else "_sampled")
                              for k, n, b, g, gr in CASES])
def test_decode_loop_vs_float64_at_node_edges(kind, N, B, G, greedy, loop):
    """Teacher-forced masked logits (finite pattern and values), greedy actions (float64 argmax up to near-ties), sampled
    log-prob sums, embeddings, costs (f32 tour length of the tape), and a second run without logits that must give the
    same tape, costs and log-probs bit for bit (it takes the idle-instance skip of the step kernels)."""
    from oracle import policy_oracle as po

    Env, Agent = _cls(kind)
    seed = 1000 + N
    model = Agent(seed=seed).model
    model.eval()
    model.coupling = G
    model.decoder.score_tables = loop == "tables"
    env = Env(N, B, 0, seed=seed, instance_rng="philox")
    runs = []
    for want_logits in (True, False):
        if runs:
            env.restart_episode()
        torch.manual_seed(seed)
        with torch.no_grad():
            model(env, rollout=greedy, want_logits=want_logits)
        runs.append(model.last_rollout)
    out, prod = runs
    T = out["steps"]
    tape = out["tape"]
    assert prod["steps"] == T
    assert torch.equal(prod["tape"], tape), "the run without logits took other actions"
    assert torch.equal(prod["cost"], out["cost"]) and torch.equal(prod["logp"], out["logp"])
    tape_np = tape.cpu().numpy()
    s = env.sampler
    xy, depot = s.get_graph_positions(), s.get_depots()[:, 0]
    assert np.allclose(out["cost"].cpu().numpy(), _tour_length_f32(xy, depot, tape_np), rtol=1e-6, atol=1e-6)

    dev = out["cost"].device
    sd = {k: v.detach().to(F64) for k, v in model.state_dict().items()}
    x, doh, masks, loads = host_inputs(kind, env, tape_np)
    h_ref = po.encoder_forward(sd, x.to(dev, F64), None if doh is None else doh.to(dev), False)
    emb_err = _rel(out["emb"], h_ref)
    assert emb_err <= EMB_TOL, ("embeddings", emb_err)
    masks = torch.from_numpy(masks).to(dev)
    loads = torch.from_numpy(loads).to(dev) if kind == "irp" else None
    a = tape.to(torch.long)
    ref = _reference_logits(sd, out["emb"].to(F64), a, masks, loads, partners(B, out["coupling"]).to(dev))
    got = out["logits"]
    fin = torch.isfinite(ref)
    assert torch.equal(fin, torch.isfinite(got)), "mask pattern differs"
    assert torch.equal(fin, masks == 0)
    err = _rel(got[fin], ref[fin])
    assert err <= LOGIT_TOL, ("logits", err)
    chosen = ref.gather(2, a[:, :, None])[:, :, 0]
    assert bool(torch.isfinite(chosen).all()), "a masked node was chosen"
    msg = f"\n[{kind}{N} B={B} G={G} {loop}] T={T} logits {err:.3g} emb {emb_err:.3g}"
    if greedy:
        assert bool((chosen >= ref.max(dim=2).values - TIE).all()), "a greedy action is not the float64 argmax"
    else:
        lp_ref = (chosen - torch.logsumexp(ref, dim=2)).sum(0)
        msg += f" logp {check_logp(lp_ref, out['logp'], T):.3g}"
    print(msg)


def _sampler_mask(N, which):
    """(N,) 1 = masked: holes at the word and lane edges 31 | 32, 63 | 64 and 96; two open nodes in different words (and
    lanes); only the last node open."""
    m = torch.zeros(N)
    if which == "holes":
        m[[n for n in (31, 32, 63, 64, 96) if n < N]] = 1
    else:
        m[:] = 1
        m[N - 1] = 0
        if which == "two_open":
            m[31] = 0
    return m


SAMPLER_B = 8192
SAMPLER_P = 1e-6   # chi-squared tail probability of the bar


@pytest.mark.parametrize("which", ["holes", "two_open", "last_only"])
@pytest.mark.parametrize("N", [33, 65, 128])
def test_sampler_distribution_at_word_edges(N, which):
    """Philox inverse-CDF sampling (warp_pointer_choice: lane totals scanned with __shfl_up, then node 4 lane + i) of one
    step of 8,192 identical instances through the single-step entry: no masked node is drawn, every returned log-prob is
    the float64 one of the drawn node, and the histogram matches softmax(float64 logits) at chi-squared tail P = 1e-6
    (the seed is fixed, so the outcome is deterministic)."""
    from scipy import stats

    from agents import GraphDecoder
    from oracle import policy_oracle as po

    torch.manual_seed(N)
    decoder = GraphDecoder(v_dim=128, k_dim=128).cuda()
    emb1 = torch.randn(1, N, 128, device="cuda")
    mask1 = _sampler_mask(N, which).cuda()
    torch.manual_seed(7)
    nxt, logp = decoder(emb1.expand(SAMPLER_B, N, 128).contiguous(), mask1.expand(SAMPLER_B, N).contiguous())
    nodes, logp = nxt[:, 0], logp[:, 0].to(F64)
    sd = {"decoder." + k: v.detach().to(F64) for k, v in decoder.state_dict().items()}
    first = sd["decoder._first_node"].reshape(1, 128)
    last = sd["decoder._last_node"].reshape(1, 128)
    m64 = mask1[None].to(F64)
    u = po.decoder_logits(sd, emb1.to(F64), m64, first, last, glimpse_mask=m64[:, None].expand(1, 8, N))[0]
    p = torch.softmax(u, 0)
    counts = torch.bincount(nodes, minlength=N).to(F64)
    assert counts.shape == (N,) and counts[mask1 > 0].sum().item() == 0, "a masked node was drawn"
    lp_ref = torch.log_softmax(u, 0)[nodes]
    assert bool(((logp - lp_ref).abs() <= 2e-5).all()), float((logp - lp_ref).abs().max())
    # bins below 5 expected draws pooled; a pool still below 5 joins the smallest bin
    expect = p * SAMPLER_B
    big = expect >= 5
    obs, exp = counts[big], expect[big]
    pool_obs, pool_exp = counts[~big].sum(), expect[~big].sum()
    if pool_exp >= 5:
        obs, exp = torch.cat([obs, pool_obs[None]]), torch.cat([exp, pool_exp[None]])
    elif pool_exp > 0:
        i = int(exp.argmin())
        obs[i] += pool_obs
        exp[i] += pool_exp
    dof = obs.numel() - 1
    if dof == 0:   # one open node (or all mass on one): no masked draw is the whole check
        return
    chi2 = (((obs - exp) ** 2) / exp).sum().item()
    bar = stats.chi2.isf(SAMPLER_P, dof)
    print(f"\n[sampler N={N} {which}] chi2 {chi2:.1f} on {dof} dof, bar {bar:.1f}")
    assert chi2 <= bar, (chi2, dof, bar)
