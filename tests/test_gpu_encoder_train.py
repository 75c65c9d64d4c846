"""The train-mode encoder forward (csrc/encoder.cu, vrpx_encoder_forward with train = 1) against float64: stage by
stage, end to end, and through the BatchNorm running statistics it leaves behind.

Train mode is a code path of its own:
* the REINFORCE forward (save=True) runs the in-projection, the out-projection and the feed-forward as separate GEMMs
  and the attention on k_enc_attention_f16 (template buckets NJJ = 2 / 4 / 7 / 8, switching at N = 32 | 33, 64 | 65,
  112 | 113), and writes every stage into the saved block that encoder_bwd.cu reads;
* without save (`GraphEncoder(...)(x)` in train mode, an agent step under no_grad), gemm_path 0 runs the fused
  in-projection + attention kernel, applies BN1 in place over the layer input and takes Y2 from ff_fused;
* BatchNorm normalises with the batch statistics of all R = B*N rows (k_bn_stats: f64 column sums; k_bn_fold: biased
  variance) and moves running_mean / running_var of all six BatchNorms with momentum 0.1 and the unbiased variance.
gemm_path 1 runs the same steps on the fp32 SIMT GEMMs and the fp32 k_enc_attention.

The encoders are the production modules of TSPAgent / VRPAgent / IRPAgent(seed).  Seed initialisation leaves the
attention biases at 0, the BatchNorm affine at 1 / 0 and the running statistics at 0 / 1, where a dropped bias, affine
term or running-statistic term changes nothing, so _encoder perturbs those tensors (seeded).  Inputs are drawn as the
envs draw them: coordinates U[0,1), IRP demand (1 + 9u) / C with C = 0.2449 N + 26.12 and zero demand at the depot,
rounded to f32 as the encoder reads them.  The reference is float64 on the GPU with the encoder's f32 weights."""
import copy
import time

import pytest
import torch
import torch.nn.functional as Fn

pytestmark = pytest.mark.gpu

F64 = torch.float64
E = 128
# Bars, each 2-4 x the largest value measured over all cases and both gemm_paths on a B200 (1000 W power limit).
# Stage by stage: max |kernel - float64| over a (layer, stage) tensor relative to that tensor's largest element, every
# stage computed from the kernel's own saved input to it.
STAGE_TOL = {"H": 5e-7,     # embedding and layer outputs: measured 1.5e-7
             "QKV": 2e-6,   # measured 7.3e-7 (SIMT) / 5.0e-7 (tcgen05)
             "ATT": 4e-6,   # measured 1.3e-6 (k_enc_attention_f16, N = 113) / 8.2e-7 (fp32 k_enc_attention)
             "Y1": 1e-6,    # measured 3.0e-7
             "H1": 1e-6,    # measured 4.3e-7
             "F": 2e-6,     # measured 6.9e-7
             "Y2": 3e-6}    # measured 9.5e-7
# The saved BatchNorm (mean, invstd) are f32 roundings of f64 column sums of the saved Y1 / Y2, against the float64
# statistics of the same rows, relative to the vector's largest element: mean measured 5.1e-8, invstd 1.2e-7.
MEAN_TOL = 1.5e-7
INVSTD_TOL = 3e-7
# End to end, not teacher-forced: |got - ref| / max(1, |ref|) elementwise.  Measured 1.7e-5 (TSP-128 x 7, save=True,
# tcgen05) and 1.6e-5 (TSP-20 x 9477, SIMT); C4 7.4e-6.  Looser than the suite's 1e-5 for the eval-mode embeddings
# because the rounding of each stage, about 1e-6 of its scale, passes through six train-mode BatchNorms and three
# layers: a plain fp32 evaluation of the same encoder (the oracle in float32, which the test prints) sits at the same
# distance, 1.7e-5 at TSP-20 x 9477 and 1.0e-5 at C4.
E2E_TOL = 4e-5
# running_mean / running_var after three passes, relative to the buffer's largest element: measured 3.0e-7
RUN_TOL = 1e-6
# eval mode on those running statistics, as E2E_TOL: measured 3.0e-6
EVAL_TOL = 1e-5
ROWS = 1 << 18   # rows per float64 chunk of the reference (a 512-wide chunk is 1 GiB)

SAVED_STAGES = (("qkv", 384), ("att", 128), ("y1", 128), ("h1", 128), ("f", 512), ("y2", 128))


def saved_stages(saved, B, N):
    """Named views of the flat block vrpx_encoder_forward(save) writes (encoder.cu, kSaved*), for R = B*N rows:
    H[0..2] (R, 128), the inputs of the three layers; then per layer QKV (R, 384), ATT, Y1, H1 (R, 128), F (R, 512),
    Y2 (R, 128); then per layer the (mean, invstd) rows (2, 128) of BN1 and BN2.  Returns (H, layers), layers[l] a dict
    with keys qkv, att, y1, h1, f, y2, bn1, bn2."""
    R = B * N
    H = [saved[l * R * E:(l + 1) * R * E].view(R, E) for l in range(3)]
    layers = []
    o = 3 * R * E
    for l in range(3):
        blk = {}
        for name, width in SAVED_STAGES:
            blk[name] = saved[o:o + R * width].view(R, width)
            o += R * width
        layers.append(blk)
    for l in range(3):
        for name in ("bn1", "bn2"):
            layers[l][name] = saved[o:o + 2 * E].view(2, E)
            o += 2 * E
    assert o == saved.numel()
    return H, layers


def _encoder(kind, seed, gemm_path):
    """The seed-initialised encoder of the kind's agent in train mode, with the attention biases, the BatchNorm affine
    and the running statistics perturbed away from 0 / 1."""
    from agents import IRPAgent, TSPAgent, VRPAgent

    enc = {"tsp": TSPAgent, "vrp": VRPAgent, "irp": IRPAgent}[kind](seed=seed).model.encoder
    enc.gemm_path = gemm_path
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for layer in enc.attention_layers:
            a = layer.attention_layer
            a.in_proj_bias.copy_(0.1 * torch.randn(3 * E, generator=g))
            a.out_proj.bias.copy_(0.1 * torch.randn(E, generator=g))
            for bn in (layer.bn1.norm, layer.bn2.norm):
                bn.weight.copy_(1 + 0.2 * torch.randn(E, generator=g))
                bn.bias.copy_(0.2 * torch.randn(E, generator=g))
                bn.running_mean.copy_(0.2 * torch.randn(E, generator=g))
                bn.running_var.copy_(0.5 + torch.rand(E, generator=g))
    return enc.train()


def _inputs(kind, B, N, seed):
    """x (B, N, f) f32, depot (B,) int32 or None, depot one-hot (B, N) bool or None, on the GPU."""
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(seed)
    xy = torch.rand(B, N, 2, generator=g, dtype=F64, device=dev)
    if kind == "tsp":
        return xy.float().contiguous(), None, None
    depot = torch.randint(N, (B,), generator=g, device=dev)
    ar = torch.arange(B, device=dev)
    feats = [xy]
    if kind == "irp":
        d = (1 + 9 * torch.rand(B, N, generator=g, dtype=F64, device=dev)) / (0.2449 * N + 26.12)
        d[ar, depot] = 0
        feats.append(d[:, :, None])
    doh = torch.zeros(B, N, dtype=torch.bool, device=dev)
    doh[ar, depot] = True
    return torch.cat(feats, -1).float().contiguous(), depot.to(torch.int32), doh


def _sd(enc, dtype=F64):
    return {"encoder." + k: v.detach().to(dtype) for k, v in enc.state_dict().items()}


def _chunks(n, step):
    return [slice(i, min(n, i + step)) for i in range(0, n, step)]


def _attention64(qkv):
    """(b, N, 384) rows [q | k | v] -> (b, N, 128): 8 heads of 16, softmax(q k^T / 4) v."""
    b, N = qkv.shape[:2]
    q, k, v = (qkv.view(b, N, 3, 8, 16)[:, :, i].transpose(1, 2) for i in range(3))
    return (torch.softmax(q @ k.transpose(-1, -2) / 4.0, dim=-1) @ v).transpose(1, 2).reshape(b, N, E)


def _column_stats(y):
    """float64 mean and 1 / sqrt(biased variance + 1e-5) over the rows of y (R, 128), two passes in row chunks."""
    R = y.shape[0]
    mean = sum(y[sl].to(F64).sum(0) for sl in _chunks(R, ROWS)) / R
    var = sum(((y[sl].to(F64) - mean) ** 2).sum(0) for sl in _chunks(R, ROWS)) / R
    return mean, 1.0 / torch.sqrt(var + 1e-5)


def _encoder_ref(enc, x, doh, train, dtype=F64):
    """The oracle encoder (oracle/policy_oracle.py) on the encoder's f32 weights, evaluated in `dtype`."""
    from oracle import policy_oracle as po

    return po.encoder_forward(_sd(enc, dtype), x.to(dtype), doh, train=train, chunk=max(1, ROWS // x.shape[1]))


def _rel(got, ref):
    return ((got.to(F64) - ref).abs() / ref.abs().clamp_min(1.0)).max().item()


def _stage_errors(enc, x, doh, saved, h):
    """max |kernel - float64| / max |float64| of every (layer, stage) of the saved block and of the returned h, each
    stage computed in float64 from the kernel's own saved input to it; the BatchNorm statistics from the kernel's saved
    Y1 / Y2.  Returns {(layer, stage): error}."""
    B, N, f = x.shape
    R = B * N
    sd = _sd(enc)
    H, layers = saved_stages(saved, B, N)
    x64 = x.reshape(R, f).to(F64)
    acc = {}

    def put(key, got, ref):
        e, s = acc.get(key, (0.0, 0.0))
        acc[key] = (max(e, (got.to(F64) - ref).abs().max().item()), max(s, ref.abs().max().item()))

    def rows(key, got, fn):
        for sl in _chunks(R, ROWS):
            put(key, got[sl], fn(sl))

    def embed(sl):
        ref = x64[sl] @ sd["encoder.node_embed.weight"].T + sd["encoder.node_embed.bias"]
        if doh is None:
            return ref
        dep = x64[sl, :2] @ sd["encoder.depot_embed.weight"].T + sd["encoder.depot_embed.bias"]
        return torch.where(doh.reshape(R)[sl, None], dep, ref)

    rows((0, "H"), H[0], embed)
    for l in range(3):
        p = f"encoder.attention_layers.{l}."
        S = layers[l]
        hin = H[l]
        hout = H[l + 1] if l < 2 else h.reshape(R, E)
        rows((l, "QKV"), S["qkv"], lambda sl: hin[sl].to(F64) @ sd[p + "attention_layer.in_proj_weight"].T
             + sd[p + "attention_layer.in_proj_bias"])
        for ib in _chunks(B, max(1, ROWS // N)):
            r = slice(ib.start * N, ib.stop * N)
            put((l, "ATT"), S["att"][r], _attention64(S["qkv"][r].to(F64).view(-1, N, 3 * E)).reshape(-1, E))
        rows((l, "Y1"), S["y1"], lambda sl: hin[sl].to(F64)
             + S["att"][sl].to(F64) @ sd[p + "attention_layer.out_proj.weight"].T
             + sd[p + "attention_layer.out_proj.bias"])
        m1, is1 = _column_stats(S["y1"])
        put((l, "mean1"), S["bn1"][0], m1)
        put((l, "invstd1"), S["bn1"][1], is1)
        w1, b1 = sd[p + "bn1.norm.weight"], sd[p + "bn1.norm.bias"]
        rows((l, "H1"), S["h1"], lambda sl: (S["y1"][sl].to(F64) - m1) * is1 * w1 + b1)
        rows((l, "F"), S["f"], lambda sl: torch.relu(S["h1"][sl].to(F64) @ sd[p + "ff.0.weight"].T
                                                     + sd[p + "ff.0.bias"]))
        rows((l, "Y2"), S["y2"], lambda sl: S["h1"][sl].to(F64) + S["f"][sl].to(F64) @ sd[p + "ff.2.weight"].T
             + sd[p + "ff.2.bias"])
        m2, is2 = _column_stats(S["y2"])
        put((l, "mean2"), S["bn2"][0], m2)
        put((l, "invstd2"), S["bn2"][1], is2)
        w2, b2 = sd[p + "bn2.norm.weight"], sd[p + "bn2.norm.bias"]
        rows((l + 1, "H"), hout, lambda sl: (S["y2"][sl].to(F64) - m2) * is2 * w2 + b2)
    return {k: e / s for k, (e, s) in acc.items()}


def _tol(stage):
    return MEAN_TOL if stage.startswith("mean") else INVSTD_TOL if stage.startswith("invstd") else STAGE_TOL[stage]


# (kind, N, B): R = 6 and 16, where R / (R - 1) is 20 % and 7 %; every bucket edge of k_enc_attention_f16 with odd
# instance counts; the training batch of test_gpu_backward_scale.py
CASES = [("tsp", 2, 3), ("tsp", 8, 2), ("tsp", 32, 7), ("vrp", 33, 5), ("irp", 64, 3), ("tsp", 65, 9), ("vrp", 112, 3),
         ("irp", 113, 5), ("tsp", 128, 7), ("vrp", 65, 11), ("tsp", 20, 9477)]
C4 = ("tsp", 50, 65536)   # the train step of bench.py: R = 3,276,800 rows, a 60 GB saved block
IDS = [f"{k}{n}_b{b}" for k, n, b in CASES]
PATH_CASES = [c + (p,) for c in CASES for p in (0, 1)] + [C4 + (0,)]
PATH_IDS = [f"{i}_path{p}" for i in IDS for p in (0, 1)] + ["c4_tsp50_b65536_path0"]


def _seed(N, B):
    return 7 * N + B


@pytest.mark.parametrize("kind,N,B,gemm_path", PATH_CASES, ids=PATH_IDS)
def test_train_forward_stages_vs_float64(kind, N, B, gemm_path):
    """The REINFORCE forward (save=True): H[0] from x, then per layer QKV, ATT, Y1, the saved BN1 (mean, invstd), H1, F,
    Y2, the saved BN2 (mean, invstd) and the layer output (H[l+1], and h after the last layer), each in float64 from the
    kernel's own saved input to that stage, so that errors do not compound."""
    t0 = time.time()
    torch.cuda.reset_peak_memory_stats()
    from agents.graph_encoder import run_encoder

    enc = _encoder(kind, _seed(N, B), gemm_path)
    x, depot, doh = _inputs(kind, B, N, _seed(N, B))
    h, saved = run_encoder(enc, x=x, depot=depot, gemm_path=gemm_path, save=True)
    errs = _stage_errors(enc, x, doh, saved, h)
    worst = {}
    for (l, stage), e in errs.items():
        worst[stage] = max(worst.get(stage, (0.0, l)), (e, l))
    print(f"\n[{kind}{N} B={B} path={gemm_path}] " + " ".join(f"{s} {e:.2g}@{l}" for s, (e, l) in worst.items())
          + f"  ({time.time() - t0:.1f} s, peak {torch.cuda.max_memory_allocated() / 2 ** 30:.1f} GiB)")
    bad = [(l, s, e) for (l, s), e in errs.items() if e > _tol(s)]
    assert not bad, bad


@pytest.mark.parametrize("kind,N,B,gemm_path", PATH_CASES, ids=PATH_IDS)
def test_train_forward_end_to_end_vs_float64(kind, N, B, gemm_path):
    """The returned h of the train-mode forward with save=True (run_encoder) and without (the public entry
    `encoder(x[, depot_mask])`) against the float64 encoder with batch statistics, not teacher-forced."""
    t0 = time.time()
    torch.cuda.reset_peak_memory_stats()
    from agents.graph_encoder import run_encoder

    enc = _encoder(kind, _seed(N, B), gemm_path)
    x, depot, doh = _inputs(kind, B, N, _seed(N, B))
    with torch.no_grad():
        h_plain = enc(x) if doh is None else enc(x, doh)
    h_save, saved = run_encoder(enc, x=x, depot=depot, gemm_path=gemm_path, save=True)
    del saved
    torch.cuda.empty_cache()
    ref = _encoder_ref(enc, x, doh, train=True)
    e_save, e_plain = _rel(h_save, ref), _rel(h_plain, ref)
    e_f32 = _rel(_encoder_ref(enc, x, doh, train=True, dtype=torch.float32), ref)
    print(f"\n[{kind}{N} B={B} path={gemm_path}] end to end: save {e_save:.3g}, no save {e_plain:.3g}, "
          f"fp32 oracle {e_f32:.3g}  "
          f"({time.time() - t0:.1f} s, peak {torch.cuda.max_memory_allocated() / 2 ** 30:.1f} GiB)")
    assert e_save <= E2E_TOL and e_plain <= E2E_TOL, (e_save, e_plain)


@pytest.mark.parametrize("gemm_path", [0, 1])
@pytest.mark.parametrize("kind,N,B", CASES, ids=IDS)
def test_running_statistics_vs_float64(kind, N, B, gemm_path):
    """Three train-mode passes on three batches (save=True, the public entry without save, save=True), then
    running_mean / running_var of all six BatchNorms against torch's own rule (F.batch_norm, training=True,
    momentum 0.1, eps 1e-5) on float64 buffers fed each pass's Y1 / Y2, and num_batches_tracked == 3.  The pass without
    save keeps no activations: its Y1 / Y2 come from a save=True run of a copy of the encoder on the same batch.  Then
    eval mode on those running statistics against the float64 eval-mode encoder, the baseline and evaluation path after
    an epoch."""
    from agents.graph_encoder import run_encoder

    enc = _encoder(kind, _seed(N, B), gemm_path)
    bns = {(l, j): bn for l, layer in enumerate(enc.attention_layers)
           for j, bn in enumerate((layer.bn1.norm, layer.bn2.norm))}
    ref = {k: (bn.running_mean.to(F64).clone(), bn.running_var.to(F64).clone()) for k, bn in bns.items()}
    assert all(int(bn.num_batches_tracked) == 0 for bn in bns.values())
    for i, save in enumerate((True, False, True)):
        x, depot, doh = _inputs(kind, B, N, _seed(N, B) + 1000 * (i + 1))
        if save:
            _, saved = run_encoder(enc, x=x, depot=depot, gemm_path=gemm_path, save=True)
        else:
            _, saved = run_encoder(copy.deepcopy(enc), x=x, depot=depot, gemm_path=gemm_path, save=True)
            with torch.no_grad():
                enc(x) if doh is None else enc(x, doh)
        _, layers = saved_stages(saved, B, N)
        for (l, j), (rm, rv) in ref.items():
            Fn.batch_norm(layers[l]["y2" if j else "y1"].to(F64), rm, rv, training=True, momentum=0.1, eps=1e-5)
        del saved, layers
    worst, bad = (0.0, None), []
    for (l, j), bn in bns.items():
        assert int(bn.num_batches_tracked) == 3, (l, j)
        for name, got, r in (("mean", bn.running_mean, ref[l, j][0]), ("var", bn.running_var, ref[l, j][1])):
            e = (got.to(F64) - r).abs().max().item() / r.abs().max().item()
            worst = max(worst, (e, (l, f"bn{j + 1}", name)), key=lambda w: w[0])
            if e > RUN_TOL:
                bad.append((l, f"bn{j + 1}", name, e))
    enc.eval()
    x, depot, doh = _inputs(kind, B, N, _seed(N, B) + 4000)
    with torch.no_grad():
        h = enc(x) if doh is None else enc(x, doh)
    e_eval = _rel(h, _encoder_ref(enc, x, doh, train=False))
    print(f"\n[{kind}{N} B={B} path={gemm_path}] running stats {worst[0]:.3g} {worst[1]}, eval on them {e_eval:.3g}")
    assert not bad, bad
    assert e_eval <= EVAL_TOL, e_eval
