"""GPU parity of the GEMM paths behind the encoder (csrc/gemm_tc4.cu tcgen05 f16-split = production, csrc/encoder.cu
SIMT cross-check)
against a float64 torch matmul, through the C ABI test hook vrpx_debug_gemm."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _run(path, R, K, NOUT, bias, relu, residual, bn, seed=0):
    import vrpx

    dev = vrpx.require_device()
    g = torch.Generator(device="cpu").manual_seed(seed)
    X = torch.randn(R, K, generator=g).to(dev)
    W = (torch.randn(NOUT, K, generator=g) / K ** 0.5).to(dev)
    b = torch.randn(NOUT, generator=g).to(dev) if bias else None
    res = torch.randn(R, NOUT, generator=g).to(dev) if residual else None
    sc = (torch.rand(NOUT, generator=g) + 0.5).to(dev) if bn else None
    sh = torch.randn(NOUT, generator=g).to(dev) if bn else None
    Y = torch.empty(R, NOUT, device=dev)
    vrpx.check(vrpx.lib().vrpx_debug_gemm(vrpx.ptr(X), R, K, vrpx.ptr(W), NOUT, vrpx.ptr(b), int(relu), vrpx.ptr(res),
                                          vrpx.ptr(sc), vrpx.ptr(sh), vrpx.ptr(Y), path, vrpx.stream_ptr(dev)))
    torch.cuda.synchronize()
    ref = X.double() @ W.double().T
    if bias:
        ref = ref + b.double()
    if relu:
        ref = ref.clamp_min(0)
    if residual:
        ref = ref + res.double()
    if bn:
        ref = ref * sc.double() + sh.double()
    return Y.double(), ref


SHAPES = [(128, 128, 128), (1000, 128, 384), (777, 128, 512), (1300, 512, 128), (5, 128, 128), (40000, 384, 128),
          (70000, 128, 384)]


@pytest.mark.parametrize("path", [1, 0], ids=["simt", "tcgen05_f16split"])
@pytest.mark.parametrize("R,K,NOUT", SHAPES)
def test_gemm_plain(path, R, K, NOUT):
    Y, ref = _run(path, R, K, NOUT, False, False, False, False)
    err = (Y - ref).abs().max().item()
    scale = ref.abs().max().item()
    # fp32-level accuracy is required of ALL paths.  SIMT: a few fp32 ulps.  The tensor paths split every operand into two
    # halves exact to 2^-21 per product (f16 hi/lo), but the tensor core accumulates the partial products into
    # TMEM with truncation: ~2e-6 of the output scale at K=512 -> bound 1e-5 * scale * sqrt(K/128).
    tol = (2e-6 if path == 1 else 1e-5) * max(scale, 1.0) * (K / 128) ** 0.5 + 1e-6
    assert err <= tol, (path, R, K, NOUT, err, scale)


@pytest.mark.parametrize("path", [1, 0], ids=["simt", "tcgen05_f16split"])
def test_gemm_epilogues(path):
    for (bias, relu, residual, bn) in [(True, False, False, False), (True, True, False, False),
                                       (True, False, True, True), (False, False, True, False)]:
        Y, ref = _run(path, 515, 128, 128, bias, relu, residual, bn, seed=3)
        err = (Y - ref).abs().max().item()
        assert err <= (1e-5 if path == 1 else 4e-5), (path, bias, relu, residual, bn, err)


def test_gemm_tc_in_place_residual():
    """The encoder runs out-proj / FF2 with Y aliasing the residual (h <- BN(h + X W^T))."""
    import vrpx

    dev = vrpx.require_device()
    R, K, NOUT = 900, 512, 128
    X = torch.randn(R, K, device=dev)
    W = torch.randn(NOUT, K, device=dev) / K ** 0.5
    h = torch.randn(R, NOUT, device=dev)
    ref = h.double() + X.double() @ W.double().T
    vrpx.check(vrpx.lib().vrpx_debug_gemm(vrpx.ptr(X), R, K, vrpx.ptr(W), NOUT, None, 0, vrpx.ptr(h), None, None,
                                          vrpx.ptr(h), 0, vrpx.stream_ptr(dev)))
    torch.cuda.synchronize()
    assert (h.double() - ref).abs().max().item() <= 6e-5


@pytest.mark.parametrize("R,M,N", [(5000, 128, 512), (33000, 384, 128), (777, 512, 128), (4097, 128, 1024), (1000, 128, 4)])
def test_gemm_tn_accumulate(R, M, N):
    """Weight-gradient reduction C[M][N] += A^T · B (tensor-pipe kernel for 64-multiples, SIMT otherwise)."""
    import vrpx

    dev = vrpx.require_device()
    g = torch.Generator(device="cpu").manual_seed(1)
    A = torch.randn(R, M, generator=g).to(dev)
    Bm = torch.randn(R, N, generator=g).to(dev)
    C0 = torch.randn(M, N, generator=g).to(dev)
    C = C0.clone()
    vrpx.check(vrpx.lib().vrpx_gemm_tn_accumulate(vrpx.ptr(A), vrpx.ptr(Bm), vrpx.ptr(C), R, M, N, vrpx.stream_ptr(dev)))
    torch.cuda.synchronize()
    ref = C0.double() + A.double().T @ Bm.double()
    err = (C.double() - ref).abs().max().item()
    assert err <= 2e-5 * ref.abs().max().item() + 1e-5, (R, M, N, err)


@pytest.mark.parametrize("R", [128, 1000, 5, 19000, 148 * 128 * 2 + 77])
@pytest.mark.parametrize("affine", [True, False], ids=["bn_affine", "plain"])
def test_ff_fused_kernel(R, affine):
    """csrc/ff_fused.cu: Y = (residual + relu(X W1^T + b1) W2^T + b2) * scale + shift in one tcgen05 kernel (the hidden
    activation stays in tensor memory) against float64; in place (Y aliases X and the residual) like the encoder calls it."""
    import vrpx

    dev = vrpx.require_device()
    g = torch.Generator(device="cpu").manual_seed(R)
    X = torch.randn(R, 128, generator=g).to(dev)
    W1 = (torch.randn(512, 128, generator=g) / 128 ** 0.5).to(dev)
    b1 = (torch.randn(512, generator=g) * 0.1).to(dev)
    W2 = (torch.randn(128, 512, generator=g) / 512 ** 0.5).to(dev)
    b2 = (torch.randn(128, generator=g) * 0.1).to(dev)
    sc = (torch.rand(128, generator=g) + 0.5).to(dev) if affine else None
    sh = torch.randn(128, generator=g).to(dev) if affine else None
    ref = X.double() + torch.relu(X.double() @ W1.double().T + b1.double()) @ W2.double().T + b2.double()
    if affine:
        ref = ref * sc.double() + sh.double()
    Y = X.clone()
    vrpx.check(vrpx.lib().vrpx_debug_ff_fused(vrpx.ptr(Y), R, vrpx.ptr(W1), vrpx.ptr(b1), vrpx.ptr(W2), vrpx.ptr(b2), vrpx.ptr(Y),
                                              vrpx.ptr(sc) if affine else None, vrpx.ptr(sh) if affine else None, vrpx.ptr(Y),
                                              vrpx.stream_ptr(dev)))
    torch.cuda.synchronize()
    err = (Y.double() - ref).abs().max().item()
    assert err <= 1e-5 * max(ref.abs().max().item(), 1.0), (R, affine, err)
    # out of place, a second call on the same stream (scratch reuse)
    Y2 = torch.empty_like(X)
    vrpx.check(vrpx.lib().vrpx_debug_ff_fused(vrpx.ptr(X), R, vrpx.ptr(W1), vrpx.ptr(b1), vrpx.ptr(W2), vrpx.ptr(b2), vrpx.ptr(X),
                                              vrpx.ptr(sc) if affine else None, vrpx.ptr(sh) if affine else None, vrpx.ptr(Y2),
                                              vrpx.stream_ptr(dev)))
    torch.cuda.synchronize()
    assert torch.equal(Y, Y2)


@pytest.mark.parametrize("B,N", [(1, 50), (7, 50), (300, 50), (5, 20), (33, 21), (9, 10), (4, 100), (3, 101), (2, 128), (3, 2),
                                 (148 * 2 * 3 + 5, 50), (11, 64), (6, 65), (5, 7)])
def test_qkv_attention_fused_kernel(B, N):
    """csrc/attn_fused.cu: the in-projection and the 8-head self-attention of an encoder layer in one kernel (Q, K, V stay
    in shared memory) against float64 (graph_encoder.py:74-104 = nn.MultiheadAttention without its out-projection);
    whole-instance tiles for every N bucket, ragged last tiles, odd N."""
    import vrpx

    dev = vrpx.require_device()
    g = torch.Generator(device="cpu").manual_seed(B * 1000 + N)
    X = torch.randn(B * N, 128, generator=g).to(dev)
    W = (torch.randn(384, 128, generator=g) / 128 ** 0.5).to(dev)
    b = (torch.randn(384, generator=g) * 0.1).to(dev)
    qkv = (X.double() @ W.double().T + b.double()).view(B, N, 3, 8, 16)
    q, k, v = (qkv[:, :, i].permute(0, 2, 1, 3) for i in range(3))     # [B][8][N][16]
    p = torch.softmax(q @ k.transpose(-1, -2) / 4.0, dim=-1)
    ref = (p @ v).permute(0, 2, 1, 3).reshape(B * N, 128)
    att = torch.full((B * N, 128), float("nan"), device=dev)
    vrpx.check(vrpx.lib().vrpx_debug_qkv_attention(vrpx.ptr(X), vrpx.ptr(W), vrpx.ptr(b), B, N, vrpx.ptr(att), vrpx.stream_ptr(dev)))
    torch.cuda.synchronize()
    err = (att.double() - ref).abs().max().item()
    assert err <= 1e-5 * max(ref.abs().max().item(), 1.0), (B, N, err)
    att2 = torch.empty_like(att)
    vrpx.check(vrpx.lib().vrpx_debug_qkv_attention(vrpx.ptr(X), vrpx.ptr(W), vrpx.ptr(b), B, N, vrpx.ptr(att2), vrpx.stream_ptr(dev)))
    torch.cuda.synchronize()
    assert torch.equal(att, att2)


@pytest.mark.parametrize("R,M,N,ascale", [(8192, 128, 128, 1.0), (65536 + 37, 128, 512, 1e-5), (100003, 512, 128, 1e-3),
                                          (50000, 384, 128, 1e-6), (65536, 1024, 128, 1e-2), (9000, 256, 256, 30.0)])
def test_gemm_tn_tcgen05(R, M, N, ascale):
    """csrc/gemm_tn_tc.cu: the weight-gradient GEMM on tcgen05 (operands transposed and f16-split on the way into shared
    memory, split-K with register drains) against float64 — O(1) to O(100) operands at 2e-5 of the result scale,
    gradient-sized ones (below 1e-3 the f16 lo half of the 2^8-scaled operand is a subnormal: about 13 bits at 1e-6) at
    2e-4, ragged row counts, and against the warp-level kernel it replaces."""
    import vrpx

    dev = vrpx.require_device()
    L = vrpx.lib()
    g = torch.Generator(device="cpu").manual_seed(R + M)
    A = (torch.randn(R, M, generator=g) * ascale).to(dev)
    Bm = torch.randn(R, N, generator=g).abs().to(dev)          # activations after a ReLU: the sums do not cancel
    C = torch.zeros(M, N, device=dev)
    vrpx.check(L.vrpx_gemm_tn_accumulate(vrpx.ptr(A), vrpx.ptr(Bm), vrpx.ptr(C), R, M, N, vrpx.stream_ptr(dev)))
    torch.cuda.synchronize()
    ref = A.double().T @ Bm.double()
    scale = ref.abs().max().item()
    err = (C.double() - ref).abs().max().item()
    tol = 2e-5 if ascale >= 1e-3 else 2e-4
    assert err <= tol * scale, (R, M, N, err / scale)
    L.vrpx_debug_gemm_tn_path(1)
    try:
        C1 = torch.zeros(M, N, device=dev)
        vrpx.check(L.vrpx_gemm_tn_accumulate(vrpx.ptr(A), vrpx.ptr(Bm), vrpx.ptr(C1), R, M, N, vrpx.stream_ptr(dev)))
        torch.cuda.synchronize()
    finally:
        L.vrpx_debug_gemm_tn_path(0)
    assert (C1.double() - ref).abs().max().item() <= 2e-5 * scale
    # bias gradient riding on the weight gradient: column sums of A, on both paths
    csum_ref = A.double().sum(0)
    cscale = max(csum_ref.abs().max().item(), A.double().abs().sum(0).max().item() * 1e-3)
    for path in (0, 1):
        L.vrpx_debug_gemm_tn_path(path)
        try:
            C3, cs = torch.zeros(M, N, device=dev), torch.zeros(M, device=dev)
            vrpx.check(L.vrpx_gemm_tn_colsum_accumulate(vrpx.ptr(A), vrpx.ptr(Bm), vrpx.ptr(C3), vrpx.ptr(cs), R, M, N,
                                                        vrpx.stream_ptr(dev)))
            torch.cuda.synchronize()
        finally:
            L.vrpx_debug_gemm_tn_path(0)
        assert (C3.double() - ref).abs().max().item() <= tol * scale
        assert (cs.double() - csum_ref).abs().max().item() <= 2e-5 * cscale, (path, R, M)
    # accumulation into a non-zero C
    C2 = C.clone()
    vrpx.check(L.vrpx_gemm_tn_accumulate(vrpx.ptr(A), vrpx.ptr(Bm), vrpx.ptr(C2), R, M, N, vrpx.stream_ptr(dev)))
    torch.cuda.synchronize()
    assert (C2.double() - 2 * ref).abs().max().item() <= 2 * tol * scale


@pytest.mark.parametrize("B,N", [(3, 50), (40, 50), (5, 20), (7, 21), (4, 10), (3, 100), (2, 101), (2, 128), (3, 7), (600, 50)])
def test_attention_backward_mma(B, N):
    """csrc/attention_bwd.cu: backward of the 8-head attention core on mma.sync (f16 hi/lo halves, both score
    orientations) against torch autograd in float64, and against the fp32 SIMT kernel it replaces."""
    import vrpx

    dev = vrpx.require_device()
    L = vrpx.lib()
    g = torch.Generator(device="cpu").manual_seed(B * 1000 + N)
    qkv = torch.randn(B * N, 384, generator=g).to(dev)
    datt = (torch.randn(B * N, 128, generator=g) * 1e-3).to(dev)
    x = qkv.double().requires_grad_(True)
    q, k, v = (x.view(B, N, 3, 8, 16)[:, :, i].permute(0, 2, 1, 3) for i in range(3))     # [B][8][N][16]
    att64 = (torch.softmax(q @ k.transpose(-1, -2) / 4.0, dim=-1) @ v).permute(0, 2, 1, 3).reshape(B * N, 128)
    (ref,) = torch.autograd.grad(att64, x, datt.double())
    att = att64.detach().float().contiguous()
    scale = ref.abs().max().item()
    outs = []
    for path in (0, 1):
        dqkv = torch.full((B * N, 384), float("nan"), device=dev)
        vrpx.check(L.vrpx_debug_attention_backward(vrpx.ptr(qkv), vrpx.ptr(att), vrpx.ptr(datt), vrpx.ptr(dqkv), B, N, path,
                                                   vrpx.stream_ptr(dev)))
        torch.cuda.synchronize()
        err = (dqkv.double() - ref).abs().max().item()
        assert err <= 2e-5 * scale, (B, N, path, err / scale)
        outs.append(dqkv)
    # each third on its own: dQ, dK, dV
    for c0 in (0, 128, 256):
        r = ref[:, c0:c0 + 128]
        assert (outs[0][:, c0:c0 + 128].double() - r).abs().max().item() <= 2e-5 * r.abs().max().item(), c0


def _score_table_tile(N):
    """Instances per tile of csrc/score_table_fused.cu (build_score_table_fused): whole instances in 128 rows, capped so
    that the k' fragments of a tile fit its KMAX = 200 keys."""
    nt = (N + 7) // 8
    bucket = 3 if nt <= 3 else (7 if nt <= 7 else (13 if nt <= 13 else 16))
    return min(128 // N, 1 + (200 - 8 * bucket) // (8 * nt))


# every N: B leaves a ragged last tile of 1 .. TI - 1 instances (TI = 1 above N = 64); then more than 37 tiles, so that
# each of the 37 streams of head-pair CTAs walks several tiles, in the three upper template buckets
SCORE_TABLE_CASES = [(N, 2 * _score_table_tile(N) + (1 + N % (_score_table_tile(N) - 1) if _score_table_tile(N) > 1 else 1))
                     for N in range(2, 129)] + [(20, 2003), (50, 2001), (105, 1999), (128, 2000)]
# largest error / largest |S1| of its (instance, head) block: measured 2.2e-6 on a B200 (1000 W power limit)
SCORE_TABLE_TOL = 1e-5


def test_score_table_fused_kernel():
    """csrc/score_table_fused.cu: S1[b][l][head][n] = q'[b,l,head] · k'[b,n,head] with q' = h (W_l / sqrt(48))^T and
    k' = h W_k^T (the rank-48 factors of the decoder's step query, vrpx/packing.py qk_w) against float64, for every
    N = 2 .. 128 (template buckets NT8 = 3 / 7 / 13 / 16, tiles of TI = 1 .. 23 instances, the float2 store of even N and
    the scalar store of odd N) and multi-tile streams.  S1 and a guard tail behind it start as NaN: every element of
    [B][N][8][N] is written and nothing beyond it."""
    import vrpx
    from agents import TSPAgent
    from vrpx import packing

    dev = vrpx.require_device()
    L = vrpx.lib()
    qk_w = packing.fold_decoder(TSPAgent(seed=5).model.decoder, False)["qk_w"].to(dev, torch.float32).contiguous()
    wq = qk_w[:384].double().view(8, 48, 128)
    wk = qk_w[384:].double().view(8, 48, 128)
    g = torch.Generator(device=dev).manual_seed(17)
    guard = 4096
    worst = (0.0, None)
    for N, B in SCORE_TABLE_CASES:
        h = torch.randn(B, N, 128, generator=g, device=dev)     # BatchNorm output scale
        n1 = B * N * 8 * N
        s1 = torch.full((n1 + guard,), float("nan"), device=dev)
        vrpx.check(L.vrpx_debug_score_table(vrpx.ptr(h), vrpx.ptr(qk_w), B, N, vrpx.ptr(s1), vrpx.stream_ptr(dev)))
        torch.cuda.synchronize()
        assert bool(torch.isnan(s1[n1:]).all()), (N, B, "wrote beyond S1")
        got = s1[:n1].view(B, N, 8, N)
        assert not bool(torch.isnan(got).any()), (N, B, "S1 element not written")
        hd = h.double()
        q = torch.einsum("bld,hjd->bhlj", hd, wq)
        k = torch.einsum("bnd,hjd->bhnj", hd, wk)
        ref = torch.einsum("bhlj,bhnj->blhn", q, k)
        err = (got.double() - ref).abs().amax(dim=(1, 3))        # (B, 8) per (instance, head) block
        scale = ref.abs().amax(dim=(1, 3))
        r = (err / scale).max().item()
        worst = max(worst, (r, (N, B)), key=lambda w: w[0])
        assert r <= SCORE_TABLE_TOL, (N, B, r)
    print(f"\n[score table] max error / block max {worst[0]:.3g} at (N, B) = {worst[1]}")
