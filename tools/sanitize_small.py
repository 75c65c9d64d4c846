#!/usr/bin/env python
"""Small-shape driver for compute-sanitizer (memcheck / racecheck / synccheck): every kernel family once —
env API kernels, tcgen05 GEMM (both accumulator modes), encoder forward (eval + train), score tables, the persistent
rollout kernel (grid barrier; multi-tile CTAs), the split-step kernels, sampling, the REINFORCE backward.

    compute-sanitizer --tool racecheck python tools/sanitize_small.py
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "vrp-gym_b200"), ROOT]
import numpy as np
import torch

import vrpx
from agents import IRPAgent, TSPAgent, VRPAgent
from gym_vrp.envs import IRPEnv, TSPEnv, VRPEnv

torch.manual_seed(0)
L = vrpx.lib()
dev = vrpx.require_device()
# GEMM shapes: K = 128 (cross-terms-first order), K = 512 (pipelined), K = 1024 (split accumulator), ragged rows
for (R, K, NOUT) in ((300, 128, 384), (260, 512, 128), (200, 1024, 128)):
    X = torch.randn(R, K, device=dev)
    W = torch.randn(NOUT, K, device=dev) / K ** 0.5
    Y = torch.empty(R, NOUT, device=dev)
    vrpx.check(L.vrpx_debug_gemm(vrpx.ptr(X), R, K, vrpx.ptr(W), NOUT, None, 1, None, None, None, vrpx.ptr(Y), 0, vrpx.stream_ptr(dev)))
# weight-gradient GEMM on tcgen05 (R >= 8192 rows, ragged last block) and the fused in-projection + attention kernel
A = torch.randn(8192 + 37, 128, device=dev) * 1e-3
Bm = torch.randn(8192 + 37, 256, device=dev)
Cw = torch.zeros(128, 256, device=dev)
vrpx.check(L.vrpx_gemm_tn_accumulate(vrpx.ptr(A), vrpx.ptr(Bm), vrpx.ptr(Cw), A.shape[0], 128, 256, vrpx.stream_ptr(dev)))
for (Bq, Nq) in ((37, 50), (9, 21), (5, 100)):
    X = torch.randn(Bq * Nq, 128, device=dev)
    W = torch.randn(384, 128, device=dev) / 128 ** 0.5
    bq = torch.randn(384, device=dev) * 0.1
    att = torch.empty(Bq * Nq, 128, device=dev)
    vrpx.check(L.vrpx_debug_qkv_attention(vrpx.ptr(X), vrpx.ptr(W), vrpx.ptr(bq), Bq, Nq, vrpx.ptr(att), vrpx.stream_ptr(dev)))
torch.cuda.synchronize()
big = int(os.environ.get("SANITIZE_B", "0"))
for Env, Agent, N, B in ((TSPEnv, TSPAgent, 12, 40), (VRPEnv, VRPAgent, 9, 24), (IRPEnv, IRPAgent, 10, 24)):
    B = big or B
    env = Env(N, B, 1, seed=3)
    st = env.get_state()
    mask = (st[0] if isinstance(st, tuple) else st)[:, :, -1]
    a = np.array([np.flatnonzero(mask[b] == 0)[0] for b in range(B)])
    env.step(a[:, None])
    agent = Agent(seed=3)
    for tables in (True, False):
        agent.model.decoder.score_tables = tables
        env.reset()
        loss = agent.evaluate(env)
    agent.model.decoder.score_tables = True
    agent.model.train()
    loss_m, loss_b, logp = agent.step(env, (False, True))
    agent.policy_gradient_step((loss_m - loss_b) * -1, logp)
    torch.cuda.synchronize()
    print(type(env).__name__, "ok", float(loss.mean()), flush=True)
# multi-tile CTAs of the persistent kernel: more than 148 x 16 instances
env = TSPEnv(8, 2600, 0, seed=1, instance_rng="philox")
agent = TSPAgent(seed=1)
agent.model.decoder.score_tables = False
print("multi-tile", float(agent.evaluate(env).mean()), flush=True)
