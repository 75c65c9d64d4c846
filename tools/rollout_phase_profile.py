"""Per-phase cycle breakdown of the persistent rollout kernel (debug counters, thread 0 of every CTA).
The split-step launches are switched off, so the whole episode runs the classic loop (no score tables) inside the
persistent kernel."""
import ctypes as C
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "vrp-gym_b200"), ROOT]
import torch
import vrpx
from agents import TSPAgent
from agents.graph_encoder import run_encoder
from gym_vrp.envs import TSPEnv

B = int(sys.argv[1]) if len(sys.argv) > 1 else 65536
N = 50
agent = TSPAgent(seed=69)
agent.model.eval()
env = TSPEnv(N, B, 0, seed=69, instance_rng="philox")
buf = torch.zeros(8, dtype=torch.int64, device="cuda")
L = vrpx.lib()
L.vrpx_debug_rollout_profile.argtypes = [C.c_void_p]
L.vrpx_debug_rollout_profile.restype = None
L.vrpx_debug_rollout_split(0)
with torch.no_grad():
    for rep in range(3):
        env.restart_episode()
        h = run_encoder(agent.model.encoder, env=env)
        if rep == 2:
            L.vrpx_debug_rollout_profile(C.c_void_p(buf.data_ptr()))
        agent.model.decoder.rollout_episode(env, h, greedy=True)
torch.cuda.synchronize()
L.vrpx_debug_rollout_profile(None)
c = buf.cpu().tolist()
names = ["P0 gather", "P1 GEMM-A", "P2 pass2 + wait for other warps", "P3 GEMM-B", "P4 logits+env", "grid barrier", "P2 pass1 (warp 0)", "P2 softmax (warp 0)"]
tot = sum(c)
for n, v in zip(names, c):
    if v:
        print(f"{n:16s} {v/tot*100:5.1f}%")
