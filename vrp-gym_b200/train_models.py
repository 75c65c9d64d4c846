"""Training driver: TSP / VRP / IRP agents for N in {20, 30, 40} and seeds {69, 123}, batch 256, 851 epochs — the runs
behind the reference's train_logs/ and check_points/ (train_models.py:4-39) — on the CUDA rollout + backward path.

    python vrp-gym_b200/train_models.py [--epochs 851] [--batch_size 256] [--nodes 20 30 40] [--seeds 69 123]
                                        [--samples K]
"""
import os
import sys
from argparse import ArgumentParser

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from agents import IRPAgent, TSPAgent, VRPAgent  # noqa: E402
from gym_vrp.envs import IRPEnv, TSPEnv, VRPEnv  # noqa: E402

if __name__ == "__main__":
    ap = ArgumentParser()
    ap.add_argument("--epochs", type=int, default=851)
    ap.add_argument("--batch_size", type=int, default=256)
    ap.add_argument("--nodes", type=int, nargs="+", default=[20, 30, 40])
    ap.add_argument("--seeds", type=int, nargs="+", default=[69, 123])
    ap.add_argument("--kinds", nargs="+", default=["tsp", "vrp", "irp"])
    ap.add_argument("--samples", type=int, default=None,
                    help="train on K sampled tours per instance from one encoder pass (default: one tour, the reference)")
    a = ap.parse_args()
    os.makedirs("./train_logs", exist_ok=True)
    table = {"tsp": (TSPEnv, TSPAgent), "vrp": (VRPEnv, VRPAgent), "irp": (IRPEnv, IRPAgent)}
    for seed in a.seeds:
        for n in a.nodes:
            for kind in a.kinds:
                Env, Agent = table[kind]
                env = Env(num_nodes=n, batch_size=a.batch_size, seed=seed)
                agent = Agent(seed=seed, csv_path=f"./train_logs/loss_log_{kind}_{n}_{seed}.csv")
                agent.train(env, epochs=a.epochs, check_point_dir=f"./check_points/{kind}_{n}_{seed}/",
                            samples=a.samples)
