"""Evaluation driver: trained agent vs RandomAgent on seeded instances -> CSV of per-instance costs.

Same command line and CSV schema as the reference script (reproduction.py:17-77), running on the CUDA rollout path:

    python vrp-gym_b200/reproduction.py --env_type VRP --num_nodes 20 --model_path ./check_points/vrp_20_123/model_epoch_850.pt

The agent plays the instances drawn in the env constructor (no reset), the random agent plays a snapshot of the same env.
Video capture is attempted only if `gym` is installed (rendering is outside the accelerated path).
"""
import csv
import os
import sys
from argparse import ArgumentParser
from copy import deepcopy

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import torch  # noqa: E402

from agents import IRPAgent, RandomAgent, TSPAgent, VRPAgent  # noqa: E402
from gym_vrp.envs import IRPEnv, TSPEnv, VRPEnv  # noqa: E402

ENVS = {"TSP": TSPEnv, "VRP": VRPEnv, "IRP": IRPEnv}
AGENTS = {"TSP": TSPAgent, "VRP": VRPAgent, "IRP": IRPAgent}


def reproduce(seeds, num_nodes, batch_size, csv_path, model_path, num_draw, env_type, video=False, allow_untrained=False,
              samples=None):
    # the reference loads the checkpoint unconditionally (reproduction.py:44) and fails without it; so does this script,
    # unless --allow_untrained asks for seed-initialised weights, which are then labelled as such in the CSV
    trained = bool(model_path) and os.path.exists(model_path)
    if not trained and not allow_untrained:
        raise FileNotFoundError(f"checkpoint {model_path!r} not found (pass --allow_untrained to evaluate seed-initialised weights)")
    label = f"{env_type}-Agent" if trained else f"{env_type}-Agent-untrained"
    with open(csv_path, "w+", newline="") as f:
        csv.writer(f).writerow(["Model", "Seed", "Mean Distance"])
    for seed in seeds:
        env = ENVS[env_type](num_nodes=num_nodes, batch_size=batch_size, num_draw=num_draw, seed=seed)
        env_random = deepcopy(env)
        if video:
            env.enable_video_capturing(video_save_path=f"./videos/video_{env_type}_{num_nodes}_{seed}.mp4")
        agent = AGENTS[env_type](seed=seed)
        if trained:
            agent.model.load_state_dict(torch.load(model_path, map_location=agent.device))
        random_agent = RandomAgent(seed=seed)
        random_agent.eval()
        cost_agent = agent.evaluate(env, samples=samples)
        cost_random = random_agent(env_random)
        with open(csv_path, "a", newline="") as f:
            w = csv.writer(f)
            for ca, cr in zip(cost_agent.tolist(), cost_random.tolist()):
                w.writerow([label, seed, ca])
                w.writerow([f"{env_type}-Random-Agent", seed, cr])


if __name__ == "__main__":
    ap = ArgumentParser()
    ap.add_argument("--seeds", type=int, nargs="+", default=[1234, 2468, 2048])
    ap.add_argument("--batch_size", type=int, default=256)
    ap.add_argument("--num_nodes", type=int, default=20)
    ap.add_argument("--num_draw", type=int, default=3)
    ap.add_argument("--csv_path", type=str, default="reproduction_results.csv")
    ap.add_argument("--model_path", type=str, default="./check_points/model_epoch__tsp_850.pt")
    ap.add_argument("--env_type", type=str, default="TSP", choices=sorted(ENVS))
    ap.add_argument("--video", action="store_true")
    ap.add_argument("--samples", type=int, default=None, help="evaluate the best of K sampled tours per instance (default: greedy)")
    ap.add_argument("--allow_untrained", action="store_true", help="evaluate seed-initialised weights when the checkpoint is missing")
    args = ap.parse_args()
    print(vars(args))
    reproduce(**vars(args))
