"""TSPModel / TSPAgent — attention policy and REINFORCE trainer for TSPEnv on the fused CUDA rollout.

Surface as in the reference (agents/graph_tsp_agent.py:19-306): `TSPModel(node_dim, emb_dim, hidden_dim,
num_attention_layers, num_heads).forward(env, rollout) -> (acc_loss, acc_log_prob)` and
`TSPAgent(...).train / step / evaluate / baseline_update / save_model`.

`forward` replaces the reference's Python `while not done` loop (:78-88: decoder on device -> actions to
host -> numpy/networkx env.step -> state back to device) by two launches: `vrpx_encoder_forward` and the
persistent `vrpx_rollout` kernel that runs every decode step and environment transition on the GPU.
"""
from __future__ import annotations

import csv
import logging
import os
import time
from copy import deepcopy
from typing import Tuple

import numpy as np
import torch
import torch.nn as nn
from scipy import stats

import vrpx

from .graph_decoder import GraphDecoder, check_samples
from .graph_encoder import GraphEncoder, run_encoder

logging.basicConfig(level=logging.INFO)


class TSPModel(nn.Module):
    _USES_DEPOT_EMBED = False

    def __init__(self, node_dim: int, emb_dim: int, hidden_dim: int, num_attention_layers: int, num_heads: int):
        super().__init__()
        self.device = torch.device("cuda:0" if torch.cuda.is_available() else "cpu")
        self.encoder = GraphEncoder(node_input_dim=node_dim, embedding_dim=emb_dim, hidden_dim=hidden_dim,
                                    num_attention_layers=num_attention_layers, num_heads=num_heads)
        self.decoder = GraphDecoder(emb_dim=emb_dim, num_heads=8, v_dim=emb_dim, k_dim=emb_dim)
        self.coupling = None      # glimpse-mask coupling group; None = the whole batch (reference semantics)
        self.sample_offset = 0    # global id of this shard's first instance (shard-invariant sampling)
        self.last_rollout = None  # dict from GraphDecoder.rollout_episode (tape, steps, ...)

    def backward(self, wts: torch.Tensor):
        """Accumulate d(sum_b wts[b] * log_prob[b])/d(theta) of the LAST sampled train-mode rollout into .grad.  After
        forward_samples(env, K), wts is (K,B) like its log-probs."""
        from vrpx import backward as bw

        ctx = self.last_rollout
        if ctx is None or "enc_saved" not in ctx:
            raise vrpx.VrpxError("no rollout recorded for backward: call model(env, rollout=False) or "
                                 "model.forward_samples(env, K) in train mode with grad enabled")
        if "samples" in ctx:
            shape = (ctx["samples"], ctx["env"].batch_size)
            if tuple(wts.shape) != shape:
                raise ValueError(f"wts of a K-sample rollout must be (K, B) = {shape}, got {tuple(wts.shape)}")
            wts = wts.reshape(-1)
        dH = bw.decoder_backward(self.decoder, ctx["env"], ctx["emb"], ctx, wts, gemm_path=self.encoder.gemm_path)
        bw.encoder_backward(self.encoder, ctx["env"], ctx["depot"], ctx["enc_saved"], dH, gemm_path=self.encoder.gemm_path)
        self.last_rollout = None  # the saved activations are large: release them

    def forward(self, env, rollout: bool = False, *, tape=None, want_logits: bool = False) -> Tuple[torch.Tensor, torch.Tensor]:
        """Play the environment to the end.  rollout=True: greedy; False: sample (Philox stream keyed by the
        torch global seed).  Returns (acc_loss = -tour length (B,), acc_log_prob (B,)) on the device."""
        if not hasattr(env, "_view"):
            raise vrpx.VrpxError("the fused rollout needs a device-resident gym_vrp env (TSPEnv/VRPEnv/IRPEnv of this package)")
        dev = env._device
        if next(self.parameters()).device != dev:
            self.to(dev)
        # host-side edits (sampler.graphs[i].nodes[n]["coordinates"] = ...) reach the device BEFORE the encoder reads them
        env._sync_instances()
        depot = env._depot if self._USES_DEPOT_EMBED else None
        # a sampled rollout of a model in train mode under grad is the REINFORCE forward: keep what backward needs
        need_grad = self.training and torch.is_grad_enabled() and (not rollout)
        enc_saved = None
        if need_grad:
            h, enc_saved = run_encoder(self.encoder, env=env, depot=depot, gemm_path=self.encoder.gemm_path, save=True)
        else:
            h = run_encoder(self.encoder, env=env, depot=depot, gemm_path=self.encoder.gemm_path)
        seed = 0 if (rollout or tape is not None) else int(torch.randint(0, 2 ** 62, (1,)).item())
        out = self.decoder.rollout_episode(env, h, greedy=rollout, tape_in=tape, want_logits=want_logits,
                                           coupling=self.coupling, seed=seed, offset=self.sample_offset,
                                           save_for_backward=need_grad)
        out["emb"] = h
        if need_grad:
            out["enc_saved"], out["env"], out["depot"] = enc_saved, env, depot
        self.last_rollout = out
        self.decoder.reset()
        return -out["cost"], out["logp"]

    def forward_samples(self, env, num_samples: int) -> Tuple[torch.Tensor, torch.Tensor]:
        """K = num_samples sampled tours per instance from one encoder pass (GraphDecoder.rollout_samples; the Philox
        seed comes from the torch global RNG as in `forward`, copy k uses offset sample_offset + k·B).  env is left
        untouched.  Returns (-cost (K,B), log_prob (K,B)) on the device.

        In train mode under grad this is the REINFORCE forward of K-sample training: the train-mode encoder runs ONCE,
        over the B instances (BatchNorm batch statistics and one running-statistic update from them), and backward(wts)
        with wts (K,B) back-propagates sum_kb wts[k,b] log_prob[k,b].  K identical copies have the batch mean and biased
        variance of one copy and their BatchNorm backward sums over the copies, so the gradient equals that of the
        K-fold replicated batch; only the running variance differs, by the replicated batch's unbiased-variance factor."""
        if not hasattr(env, "_view"):
            raise vrpx.VrpxError("the fused rollout needs a device-resident gym_vrp env (TSPEnv/VRPEnv/IRPEnv of this package)")
        need_grad = self.training and torch.is_grad_enabled()
        check_samples(env, num_samples, self.coupling, train=need_grad)
        dev = env._device
        if next(self.parameters()).device != dev:
            self.to(dev)
        env._sync_instances()
        depot = env._depot if self._USES_DEPOT_EMBED else None
        enc_saved = None
        if need_grad:
            h, enc_saved = run_encoder(self.encoder, env=env, depot=depot, gemm_path=self.encoder.gemm_path, save=True)
        else:
            h = run_encoder(self.encoder, env=env, depot=depot, gemm_path=self.encoder.gemm_path)
        seed = int(torch.randint(0, 2 ** 62, (1,)).item())
        out = self.decoder.rollout_samples(env, h, num_samples, seed=seed, offset=self.sample_offset,
                                           coupling=self.coupling, save_for_backward=need_grad)
        out["emb"] = h
        if need_grad:
            out["enc_saved"], out["env"], out["depot"] = enc_saved, env, depot
        self.last_rollout = out
        return -out["cost"], out["logp"]

    @torch.no_grad()
    def sample_best(self, env, num_samples: int) -> dict:
        """Best of K = num_samples sampled tours per instance from one encoder pass (GraphDecoder.rollout_samples; the
        Philox seed comes from the torch global RNG as in `forward`).  Records nothing for backward and leaves env
        untouched.  Returns dict(cost (B,) smallest tour length, tour (steps,B) its actions, logp (B,) its log-prob,
        index (B,) its copy k (the lowest k on ties), costs (K,B) every copy's tour length)."""
        if not hasattr(env, "_view"):
            raise vrpx.VrpxError("the fused rollout needs a device-resident gym_vrp env (TSPEnv/VRPEnv/IRPEnv of this package)")
        dev = env._device
        if next(self.parameters()).device != dev:
            self.to(dev)
        env._sync_instances()
        h = run_encoder(self.encoder, env=env, depot=env._depot if self._USES_DEPOT_EMBED else None,
                        gemm_path=self.encoder.gemm_path)
        seed = int(torch.randint(0, 2 ** 62, (1,)).item())
        out = self.decoder.rollout_samples(env, h, num_samples, seed=seed, offset=self.sample_offset,
                                           coupling=self.coupling)
        costs = out["cost"]
        K, B = costs.shape
        ks = torch.arange(K, device=dev)[:, None].expand(K, B)
        best = torch.where(costs == costs.min(0, keepdim=True).values, ks, K).min(0).values
        ar = torch.arange(B, device=dev)
        return {"cost": costs[best, ar], "tour": out["tape"][:, best, ar], "logp": out["logp"][best, ar], "index": best,
                "costs": costs}


class TSPAgent:
    _MODEL = TSPModel

    def __init__(self, node_dim: int = 2, emb_dim: int = 128, hidden_dim: int = 512, num_attention_layers: int = 3,
                 num_heads: int = 8, lr: float = 1e-4, csv_path: str = "loss_log.csv", seed=69):
        torch.manual_seed(seed)
        np.random.seed(seed)
        self.device = torch.device("cuda:0" if torch.cuda.is_available() else "cpu")
        self.csv_path = csv_path
        kw = dict(node_dim=node_dim, emb_dim=emb_dim, hidden_dim=hidden_dim,
                  num_attention_layers=num_attention_layers, num_heads=num_heads)
        # construction order matters: it fixes the torch RNG stream and therefore the initial weights
        self.model = TSPModel(**kw).to(self.device)
        self.target_model = TSPModel(**kw).to(self.device)
        self._finish_init(lr)

    def _finish_init(self, lr):
        self.target_model.load_state_dict(self.model.state_dict())
        self.target_model.eval()
        self.opt = torch.optim.Adam(self.model.parameters(), lr=lr)

    # ------------------------------------------------------------------ rollouts
    def step(self, env, rollouts: Tuple[bool, bool], samples: int = None):
        """Reset the env, then play it with the model and (on a snapshot) with the baseline.  As in the
        reference (:251-253) BOTH use rollouts[0].  samples = K: both play K sampled tours per instance instead
        (TSPModel.forward_samples; rollouts is not read) and every result is (K,B)."""
        env.reset()
        if samples is not None:
            loss, log_prob = self.model.forward_samples(env, samples)
            with torch.no_grad():
                loss_b, _ = self.target_model.forward_samples(env, samples)
            return loss, loss_b, log_prob
        env_baseline = deepcopy(env)
        loss, log_prob = self.model(env, rollouts[0])
        with torch.no_grad():
            loss_b, _ = self.target_model(env_baseline, rollouts[0])
        return loss, loss_b, log_prob

    def evaluate(self, env, samples: int = None):
        """Reward (-cost) per instance of the current model: the greedy rollout, or with `samples` = K the best of K
        sampled tours (TSPModel.sample_best; env is left untouched)."""
        self.model.eval()
        if samples is not None:
            return -self.model.sample_best(env, samples)["cost"]
        with torch.no_grad():
            loss, _ = self.model(env, rollout=True)
        return loss

    # ------------------------------------------------------------------ training
    def train(self, env, epochs: int = 100, eval_epochs: int = 1, check_point_dir: str = "./check_points/",
              samples: int = None):
        """REINFORCE with the rollout baseline (reference :155-177).  samples = K: every epoch trains on K sampled tours
        per instance against K sampled baseline tours, from one train-mode encoder pass (TSPModel.forward_samples);
        the baseline update is unchanged."""
        if samples is not None:
            check_samples(env, samples, self.model.coupling, train=True)
        logging.info("Start Training")
        with open(self.csv_path, "w+", newline="") as file:
            csv.writer(file).writerow(["Epoch", "Loss", "Cost", "Advantage", "Time"])
        start_time = time.time()
        for e in range(epochs):
            self.model.train()
            loss_m, loss_b, log_prob = self.step(env, (False, True), samples=samples)
            advantage = (loss_m - loss_b) * -1
            loss = self.policy_gradient_step(advantage, log_prob, samples=samples)
            self.baseline_update(env, eval_epochs)
            logging.info(f"Epoch {e} finished - Loss: {loss}, Advantage: {advantage.mean()} Dist: {loss_m.mean()}")
            with open(self.csv_path, "a", newline="") as file:
                csv.writer(file).writerow([e, float(loss), loss_m.mean().item(), advantage.mean().item(),
                                           time.time() - start_time])
            self.save_model(episode=e, check_point_dir=check_point_dir)

    def policy_gradient_step(self, advantage, log_prob, samples: int = None):
        """loss = mean(advantage * log_prob); backward; Adam step (reference :179-186).  samples = K: advantage and
        log_prob are (K,B) from step(env, ..., samples=K) and the mean runs over all K·B tours."""
        if samples is not None and (advantage.dim() != 2 or advantage.shape[0] != samples):
            raise ValueError(f"with samples={samples} the advantage must be (K, B), got {tuple(advantage.shape)}")
        B = advantage.numel()
        loss = (advantage * log_prob).mean()
        self.opt.zero_grad()
        # d loss / d log_prob_b = advantage_b / B; the gradient flows only through log_prob (advantage is data)
        self.model.backward(advantage.detach() / B)
        self._allreduce_gradients()
        self.opt.step()
        return loss

    def _allreduce_gradients(self):
        """Data-parallel training: every rank holds a shard of the batch (its own reference batch); the gradient of
        the global mean loss is the mean over ranks of the local gradients — one flat NCCL all-reduce."""
        import torch.distributed as dist

        if not (dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1):
            return
        from vrpx import sharding

        grads = [p.grad for p in self.model.parameters() if p.grad is not None]
        flat = torch.cat([g.reshape(-1) for g in grads])
        sharding.allreduce_mean_(flat)
        off = 0
        for g in grads:
            g.copy_(flat[off:off + g.numel()].view_as(g))
            off += g.numel()

    def save_model(self, episode: int, check_point_dir: str) -> None:
        if not os.path.exists(check_point_dir):
            os.makedirs(check_point_dir)
        if episode % 50 == 0 and episode != 0:
            torch.save(self.model.state_dict(), check_point_dir + f"model_epoch_{episode}.pt")

    def baseline_update(self, env, batch_steps: int = 3):
        """Replace the baseline by the current model iff it is significantly better (paired t-test, :275-306)."""
        logging.info("Update Baseline")
        self.model.eval()
        self.target_model.eval()
        current_model_cost, baseline_model_cost = [], []
        with torch.no_grad():
            for _ in range(batch_steps):
                loss, loss_b, _ = self.step(env, [True, True])
                current_model_cost.append(loss)
                baseline_model_cost.append(loss_b)
        current_model_cost = torch.cat(current_model_cost)
        baseline_model_cost = torch.cat(baseline_model_cost)
        import torch.distributed as dist

        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            from vrpx import sharding  # same decision on every rank from 3 all-reduced doubles

            mean_d, p_value = sharding.paired_ttest_allreduce(-current_model_cost, -baseline_model_cost)
            advantage = torch.tensor(mean_d)
        else:
            advantage = ((current_model_cost - baseline_model_cost) * -1).mean()
            _, p_value = stats.ttest_rel(current_model_cost.tolist(), baseline_model_cost.tolist())
        if advantage.item() <= 0 and p_value <= 0.05:
            print("replacing baceline")
            self.target_model.load_state_dict(self.model.state_dict())
