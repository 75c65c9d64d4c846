#!/usr/bin/env python
"""Record the state_dict layout of the unmodified reference's models (key order, shape, dtype per tensor) as
tests/golden/reference_state_dict_layout.json, the target a checkpoint written by this repo must load into strictly.

TSP and VRP are read from the state_dicts the reference itself saved (ckpt_<kind>_20_123.pt, make_checkpoints.py).
The reference's IRP model is its VRP model built with node_dim=3 (graph_irp_agent.py; SURVEY App. A.5): the VRP layout
with a (128, 3) `encoder.node_embed.weight`.  Its initial values are pinned separately by the reference weight sums in
policy_irp.npz (tests/test_oracle_policy.py::test_seeded_weights_equal_reference).

    python tests/golden/make_layout.py
"""
import json
import os

import torch

HERE = os.path.dirname(os.path.abspath(__file__))


def _layout(sd):
    return [[k, list(v.shape), str(v.dtype).replace("torch.", "")] for k, v in sd.items()]


def main():
    out = {}
    for kind in ("tsp", "vrp"):
        sd = torch.load(os.path.join(HERE, f"ckpt_{kind}_20_123.pt"), map_location="cpu")
        out[kind] = {"source": f"state_dict saved by the reference (ckpt_{kind}_20_123.pt)", "tensors": _layout(sd)}
    irp = [[k, [128, 3] if k == "encoder.node_embed.weight" else s, d] for k, s, d in out["vrp"]["tensors"]]
    out["irp"] = {"source": "the reference VRP layout with node_dim=3 (the reference IRP model)", "tensors": irp}
    kinds = []
    for kind, v in out.items():
        rows = ",\n".join("    " + json.dumps(t) for t in v["tensors"])
        kinds.append(f' "{kind}": {{\n  "source": {json.dumps(v["source"])},\n  "tensors": [\n{rows}\n  ]\n }}')
    with open(os.path.join(HERE, "reference_state_dict_layout.json"), "w") as f:
        f.write("{\n" + ",\n".join(kinds) + "\n}\n")


if __name__ == "__main__":
    main()
