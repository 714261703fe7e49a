"""ORACLE (test infrastructure) — tests/golden on disk.

Every file stays under 1 MB, so the two larger vector sets are stored a piece per file:
  ext_attn/<i>_<name>.pt        one extended-attention case each, in generation order
  block_passes/pivotal.pt       the block's configuration, weights and pivotal pass
  block_passes/frame_<i>.pt     the frame pass of keyframe batch i (i < K)
The loaders return the structures oracle/gen_golden.py builds: a list of case dicts, and one dict with
a "frames" list.
"""
from __future__ import annotations

import os

import torch


def _load(path):
    return torch.load(path, weights_only=False)


def save_ext_attn(golden_dir, cases):
    d = os.path.join(golden_dir, "ext_attn")
    os.makedirs(d, exist_ok=True)
    for i, c in enumerate(cases):
        torch.save(c, os.path.join(d, f"{i}_{c['name']}.pt"))


def load_ext_attn(golden_dir):
    d = os.path.join(golden_dir, "ext_attn")
    files = sorted((f for f in os.listdir(d) if f.endswith(".pt")), key=lambda f: int(f.split("_", 1)[0]))
    return [_load(os.path.join(d, f)) for f in files]


def save_block_passes(golden_dir, case):
    d = os.path.join(golden_dir, "block_passes")
    os.makedirs(d, exist_ok=True)
    head = {k: v for k, v in case.items() if k != "frames"}
    assert len(case["frames"]) == case["K"]
    torch.save(head, os.path.join(d, "pivotal.pt"))
    for i, fr in enumerate(case["frames"]):
        torch.save(fr, os.path.join(d, f"frame_{i}.pt"))


def load_block_passes(golden_dir):
    d = os.path.join(golden_dir, "block_passes")
    case = _load(os.path.join(d, "pivotal.pt"))
    case["frames"] = [_load(os.path.join(d, f"frame_{i}.pt")) for i in range(case["K"])]
    return case
