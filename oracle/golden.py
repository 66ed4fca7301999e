"""Reader and writer of tests/golden/*.npz.

The fixtures stay small.  Two of them would not if they stored their large arrays whole, so:
  * an input that `pigeon_b200.synthetic` or a seeded torch generator rebuilds is stored as the XOR of its bytes with the
    rebuilt array (`<key>_xor`: zero wherever the two agree, which compresses to almost nothing), or not at all when the
    rebuild is already bit-identical;
  * the reference's (1000, D) weight and gradient outputs of the head fine-tune (train_head) are kept for a fixed, seeded
    sample of their elements (`sample`, indices into the flattened matrix).
`meta["sha256"]` records every array rebuilt on load, so a generator that no longer reproduces its input is an error
rather than a silently different comparison.
"""
from __future__ import annotations

import hashlib
import json
import os

import numpy as np
import torch

from pigeon_b200 import synthetic

GOLD = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

# (C, D) reference outputs of train_head.npz stored for the sampled elements only
TRAIN_HEAD_SAMPLED = ("smooth_grad_w_step1", "smooth_w_step1", "smooth_w_final", "index_grad_w_step1", "index_w_step1",
                      "index_w_final", "multitask_w_final")
TRAIN_HEAD_SAMPLE = 3072


def head_weights(C, D, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(C, D, generator=g) * 0.03, torch.randn(C, generator=g) * 0.01


def sha256(a: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _rebuilt(name: str, meta: dict) -> dict:
    """The arrays of fixture `name` that are rebuilt from seeds, before any stored XOR residual is applied."""
    if name == "train_head":
        w0, b0 = head_weights(meta["C"], meta["D"], meta["w_seed"])
        g = torch.Generator().manual_seed(meta["emb_seed"])
        emb = torch.randn(meta["steps"] * meta["acc"], meta["B"], 4, meta["D"], generator=g) * 0.5
        return dict(w0=w0.numpy(), b0=b0.numpy(), emb=emb.numpy(), centroids=synthetic.synthetic_geocells(meta["C"], 0))
    if name == "loops":
        bk = meta["bank"]
        bank = synthetic.synthetic_bank(bk["C"], bk["P"], bk["D"], seed=bk["seed"], members_mean=bk["members"],
                                        empty_cells=bk["empty_cells"])
        return {"head_w": head_weights(meta["C"], meta["D"], meta["head_seed"])[0].numpy(),
                "centroids": synthetic.synthetic_geocells(meta["C"], 0), **{f"bank_{k}": v for k, v in bank.items()}}
    return {}


def _bytes(a: np.ndarray) -> np.ndarray:
    return np.ascontiguousarray(a).reshape(-1).view(np.uint8)


def load(name: str):
    """(dict of full arrays, meta) of tests/golden/<name>.npz."""
    z = np.load(os.path.join(GOLD, name + ".npz"), allow_pickle=False)
    d = {k: z[k] for k in z.files}
    meta = json.loads(str(d["meta"])) if "meta" in d else {}
    for k, base in _rebuilt(name, meta).items():
        x = d.pop(k + "_xor", None)
        full = base if x is None else (_bytes(base) ^ x).view(base.dtype).reshape(base.shape)
        if sha256(full) != meta["sha256"][k]:
            raise AssertionError(f"{name}.npz: the rebuilt {k} is not the array the reference was run on")
        d[k] = full
    return d, meta


def save(name: str, arrays: dict, meta: dict) -> None:
    """Writes tests/golden/<name>.npz, storing what `load` rebuilds as described in the module docstring."""
    arrays, meta = dict(arrays), dict(meta)
    if name == "train_head":
        sample = np.sort(np.random.default_rng(0).choice(meta["C"] * meta["D"], TRAIN_HEAD_SAMPLE, replace=False))
        arrays["sample"] = sample.astype(np.int32)
        for k in TRAIN_HEAD_SAMPLED:
            arrays[k] = arrays[k].reshape(-1)[sample]
    meta["sha256"] = {}
    for k, base in _rebuilt(name, meta).items():
        full = arrays.pop(k)
        assert full.dtype == base.dtype and full.shape == base.shape, k
        x = _bytes(full) ^ _bytes(base)
        if x.any():
            arrays[k + "_xor"] = x
        meta["sha256"][k] = sha256(full)
    np.savez_compressed(os.path.join(GOLD, name + ".npz"), meta=json.dumps(meta), **arrays)
