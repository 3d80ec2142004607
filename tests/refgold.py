"""Recorded outputs of the original lora_diffusion package (tests/golden/reference_*.json, written by
scripts/make_golden.py) and the canonical forms they are stored in, so that tests compare with the
original project without needing its source tree.

A tensor is stored as a digest of its dtype, shape and bytes: two digests are equal exactly when
torch.equal holds and the dtypes match, and a whole model's worth of factors fits in a few KB."""
import hashlib
import inspect
import json
import os

import torch

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
TARGET_KEYS = ("unet", "text_encoder")      # metadata entries holding json.dumps(list(set)) target lists


def digest(t: torch.Tensor) -> str:
    t = t.detach().cpu().contiguous()
    h = hashlib.sha256(f"{t.dtype}{tuple(t.shape)}".encode())
    h.update(t.reshape(-1).view(torch.uint8).numpy().tobytes())
    return h.hexdigest()[:16]


def canon_default(v):
    if v is inspect.Parameter.empty:
        return {"empty": True}
    if isinstance(v, (set, frozenset)):
        return {"set": sorted(v)}
    if v is None or isinstance(v, (bool, int, float, str)):
        return v
    return {"repr": repr(v)}


def canon_signature(fn):
    """[[parameter name, canonical default], ...] in declaration order."""
    return [[k, canon_default(p.default)] for k, p in inspect.signature(fn).parameters.items()]


def canon_metadata(meta: dict) -> dict:
    """safetensors metadata with the target-module lists sorted: the original writes list(set), whose
    order depends on the interpreter's string hash seed."""
    return {k: (sorted(json.loads(v)) if k in TARGET_KEYS else v) for k, v in meta.items()}


def load(name: str):
    with open(os.path.join(GOLD, name)) as fh:
        return json.load(fh)
