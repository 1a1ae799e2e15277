"""Loading helpers for the reference-generated fixtures under tests/golden/ (see
tests/golden/make_reference_vectors.py for how they were produced)."""
import itertools
import os

import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def unpack_state_dict(sd):
    """Inverse of make_reference_vectors.pack_state_dict: densify the (shape, idx, val) `w3j` records."""
    out = {}
    for k, v in sd.items():
        if isinstance(v, dict):
            t = torch.zeros(v["w3j_shape"], dtype=v["dtype"])
            t[tuple(v["idx"].long().T)] = v["val"]
            out[k] = t
        else:
            out[k] = v
    return out


def _load_parts(stem):
    """Join <stem>_1.pt, <stem>_2.pt, ... (dicts of lists, split to keep every file small) into one dict of lists."""
    out = {}
    for k in itertools.count(1):
        path = os.path.join(GOLDEN, f"{stem}_{k}.pt")
        if not os.path.exists(path):
            break
        for key, records in torch.load(path, weights_only=False).items():
            out.setdefault(key, []).extend(records)
    if not out:
        raise FileNotFoundError(f"no {stem}_<k>.pt under {GOLDEN}")
    return out


def load_models():
    return _load_parts("ref_models")["models"]


def load_ops():
    return _load_parts("ref_ops")


def model_case_ids():
    return [r["name"] for r in load_models()]
