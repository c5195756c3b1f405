"""Golden arrays too large for one file: <stem>.part<k>.npz, every array split along axis 0 across the parts (0-d arrays
live in part 0), so that each file of the repository stays under 1 MB.  load() puts them back together."""
from __future__ import annotations

import glob

import numpy as np


def save(stem: str, arrays: dict, parts: int = 2) -> None:
    split = {k: np.array_split(np.asarray(a), parts) if np.ndim(a) else [np.asarray(a)] for k, a in arrays.items()}
    for p in range(parts):
        np.savez_compressed(f"{stem}.part{p}.npz", **{k: v[p] for k, v in split.items() if p < len(v)})


def load(stem: str) -> dict:
    files = sorted(glob.glob(f"{stem}.part*.npz"), key=lambda f: int(f.rsplit(".part", 1)[1][:-4]))
    if not files:
        raise FileNotFoundError(f"{stem}.part0.npz")
    pieces: dict = {}
    for f in files:
        with np.load(f) as z:
            for k in z.files:
                pieces.setdefault(k, []).append(z[k])
    return {k: v[0] if v[0].ndim == 0 else np.concatenate(v) for k, v in pieces.items()}
