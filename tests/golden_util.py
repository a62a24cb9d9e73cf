"""Golden fixtures of the step path (tests/golden/*.npz): array <-> state-dict conversion shared by the generator
(tests/golden/make_golden.py) and tests/test_golden.py.  TEST INFRASTRUCTURE."""
from __future__ import annotations

import zipfile

import numpy as np

MAXC = 32
FIELDS_F = ("pos", "vel", "ang", "angvel", "vbias", "wbias")
FIELDS_I = ("steps", "mode", "spawn_count", "seed")
HIST_F = ("pos", "vel", "ang", "angvel")


def pack(states: list, prefix: str) -> dict:
    n = len(states)
    out = {}
    for k in FIELDS_F:
        out[f"{prefix}_{k}"] = np.stack([np.asarray(s[k], np.float64) for s in states])
    for k in FIELDS_I:
        out[f"{prefix}_{k}"] = np.array([int(s[k]) for s in states], np.int64)
    out[f"{prefix}_score"] = np.array([s["score"] for s in states], np.int64).reshape(n, 2)
    out[f"{prefix}_obs"] = np.stack([np.asarray(s["obs"], np.float32).reshape(4, 66) for s in states])
    cn = np.zeros(n, np.int64)
    ci = np.zeros((n, MAXC, 3), np.int64)
    cf = np.zeros((n, MAXC, 2), np.float64)
    for i, s in enumerate(states):
        cn[i] = len(s["cache"])
        for j, (p, key, age, jn, jt) in enumerate(s["cache"]):
            ci[i, j] = (p, key, age)
            cf[i, j] = (jn, jt)
    out[f"{prefix}_cache_n"], out[f"{prefix}_cache_i"], out[f"{prefix}_cache_f"] = cn, ci, cf
    if all("hist" in s for s in states):  # the two poses behind the emitted frames t-2, t-1
        for k in HIST_F:
            out[f"{prefix}_hist_{k}"] = np.stack([np.stack([np.asarray(s["hist"][j][k], np.float64) for j in range(2)])
                                                  for s in states])
    return out


def save(path: str, arrays: dict) -> None:
    """np.savez with LZMA instead of deflate, which keeps step_v2.npz under 1 MB; np.load reads it like any .npz."""
    with zipfile.ZipFile(path, "w", compression=zipfile.ZIP_LZMA) as zf:
        for k, v in arrays.items():
            with zf.open(f"{k}.npy", "w") as f:
                np.lib.format.write_array(f, np.asanyarray(v), allow_pickle=False)


def unpack(z, prefix: str) -> list:
    n = len(z[f"{prefix}_steps"])
    states = []
    for i in range(n):
        s = {k: np.array(z[f"{prefix}_{k}"][i]) for k in FIELDS_F}
        for k in FIELDS_I:
            s[k] = int(z[f"{prefix}_{k}"][i])
        s["score"] = (int(z[f"{prefix}_score"][i, 0]), int(z[f"{prefix}_score"][i, 1]))
        s["obs"] = np.array(z[f"{prefix}_obs"][i], np.float32)
        s["cache"] = [(int(a), int(b), int(c), float(z[f"{prefix}_cache_f"][i, j, 0]), float(z[f"{prefix}_cache_f"][i, j, 1]))
                      for j, (a, b, c) in enumerate(z[f"{prefix}_cache_i"][i][: int(z[f"{prefix}_cache_n"][i])])]
        if f"{prefix}_hist_pos" in z:
            s["hist"] = [{k: np.array(z[f"{prefix}_hist_{k}"][i][j]) for k in HIST_F} for j in range(2)]
        states.append(s)
    return states
