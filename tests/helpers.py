"""Shared helpers for the parity tests (test infrastructure; may import oracle/)."""
import glob
import hashlib
import json
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden")

EXACT_KEYS = ("info:env_id", "info:players.env_id", "elapsed_step", "done", "discount",
              "step_type", "trunc")
INT_TASKS = ("FrozenLake", "Catch", "Taxi", "NChain", "CliffWalking", "Blackjack")
N_ACT = {"CartPole": 2, "Acrobot": 3, "MountainCar": 3, "FrozenLake": 4, "Catch": 3,
         "Taxi": 6, "NChain": 2, "CliffWalking": 4, "Blackjack": 2}
# registered max_episode_steps (envpool/*/registration.py) and default iopt per task
REGISTERED = {
    "CartPole": (500, -1), "Pendulum": (200, 1), "Acrobot": (500, -1),
    "MountainCar": (200, -1), "MountainCarContinuous": (999, -1),
    "FrozenLake": (100, 4), "Catch": (-1, -1), "Taxi": (200, -1), "NChain": (1000, -1),
    "CliffWalking": (-1, 0), "Blackjack": (-1, 2),
}


def golden_cases():
    return sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "*.npz")))


def load_golden(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    meta = json.loads(str(z["meta"]))
    data = {k: z[k] for k in z.files if k != "meta"}
    return meta, data


def space_desc(sp):
    """JSON description of a gymnasium space or dm_env spec."""
    d = {"type": type(sp).__name__, "shape": list(sp.shape or ()), "dtype": str(sp.dtype)}
    for k in ("low", "high", "minimum", "maximum"):
        if hasattr(sp, k):
            d[k] = [float(x) for x in np.ravel(getattr(sp, k))]
    for k in ("n", "start", "num_values"):
        if hasattr(sp, k) and isinstance(getattr(sp, k), int):
            d[k] = getattr(sp, k)
    return d


def jsonable(v):
    """A config value as JSON would give it back (tuples and arrays as lists)."""
    if isinstance(v, dict):
        return {k: jsonable(x) for k, x in v.items()}
    if isinstance(v, (list, tuple, np.ndarray)):
        return [jsonable(x) for x in v]
    return v.item() if isinstance(v, np.generic) else v


def batch_digest(batch):
    """64-bit digest of a batch: name, dtype, shape and bytes of every key, in name order."""
    h = hashlib.blake2b(digest_size=8)
    for k in sorted(batch):
        a = np.ascontiguousarray(batch[k])
        h.update(f"{k}|{a.dtype.str}|{a.shape}|".encode())
        h.update(a.tobytes())
    return int.from_bytes(h.digest(), "little")


def random_actions(task, rng, shape_prefix, act_dtype=None):
    if task in ("Pendulum", "MountainCarContinuous"):
        return rng.uniform(-2.5, 2.5, size=tuple(shape_prefix) + (1,)).astype(np.float32)
    if task == "HalfCheetah":
        return rng.uniform(-1.0, 1.0, size=tuple(shape_prefix) + (6,)).astype(np.float64)
    return rng.integers(0, N_ACT[task], size=tuple(shape_prefix)).astype(np.int32)


def row_tolerance(task, float_atol, elapsed):
    """Per-row float tolerance for FREE-RUNNING trajectory comparisons.  Acrobot is a
    chaotic double pendulum: the <= 2 ulp difference between CUDA's and glibc's double
    sin/cos (1e-16) is amplified along an episode (measured 1.5e-6 after 400 steps), so its
    free-running tolerance opens with the depth into the episode.  Its per-step arithmetic
    is pinned separately, without amplification, by the teacher-forced test
    (test_gpu_parity.py::test_teacher_forced_single_step).  Every other env keeps
    float_atol for the whole episode."""
    tol = np.full(elapsed.shape, float_atol, dtype=np.float64)
    if task == "Acrobot" and float_atol > 0:
        tol = np.where(elapsed > 300, 5e-2, np.where(elapsed > 150, 1e-4, float_atol))
    return tol


def assert_batch_equal(got, want, task, float_atol=0.0, ctx=""):
    """Integer/bool/flag columns bit-exact; float columns within float_atol (0 = exact),
    relative-absolute: |err| <= tol * (1 + |ref|)."""
    row_tol = row_tolerance(task, float_atol, want["elapsed_step"])
    for k, w in want.items():
        g = got[k]
        assert g.shape == w.shape, (ctx, k, g.shape, w.shape)
        assert g.dtype == w.dtype, (ctx, k, g.dtype, w.dtype)
        if g.dtype.kind in "ib" or k in EXACT_KEYS or task in INT_TASKS or float_atol == 0.0:
            if not np.array_equal(g, w):
                bad = np.argwhere(np.asarray(g != w))[:5]
                raise AssertionError(f"{ctx} key {k}: mismatch at {bad.tolist()} "
                                     f"got {g[tuple(bad[0])]} want {w[tuple(bad[0])]}")
        else:
            err = np.abs(g.astype(np.float64) - w.astype(np.float64))
            rt = row_tol.reshape((-1,) + (1,) * (w.ndim - 1))
            tol = rt * (1.0 + np.abs(w.astype(np.float64)))
            if not np.all(err <= tol):
                i = np.unravel_index(np.argmax(err - tol), err.shape)
                raise AssertionError(f"{ctx} key {k}: |err|={err[i]:.3e} > tol at {i} "
                                     f"got {g[i]} want {w[i]}")
