"""Generate the golden fixtures in this directory FROM THE REFERENCE ITSELF.

Runs in the build container only (needs /root/reference, compiled by
`make -C oracle ref` into oracle/_ref/libenvpool_ref.so: the reference's own
AsyncEnvPool<Env> + env headers, unmodified).  The reference ships no golden vectors
for these envs (SURVEY.md section 8c), so these recorded trajectories are the pin for
both the CPU restatement (oracle/ep_oracle.c) and the CUDA path.

    python tests/golden/make_golden.py

Each <name>.npz holds: meta (json string: task, seed, max_episode_steps, iopt,
num_envs), `actions` [T, N, ...] and one `[T+1, N, ...]` array per state key (index 0
= the reset() batch, index t+1 = the batch returned by step(actions[t])).

digests/ref_stream.npz: one 32-env, 300-step run of every registered task on seed 19, the
actions of all tasks drawn in turn from one random stream (seed 31).  Stored as digests
(helpers.batch_digest) of the action stream and of every batch the reference returned, so
that a comparison stays bit-exact at every step while the file stays a few kB.
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle.ref_lib import ENV_TABLE, RefPool  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from helpers import REGISTERED, batch_digest, random_actions  # noqa: E402

# name, task, registered max_episode_steps (envpool/*/registration.py), iopt, N, T
CASES = [
    ("cartpole_v1", "CartPole", 500, -1, 16, 400),
    ("cartpole_v0_short", "CartPole", 200, -1, 8, 300),
    ("cartpole_trunc12", "CartPole", 12, -1, 16, 200),
    ("pendulum_v0", "Pendulum", 200, 0, 16, 450),
    ("pendulum_v1", "Pendulum", 200, 1, 16, 450),
    ("acrobot_v1", "Acrobot", 500, -1, 16, 1100),
    ("mountain_car_v0", "MountainCar", 200, -1, 16, 450),
    ("mountain_car_continuous_v0", "MountainCarContinuous", 999, -1, 8, 1100),
    ("frozen_lake_v1", "FrozenLake", 100, 4, 32, 400),
    ("frozen_lake8x8_v1", "FrozenLake", 200, 8, 32, 500),
    ("catch_v0", "Catch", -1, -1, 16, 60),
    ("taxi_v3", "Taxi", 200, -1, 32, 500),
    ("nchain_v0", "NChain", 1000, -1, 16, 1100),
    ("cliffwalking_v0", "CliffWalking", -1, 0, 32, 400),
    ("cliffwalking_slippery_v1", "CliffWalking", -1, 1, 32, 400),
    ("blackjack_v1", "Blackjack", -1, 2, 64, 200),
    ("blackjack_natural", "Blackjack", -1, 1, 64, 200),
]
N_ACT = {"CartPole": 2, "Acrobot": 3, "MountainCar": 3, "FrozenLake": 4, "Catch": 3,
         "Taxi": 6, "NChain": 2, "CliffWalking": 4, "Blackjack": 2}


def actions_for(task, rng, T, N):
    dt, shape = ENV_TABLE[task]["act"]
    if dt == np.float32:
        # exceeds the action bounds on purpose: exercises the clipping branches
        return rng.uniform(-2.5, 2.5, size=(T, N) + shape).astype(np.float32)
    return rng.integers(0, N_ACT[task], size=(T, N)).astype(np.int32)


def record(path, task, seed, ms, iopt, acts):
    T, N = acts.shape[:2]
    pool = RefPool(task, N, seed=seed, max_episode_steps=ms, iopt=iopt)
    frames = [pool.reset()]
    for t in range(T):
        frames.append(pool.step(acts[t]))
    pool.close()
    if path is None:
        return frames
    out = {k: np.stack([f[k] for f in frames]) for k in frames[0]}
    meta = dict(task=task, seed=seed, max_episode_steps=ms, iopt=iopt,
                num_envs=N, steps=T, reference="sail-sg/envpool@9cbcd26")
    np.savez_compressed(path, meta=json.dumps(meta), actions=acts, **out)
    return out


def record_stream(N=32, T=300, seed=19):
    rng = np.random.default_rng(31)
    arrays, keys = {}, {}
    for task, (ms, iopt) in REGISTERED.items():
        acts = np.stack([random_actions(task, rng, (N,)) for _ in range(T)])
        frames = record(None, task, seed, ms, iopt, acts)
        keys[task] = sorted(frames[0])
        arrays[task] = np.array([batch_digest(f) for f in frames], dtype=np.uint64)
        arrays[task + ":actions"] = np.array([batch_digest({"actions": acts})], dtype=np.uint64)
    meta = dict(num_envs=N, steps=T, seed=seed, action_seed=31, keys=keys,
                reference="sail-sg/envpool@9cbcd26")
    os.makedirs(os.path.join(HERE, "digests"), exist_ok=True)
    np.savez_compressed(os.path.join(HERE, "digests", "ref_stream.npz"),
                        meta=json.dumps(meta), **arrays)


def main():
    for name, task, ms, iopt, N, T in CASES:
        seed = 7
        rng = np.random.default_rng(sum(map(ord, name)))
        acts = actions_for(task, rng, T, N)
        out = record(os.path.join(HERE, name + ".npz"), task, seed, ms, iopt, acts)
        print(f"{name}: N={N} T={T} dones={int(out['done'].sum())} "
              f"truncs={int(out['trunc'].sum())}")
    record_stream()


if __name__ == "__main__":
    main()
