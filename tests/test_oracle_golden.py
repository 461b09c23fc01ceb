"""CPU: the oracle (oracle/ep_oracle.c) against the golden fixtures recorded from the
reference itself, plus RNG known-answer tests.  This is what pins the oracle."""
import json
import os

import numpy as np
import pytest

from helpers import assert_batch_equal, golden_cases, load_golden


@pytest.mark.parametrize("case", golden_cases())
def test_oracle_reproduces_reference_golden(case):
    from oracle.oracle_lib import OraclePool

    meta, gold = load_golden(case)
    orc = OraclePool(meta["task"], meta["num_envs"], seed=meta["seed"],
                     max_episode_steps=meta["max_episode_steps"], iopt=meta["iopt"])
    keys = [k for k in gold if k != "actions"]
    assert_batch_equal(orc.reset(), {k: gold[k][0] for k in keys}, meta["task"], 0.0,
                       f"{case} reset")
    acts = gold["actions"]
    for t in range(acts.shape[0]):
        assert_batch_equal(orc.step(acts[t]), {k: gold[k][t + 1] for k in keys},
                           meta["task"], 0.0, f"{case} t={t}")


def test_mt19937_known_answers():
    """std::mt19937 known answers: the C++ standard requires the 10000th draw of a
    default-seeded (5489) engine to be 4123659995; first draws of seed 5489 are the
    published MT19937 reference outputs."""
    from oracle.oracle_lib import OraclePool

    pool = OraclePool("CartPole", 1, env_seed=[5489])
    first = [pool.draw(0) for _ in range(5)]
    assert first == [3499211612, 581869302, 3890346734, 3586334585, 545404204]
    for _ in range(10000 - 5 - 1):
        pool.draw(0)
    assert pool.draw(0) == 4123659995


def test_survey_known_answers():
    """Numbers printed by the reference binary during the survey (SURVEY.md 8c)."""
    from oracle.oracle_lib import OraclePool

    p = OraclePool("CartPole", 2, seed=7, max_episode_steps=500)
    obs = p.reset()["obs"]
    np.testing.assert_array_equal(
        obs[0], np.array([-0.0272660926, -0.0181027781, 0.0478222892, -0.00444150902],
                         dtype=np.float32))
    p = OraclePool("FrozenLake", 1, seed=7, max_episode_steps=100, iopt=4)
    p.reset()
    seq = []
    for _ in range(12):
        s = p.step(np.ones(1, np.int32))
        seq.append((int(s["obs"][0]), float(s["reward"][0]), int(s["done"][0])))
    assert seq == [(0, 0, 0), (0, 0, 0), (1, 0, 0), (0, 0, 0), (4, 0, 0), (5, 0, 1),
                   (0, 0, 0), (1, 0, 0), (5, 0, 1), (0, 0, 0), (1, 0, 0), (0, 0, 0)]
    p = OraclePool("Catch", 4, seed=7)
    assert p.reset()["obs"][:, 0, :].argmax(1).tolist() == [0, 4, 0, 3]


def test_oracle_matches_compiled_reference_when_present():
    """The restatement against the reference's own AsyncEnvPool on a fresh seed/action
    stream: every batch must match, bit for bit, the digest of the batch the reference
    returned (golden/digests/ref_stream.npz, recorded by golden/make_golden.py)."""
    from oracle.oracle_lib import OraclePool
    from helpers import GOLDEN, REGISTERED, batch_digest, random_actions

    rec = np.load(os.path.join(GOLDEN, "digests", "ref_stream.npz"))
    meta = json.loads(str(rec["meta"]))
    N, T = meta["num_envs"], meta["steps"]
    rng = np.random.default_rng(meta["action_seed"])
    for task, (ms, iopt) in REGISTERED.items():
        acts = np.stack([random_actions(task, rng, (N,)) for _ in range(T)])
        assert batch_digest({"actions": acts}) == int(rec[task + ":actions"][0]), \
            f"{task}: the action stream is not the recorded one"
        keys = meta["keys"][task]
        o = OraclePool(task, N, seed=meta["seed"], max_episode_steps=ms, iopt=iopt)
        got = [o.reset()] + [o.step(a) for a in acts]
        got = [batch_digest({k: b[k] for k in keys}) for b in got]
        bad = np.flatnonzero(np.array(got, dtype=np.uint64) != rec[task])
        assert bad.size == 0, f"{task}: first differing batch {bad[0]} (0 = reset)"
