"""CPU: this repo's Python layer against a record of the REFERENCE's own Python layer --
envpool/python/{api,env_spec,dm_envpool,gymnasium_envpool,envpool,data}.py,
envpool/registration.py and the family packages' __init__/registration, imported unmodified
and run on top of THIS repo's pybind11 modules (tests/ref_layer_check.py wrote the record,
tests/golden/reference_python_layer.json).  That is the drop-in boundary of SURVEY.md 8(b)
seen from the reference's side (INTEGRATION.md section 1): for every task id the reference's
make_spec() over our modules gave the config, key lists and spaces that ours gives."""
import json
import os

import numpy as np
import pytest

from helpers import GOLDEN, jsonable, space_desc


@pytest.fixture(scope="module")
def report():
    with open(os.path.join(GOLDEN, "reference_python_layer.json")) as f:
        return json.load(f)


def _same_space(ref, ours):
    """Equal shape, bounds (where the reference's space has them) and number of values."""
    return (ref["shape"] == ours["shape"] and ref.get("n") == ours.get("n")
            and all(ref[k] == ours[k] for k in ("low", "high") if k in ref))


def test_reference_make_spec_over_our_modules_equals_ours(report, engine_built):
    import envpool_b200

    envpool_b200._ensure_registered()
    from envpool_b200.registration import registry

    ours = sorted(t for t, (path, _, _) in registry.specs.items()
                  if path.endswith(("classic_control", "toy_text", "mujoco.gym")))
    assert ours == sorted(report["tasks"])
    assert len(ours) >= 24
    for v in ("v3", "v4", "v5"):   # via the reference's mujoco/gym registration.py
        hc = report["tasks"][f"HalfCheetah-{v}"]
        assert hc["obs_space"]["shape"] == [17] and hc["dm_action"]["shape"] == [6]
        assert hc["reward_threshold"] == 4800.0
    for task in ours:
        ref = report["tasks"][task]
        assert task in report["registry"], task
        spec = envpool_b200.make_spec(task, num_envs=3, seed=11)
        config = spec.config._asdict()
        config.pop("base_path", None)   # the install directory of the registering package
        assert json.loads(json.dumps(jsonable(config))) == ref["config"], task
        assert list(spec._state_keys) == ref["state_keys"], task
        assert list(spec._action_keys) == ref["action_keys"], task
        assert _same_space(ref["obs_space"], space_desc(spec.observation_space)), task
        assert _same_space(ref["act_space"], space_desc(spec.action_space)), task
        assert list(spec.observation_spec()._fields) == ref["dm_obs_fields"], task
        assert list(spec.action_spec().shape or ()) == ref["dm_action"]["shape"], task
        assert spec.reward_threshold == ref["reward_threshold"], task
    cp = report["tasks"]["CartPole-v1"]
    assert cp["obs_space"]["shape"] == [4] and cp["act_space"]["n"] == 2
    assert cp["reward_threshold"] == 475.0
    assert cp["dm_obs_fields"] == ["env_id", "players", "obs"]
    assert report["tasks"]["Acrobot-v1"]["dm_obs_fields"] == ["env_id", "players", "obs", "state"]
    assert report["tasks"]["Pendulum-v1"]["act_space"]["type"] == "Box"


def test_reference_dm_fold_over_our_key_order(report, engine_built):
    """Our dm fold of a batch in our column order gives the TimeStep the reference's gave."""
    import envpool_b200.classic_control as cc

    f = report["dm_fold"]
    assert f["obs_is_same_object"] and f["players_env_id"] == [0, 1, 2]
    assert f["last"] == [False, True, True]
    n = 3
    ids = np.arange(n, dtype=np.int32)
    done, trunc = np.array([0, 1, 1], bool), np.array([0, 0, 1], bool)
    obs = np.arange(4 * n, dtype=np.float32).reshape(n, 4)
    cols = [ids, ids, np.full(n, 7, np.int32), done, np.ones(n, np.float32),
            (~done).astype(np.float32), np.array([1, 2, 2], np.int32), trunc, obs]
    ts = cc.CartPoleDMEnvPool._to(None, cols, False, True)
    assert (ts.observation.obs is obs) == f["obs_is_same_object"]
    assert ts.observation.players.env_id.tolist() == f["players_env_id"]
    assert ts.last().tolist() == f["last"]
    assert ts.reward.tolist() == f["reward"]
    assert [int(x) for x in ts.step_type] == f["step_type"]
