"""Record what the REFERENCE's own Python layer (envpool/python/*.py, registration.py and the
family packages, imported unmodified from a reference checkout) makes of this repo's pybind11
extension modules, as tests/golden/reference_python_layer.json -- the record that
tests/test_reference_python_layer.py compares this repo's own layer against:

    python tests/ref_layer_check.py <reference checkout>

optree / dm_env / gymnasium need not be installed: tests/refstubs holds stand-ins for the few
names that layer uses.  What the layer consumes is the drop-in boundary of SURVEY.md 8(b): its
`py_env()` metaclasses, `EnvSpec` mixin, registry and `make_spec()` read
`_config_keys / _default_config_values / _state_keys / _action_keys / _state_spec /
_action_spec` and the tuple constructor of OUR `_XxxEnvSpec` / `_XxxEnvPool` classes exactly
as they read the Bazel-built ones (INTEGRATION.md section 1)."""
import importlib
import json
import os
import sys

sys.dont_write_bytecode = True  # the reference checkout is left untouched
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN = os.path.join(HERE, "golden", "reference_python_layer.json")

FAMILIES = {
    # reference package            compiled module it imports            ours
    "envpool.classic_control": ("classic_control_envpool",
                                "envpool_b200.classic_control.classic_control_envpool"),
    "envpool.toy_text": ("toy_text_envpool", "envpool_b200.toy_text.toy_text_envpool"),
}


def main(ref):
    import numpy as np

    from helpers import jsonable, space_desc

    sys.path.insert(0, ROOT)
    import envpool_b200  # noqa: F401  (ours, real spaces stand-ins of its own)

    envpool_b200._ensure_registered()
    from envpool_b200.registration import registry as our_registry

    sys.path.insert(0, os.path.join(HERE, "refstubs"))
    sys.path.insert(0, ref)
    for pkg, (mod, ours) in FAMILIES.items():
        sys.modules[f"{pkg}.{mod}"] = importlib.import_module(ours)
    # envpool/entry.py imports EVERY family's registration, and each family package imports
    # its Bazel-built extension (atari_envpool, box2d_envpool, ...), none of which exists
    # here: register only the two families on the accelerated path.
    import types

    sys.modules["envpool.entry"] = types.ModuleType("envpool.entry")
    import envpool  # the reference package, from the checkout
    import envpool.classic_control.registration  # noqa: F401
    import envpool.toy_text.registration  # noqa: F401

    # mujoco/gym: the reference's family package imports ALL eleven MuJoCo tasks from one
    # extension module, of which only HalfCheetah exists here.  Stand in for the package
    # object only (its registration.py and the rest of the layer stay the reference's): the
    # three HalfCheetah classes are built by the REFERENCE's py_env() over our pybind pair.
    from envpool.python.api import py_env as ref_py_env

    ours_mj = importlib.import_module("envpool_b200.mujoco.mujoco_gym_envpool")
    pkg = types.ModuleType("envpool.mujoco.gym")
    pkg.__path__ = [os.path.join(ref, "envpool", "mujoco", "gym")]
    (pkg.GymHalfCheetahEnvSpec, pkg.GymHalfCheetahDMEnvPool,
     pkg.GymHalfCheetahGymnasiumEnvPool) = ref_py_env(ours_mj._GymHalfCheetahEnvSpec,
                                                      ours_mj._GymHalfCheetahEnvPool)
    import envpool.mujoco  # noqa: F401  (plain namespace package in the reference)

    sys.modules["envpool.mujoco.gym"] = pkg
    import envpool.mujoco.gym.registration  # noqa: F401

    assert os.path.abspath(envpool.__file__).startswith(os.path.abspath(ref))
    report = {"reference": "sail-sg/envpool@9cbcd26",
              "registry": sorted(envpool.list_all_envs()), "tasks": {}}
    for task, (import_path, _, _) in sorted(our_registry.specs.items()):
        if not import_path.endswith(("classic_control", "toy_text", "mujoco.gym")):
            continue
        rs = envpool.make_spec(task, num_envs=3, seed=11)
        rc = rs.config._asdict()
        rc.pop("base_path", None)   # the install directory of the registering package
        report["tasks"][task] = {
            "config": jsonable(rc), "state_keys": list(rs._state_keys),
            "action_keys": list(rs._action_keys),
            "obs_space": space_desc(rs.observation_space),
            "act_space": space_desc(rs.action_space),
            "dm_obs_fields": list(rs.observation_spec()._fields),
            "dm_action": space_desc(rs.action_spec()),
            "reward_threshold": rs.reward_threshold}

    # the reference's dm fold over a batch in OUR column order
    import envpool.classic_control as rcc

    n = 3
    ids = np.arange(n, dtype=np.int32)
    done, trunc = np.array([0, 1, 1], bool), np.array([0, 0, 1], bool)
    obs = np.arange(4 * n, dtype=np.float32).reshape(n, 4)
    cols = [ids, ids, np.full(n, 7, np.int32), done, np.ones(n, np.float32),
            (~done).astype(np.float32), np.array([1, 2, 2], np.int32), trunc, obs]
    ts = rcc.CartPoleDMEnvPool._to(None, cols, False, True)
    report["dm_fold"] = {
        "obs_is_same_object": ts.observation.obs is obs,
        "players_env_id": ts.observation.players.env_id.tolist(),
        "last": ts.last().tolist(), "reward": ts.reward.tolist(),
        "step_type": [int(x) for x in ts.step_type],
    }
    with open(GOLDEN, "w") as f:
        json.dump(report, f, indent=1, sort_keys=True)
        f.write("\n")


if __name__ == "__main__":
    main(sys.argv[1])
