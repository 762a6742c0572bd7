"""Pin the oracle: every robot_lab-owned piece of oracle/mdp_port.py against the outputs of the reference's OWN
functions (the unmodified robot_lab files run through oracle/isaaclab_shim.py), stored in tests/golden/ by
tests/golden/make_golden.py. The reward, command and observation checks read the same fixtures as
test_oracle_golden.py (their seeded inputs stored beside the outputs); the reset check keeps its own inputs, whose
reference outputs are in reference_pins.npz."""

from pathlib import Path

import numpy as np
import pytest
import torch

import helpers as H
from oracle import mdp_port as port
from robot_lab_b200 import terrain as terrain_host

GOLDEN = Path(__file__).resolve().parent / "golden"


def _golden(name: str, group: str) -> dict:
    z = np.load(GOLDEN / f"{name}.npz")
    return {k[len(group) + 1:]: torch.from_numpy(z[k]) for k in z.files if k.startswith(group + "/")}


@pytest.mark.parametrize("key", ["a1_flat", "go2_rough", "g1_rough", "g1_rough_37", "catalogue"])
def test_reward_terms_match_reference_functions(key):
    cfg, spec = H.make_catalogue_spec() if key == "catalogue" else H.make_spec(key)
    name = "go2_catalogue" if key == "catalogue" else key
    st, ref = _golden(name, "in"), _golden(name, "reward")
    d = port.Derived(st, spec)
    checked = 0
    for t in spec.rewards:
        if t.name not in ref:
            continue  # IsaacLab-owned: no reference source, parity unpinned
        torch.testing.assert_close(port.reward_term(t, st, spec, d), ref[t.name].float(), rtol=1e-6, atol=1e-6, msg=t.name)
        checked += 1
    assert checked >= {"a1_flat": 12, "go2_rough": 16, "g1_rough": 8, "g1_rough_37": 8, "catalogue": 26}[key]


@pytest.mark.parametrize("key,terrain", [("go2_rough", "generator"), ("go2_flat", "plane"), ("g1_rough", "generator")])
def test_command_term_matches_reference_class(key, terrain):
    cfg, spec = H.make_spec(key)
    st, ref = _golden(key, "in"), _golden(key, "command")
    assert spec.layout.terrain.terrain_type == terrain
    # no "pits" sub-terrain in the in-scope terrains (V/mdp/utils.py:27-28): the reference's was_on_pit stays all False
    assert terrain_host.terrain_column_range(spec.layout.terrain, "pits") is None
    got = port.compute_command(spec, st, {"cmd_uniforms": st["cmd_uniforms"]})
    assert set(ref) == set(got) - {"was_on_pit"}
    for k, v in ref.items():
        assert torch.equal(got[k], v), k  # same op sequence -> bit-identical


def test_observation_functions_match_reference():
    from robot_lab_b200.spec import ObsGroupSpec, ObsTermSpec

    cfg, spec = H.make_spec("go2_rough")
    st, ref = _golden("go2_rough", "in"), _golden("go2_rough", "obs")
    wheel = ref["_wheel_ids"].tolist()
    terms = [ObsTermSpec("phase", "phase", 10, 2, p=[0.8, 0.0]),
             ObsTermSpec("jp", "joint_pos_rel_without_wheel", 9, spec.J, ids=list(range(spec.J)), zero_cols=wheel)]
    spec.obs[0] = ObsGroupSpec("policy", False, terms)
    got = port.compute_obs_group(spec, 0, st, {})
    torch.testing.assert_close(got[:, :2], ref["phase"].float(), rtol=1e-6, atol=1e-6)
    assert torch.equal(got[:, 2:], ref["joint_pos_rel_without_wheel"])


@pytest.mark.parametrize("key", ["go2_rough", "g1_rough"])
def test_reset_root_state_matches_reference_function(key):
    """oracle.reset_scene_state vs the unmodified reset_root_state_uniform (V/mdp/events.py:205-271) on a fake asset,
    same uniforms (the [IL] helpers quat_from_euler_xyz / quat_mul / sample_uniform are restated in both), with the
    default ranges and with the Go2 rough ones (GO2/rough_env_cfg.py:56-73); reference output in reference_pins.npz."""
    from robot_lab_b200.cfg import ResetStateCfg

    cfg, spec = H.make_spec(key)
    st, ids, org, u = H.reset_inputs(spec)
    n = st["root_pos_w"].shape[0]
    pins = H.reference_pins()
    for name, rc in (("default", ResetStateCfg()), ("go2_rough", ResetStateCfg.go2_rough())):
        got = port.reset_scene_state(spec, st, ids, rc, org, u)
        for k in ("root_pos_w", "root_quat_w", "root_lin_vel_w", "root_ang_vel_w"):
            torch.testing.assert_close(got[k][ids.long()], pins[f"reset/{key}/{name}/{k}"], rtol=0, atol=0, msg=k)
        untouched = torch.ones(n, dtype=torch.bool)
        untouched[ids.long()] = False
        assert torch.equal(got["root_pos_w"][untouched], st["root_pos_w"][untouched])
