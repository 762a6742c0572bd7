"""Decision boundaries of the path (SURVEY.md section 4, item 3): envs that sit EXACTLY on a threshold - gate 0 / 1,
|cmd| == 0.1, |F| == 1 N and 100 N, +-inf ray hits, the step before / at the time-out, a root position on the terrain
bound, timers equal to step_dt / 0.5 s, joints on their soft limits - evaluated by the oracle and by the reference's
own functions (stored in tests/golden/reference_pins.npz): the oracle must take the same side of every comparison.
The GPU counterpart is tests/test_gpu_edge_cases.py."""

import pytest
import torch

import helpers as H
from oracle import mdp_port as port


def test_edge_state_hits_the_boundaries_it_claims():
    cfg, spec = H.make_spec("go2_rough")
    st = H.make_edge_case_state(spec)
    out = H.oracle_step(spec, st)
    d = port.Derived(st, spec)
    gate = d.gate() if callable(d.gate) else d.gate
    assert gate[0] == 1.0 and gate[1] == 0.0 and abs(float(gate[2])) < 1e-6     # upright / inverted / on its side
    assert not out["truncated"][10] and out["truncated"][11]                 # 999 vs 1000 steps
    assert not out["truncated"][12] and out["truncated"][13]                 # on the bound vs just outside
    assert not out["terminated"][:17].any()                                  # Go2 has no illegal-contact term
    crit = out["obs_critic"]
    assert (crit[7, -187:] == -1.0).all() and (crit[8, -187:] == 1.0).all()   # +-inf ray hits clip to -+1
    assert torch.isfinite(crit).all() and torch.isfinite(out["obs_policy"]).all() and torch.isfinite(out["reward"]).all()
    names = [t.name for t in spec.rewards]
    step = out["step_reward"]
    # |F| == 1.0 exactly is not an undesired contact; |F| == 100 adds nothing to contact_forces
    assert step[5, names.index("undesired_contacts")] == 0.0
    assert step[5, names.index("contact_forces")] == 0.0
    assert step[15, names.index("joint_pos_limits")] == 0.0 and step[16, names.index("joint_pos_limits")] == 0.0


@pytest.mark.parametrize("key", ["go2_rough", "a1_flat"])
def test_oracle_takes_the_reference_side_of_every_threshold(key):
    cfg, spec = H.make_spec(key)
    st = H.make_edge_case_state(spec)
    pins = H.reference_pins()
    d = port.Derived(st, spec)
    checked = 0
    for t in spec.rewards:
        want = pins.get(f"edge/{key}/reward/{t.name}")
        if want is None:
            continue   # IsaacLab-owned: no reference source
        got = port.reward_term(t, st, spec, d)
        torch.testing.assert_close(got, want.float(), rtol=1e-6, atol=1e-6, msg=t.name)
        assert torch.equal(got[:17] == 0, want[:17] == 0), t.name           # exact zeros (masks, strict comparisons) agree
        checked += 1
    assert checked >= 12
    got_cmd = port.compute_command(spec, st, {"cmd_uniforms": st["cmd_uniforms"]})
    ref_cmd = {k.rsplit("/", 1)[1]: v for k, v in pins.items() if k.startswith(f"edge/{key}/command/")}
    assert len(ref_cmd) == 7
    for k, v in ref_cmd.items():
        assert torch.equal(got_cmd[k], v), k
