"""CPU: the gym layer (rl4rs_b200.env.base.RecEnvBase / build_spaces) over a fake simulator, held against the
reference's OWN RecEnvBase (rl4rs/env/base.py:178-273, run through oracle/ref_harness.py over the same fake simulator;
what it showed is stored in tests/golden/reference/expected.json by tests/golden/make_reference_golden.py)."""
import hashlib
import json
import os

import numpy as np
import pytest

from golden_util import REFERENCE_DIR
from rl4rs_b200.env.base import RecEnvBase, build_spaces

A, OBS = 284, 256
CONFIGS = {
    "plain": {},
    "rllib": {"support_rllib_mask": True},
    "conti": {"support_conti_env": True, "action_emb_size": 32},
    "raw": {"rawstate_as_obs": True},
    "raw_rllib": {"rawstate_as_obs": True, "support_rllib_mask": True},
}


class FakeSamples(object):
    def __init__(self, n, draw):
        self.user = [100 * draw + i for i in range(n)]
        self.offline_action = [7 + i for i in range(n)]
        self.offline_reward = [0.5 * (i + 1) for i in range(n)]

    def to_string(self):
        return "fake"


class FakeSim(object):
    """Duck-typed RecSimBase: list outputs like the reference's (slate.py:244-279), every call recorded."""
    obs_dim = OBS

    def __init__(self, config):
        self.config, self.calls, self.draws = config, [], 0

    def _obs(self, n):
        c = self.config
        if c.get("rawstate_as_obs", False):
            row = {"category_feature": [0] * 21, "dense_feature": [0.0] * 432, "sequence_feature": [[0] * 64, [0] * 64]}
        else:
            row = {"obs": [0.25] * OBS}
        if c.get("support_rllib_mask", False):
            return [dict(row, action_mask=[1] * A) for _ in range(n)]
        return [row if "obs" not in row else row["obs"] for _ in range(n)]

    def reset(self, reset_file=False):
        self.calls.append(("reset", reset_file))

    def seed(self, sd):
        self.calls.append(("seed", sd))

    def sample(self, n):
        self.draws += 1
        self.calls.append(("sample", n))
        return FakeSamples(n, self.draws), self._obs(n)

    def _step(self, samples, action, **kw):
        self.calls.append(("step", [int(a) for a in action], kw["step"]))
        n = self.config["batch_size"]
        return self._obs(n), [1.0 + i for i in range(n)], [0] * n, [{"k": i} for i in range(n)]


def space_sig(s):
    if hasattr(s, "spaces"):
        return {k: space_sig(v) for k, v in s.spaces.items()}
    if hasattr(s, "n"):
        return ("discrete", int(s.n))
    return ("box", float(s.low), float(s.high), tuple(int(x) for x in s.shape))


EXPECTED_SPACES = {
    "plain": (("box", -1e5, 1e5, (OBS,)), ("discrete", A)),
    "rllib": ({"action_mask": ("box", 0.0, 1.0, (A,)), "obs": ("box", -1e5, 1e5, (OBS,))}, ("discrete", A)),
    "conti": (("box", -1e5, 1e5, (OBS,)), ("box", -1.0, 1.0, (32,))),
    "raw": ({"category_feature": ("box", -1e6, 1e6, (21,)), "dense_feature": ("box", -1e6, 1e6, (432,)),
             "sequence_feature": ("box", -1e6, 1e6, (2, 64))}, ("discrete", A)),
    "raw_rllib": ({"action_mask": ("box", 0.0, 1.0, (A,)), "category_feature": ("box", -1e6, 1e6, (21,)),
                   "dense_feature": ("box", -1e6, 1e6, (432,)), "sequence_feature": ("box", -1e6, 1e6, (2, 64))},
                  ("discrete", A)),
}


def drive(env_cls, config):
    """The README loop + the accessors; returns everything a caller can observe."""
    sim = FakeSim(config)
    env = env_cls(sim)
    seen = {"spaces": (space_sig(env.observation_space), space_sig(env.action_space)),
            "after_init": list(sim.calls), "step0": env.cur_step}
    env.seed(5)
    seen["user"], seen["oa"], seen["orew"] = env.user_id, env.offline_action, env.offline_reward
    seen["state_is_obs"] = env.state == (env.obs[0] if config["batch_size"] == 1 else env.obs)
    act = env.offline_action
    r1 = env.step(act)
    r2 = env.step(np.array(act) if config["batch_size"] > 1 else act)
    seen["r1"], seen["r2"], seen["cur_step"] = list(r1), list(r2), env.cur_step
    seen["reset"] = env.reset(reset_file=True) == seen_state(env, config)
    seen["calls"], seen["cur_step_after_reset"] = list(sim.calls), env.cur_step
    return seen


def seen_state(env, config):
    return env.obs[0] if config["batch_size"] == 1 else env.obs


@pytest.mark.parametrize("name", sorted(CONFIGS))
@pytest.mark.parametrize("batch", [1, 3])
def test_env_layer_matches_reference_env_layer(name, batch):
    config = dict(CONFIGS[name], batch_size=batch, action_size=A)
    ours = drive(RecEnvBase, config)
    assert ours["spaces"] == EXPECTED_SPACES[name]
    # two draws while constructing (base.py:186-187,230; SURVEY Q19), then one per reset
    assert ours["after_init"] == [("reset", False), ("sample", batch)] * 2
    assert ours["calls"][-2:] == [("reset", True), ("sample", batch)] and ours["cur_step_after_reset"] == 0
    assert ours["cur_step"] == 2 and [c[2] for c in ours["calls"] if c[0] == "step"] == [0, 1]
    if batch == 1:
        assert ours["user"] == 200 and ours["oa"] == 7 and ours["orew"] == 0.5
        assert ours["r1"][1:] == [1.0, 0, {"k": 0}]
        assert [c[1] for c in ours["calls"] if c[0] == "step"] == [[7], [7]]        # a bare action is wrapped
    else:
        assert ours["user"] == [200, 201, 202] and ours["r1"][1] == [1.0, 2.0, 3.0]
    with open(os.path.join(REFERENCE_DIR, "expected.json")) as f:
        ref = json.load(f)["env_layer"]["%s/%d" % (name, batch)]
    assert seen_digest(ours) == ref, ours


def seen_digest(seen):
    """What drive() saw, as a digest of its JSON form (tuples become lists)."""
    return hashlib.sha256(json.dumps(seen, sort_keys=True).encode()).hexdigest()


def test_build_spaces_takes_the_widths_from_the_config():
    obs, act = build_spaces({"action_size": 50, "rawstate_as_obs": True, "category_feature_num": 5, "dense_feature_num": 9,
                             "seq_num": 3, "maxlen": 16}, 0)
    assert space_sig(obs) == {"category_feature": ("box", -1e6, 1e6, (5,)), "dense_feature": ("box", -1e6, 1e6, (9,)),
                              "sequence_feature": ("box", -1e6, 1e6, (3, 16))}
    assert space_sig(act) == ("discrete", 50)
    assert space_sig(build_spaces({"action_size": 50}, 3072)[0]) == ("box", -1e5, 1e5, (3072,))       # widedeep


def test_per_env_values_are_read_only():
    env = RecEnvBase(FakeSim({"batch_size": 2, "action_size": A}))
    with pytest.raises(AttributeError):
        env.user_id = [1, 2]
    assert RecEnvBase.user_id.__doc__.startswith("session ids")
