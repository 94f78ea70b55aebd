"""Dev-container only: the C oracle in lockstep with the UNMODIFIED reference (imported from /root/reference,
injected position-indexed draws).  Skipped wherever the reference is absent (the GPU box)."""
import os
import sys

import pytest

import lockstep as ls
from oracle import refshim

pytestmark = [pytest.mark.needs_reference,
              pytest.mark.skipif(not refshim.reference_available(), reason="/root/reference not present")]


def _ref_backend():
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import make_golden
    return make_golden.RefBackend


@pytest.mark.parametrize("key,seed,rnd", [("cleanup5", 301, True), ("cleanup10_full", 302, False), ("cleanup3", 303, True),
                                          ("harvest5", 304, False), ("harvest10_full", 305, True)])
def test_oracle_lockstep_with_live_reference(key, seed, rnd):
    RefBackend = _ref_backend()
    kw = dict(teleport_every=6)
    ref = ls.run_trace(RefBackend(key, random_spawn=rnd), ls.schedule_for(key, seed, **kw), 90)
    ob = ls.OracleBackend(key, random_spawn=rnd)
    ora = ls.run_trace(ob, ls.schedule_for(key, seed, **kw), 90)
    ls.assert_traces_equal(ref, ora, key)
    assert int(ob.o.envs["error"][0]) == 0


def test_seeded_anchor_hashes_of_the_reference():
    """SURVEY Appendix C.3 anchor: unmodified reference, numpy/python RNG seeded with 0, 1000 steps of
    cleanup default5 -- proves the import shim runs the same reference the survey measured."""
    import hashlib
    import random
    import numpy as np
    env = refshim.make("cleanup", 5, "default5", 7)
    np.random.seed(0)
    random.seed(0)
    env.reset()
    acts = np.random.RandomState(123).randint(0, env.n_actions, size=(1000, 5))
    hA, hB = hashlib.sha256(), hashlib.sha256()
    for s in range(1000):
        r, term, info = env.step(acts[s])
        hA.update(env.world_map.astype("S1").tobytes())
        hA.update(env.get_agent_pos().astype(np.int16).tobytes())
        hA.update(r.astype(np.int8).tobytes())
        hA.update(info["clean_num"].astype(np.int8).tobytes())
        hB.update(np.uint8(np.stack(env.get_obs()) * 256).tobytes())
    assert hA.hexdigest()[:16] == "bd7111014f50657d" and hB.hexdigest()[:16] == "a45f7cb95a093744"
    assert env.rewards.tolist() == [-93.0, -114.0, -116.0, -86.0, -100.0]
    assert info["equality_metric"] == 0.9363457760314342


def test_fakebatch_has_the_update_semantics_of_the_reference_episodebatch():
    """The batched-runner tests check the runner through a stand-in EpisodeBatch (harness.FakeBatch); this pins the stand-in
    against the reference's EpisodeBatch.update (src/components/episode_buffer.py:87-116) on the CPU."""
    import numpy as np
    import torch
    refshim._import_registry()
    from components.episode_buffer import EpisodeBatch
    from harness import FakeBatch, _scheme
    n, A, H, W, N, B, T = 3, 9, 10, 10, 15, 2, 4
    fs = _scheme(n, A, H, W, N)
    scheme = {"state": {"vshape": (3, H, W)}, "obs": {"vshape": (3, N, N), "group": "agents"},
              "actions": {"vshape": (1,), "group": "agents", "dtype": torch.long},
              "avail_actions": {"vshape": (A,), "group": "agents", "dtype": torch.int}, "reward": {"vshape": (n,)},
              "terminated": {"vshape": (1,), "dtype": torch.uint8}, "clean_num": {"vshape": (n,)}, "apple_den": {"vshape": (n,)},
              "agent_pos": {"vshape": (n, 2)}, "agent_orientation": {"vshape": (n, 2)},
              "actions_inc": {"vshape": (n, 1), "group": "agents", "dtype": torch.long}}
    ref = EpisodeBatch(scheme, {"agents": n}, B, T, device="cpu")
    fake = FakeBatch(fs, B, T, "cpu")
    rs = np.random.RandomState(0)
    for t in range(T):
        data = {"state": torch.from_numpy(rs.randint(0, 256, (B, 3, H, W)).astype(np.uint8)).float() / 256,
                "obs": torch.from_numpy(rs.randint(0, 256, (B, n, 3, N, N)).astype(np.uint8)).float() / 256,
                "avail_actions": torch.ones(B, n, A, dtype=torch.int32), "agent_pos": torch.rand(B, n, 2),
                "agent_orientation": torch.rand(B, n, 2), "actions": torch.randint(0, A, (B, n, 1)),
                "reward": torch.randint(-1, 2, (B, n)).float(), "terminated": torch.zeros(B, 1, dtype=torch.uint8),
                "clean_num": torch.rand(B, n), "apple_den": torch.rand(B, n, dtype=torch.float64),
                "actions_inc": torch.randint(0, 3, (B, n, n, 1))}
        ref.update(data, ts=t)
        fake.update(data, ts=t)
    for k in fs:
        assert torch.equal(ref[k], fake[k]) and ref[k].dtype == fake[k].dtype, k
    assert torch.equal(ref["filled"], fake["filled"])


def test_hit_penalty_and_fire_cost_semantics_against_patched_reference():
    """north_star 'penalties': the reference hard-codes hit -= 0 / fire -= 1 (agent.py:184-190, 239-248).  Patching just
    those two constants in the live reference pins the oracle's fire_cost / hit_penalty parameters (who gets hit: the
    agent `agent_by_pos` returns, i.e. the last index on the cell)."""
    import numpy as np
    from homophily_marl_b200 import mapspec
    from oracle.oracle import OracleBatch
    RefBackend = _ref_backend()
    refshim._import_registry()
    import envs.ssd.agent as ag

    def hit(self, char):
        if char == 'F':
            self.reward_this_turn -= 5

    def fire_beam(self, char):
        if char == 'F':
            self.reward_this_turn -= 2

    saved = (ag.HarvestAgent.hit, ag.HarvestAgent.fire_beam)
    ag.HarvestAgent.hit, ag.HarvestAgent.fire_beam = hit, fire_beam
    try:
        key = "harvest10_full"
        ref = RefBackend(key, random_spawn=True)
        spec = mapspec.compile_map("harvest", "default10", 10, 7, 1000, obs_color="full", fire_cost=2, hit_penalty=5)
        ora = ls.OracleBackend(key, random_spawn=True)
        ora.o = OracleBatch.from_spec(spec, n_envs=1, random_spawn_point=True, spawn_rotation=None)
        sched_a = ls.schedule_for(key, 77, teleport_every=4)
        sched_b = ls.schedule_for(key, 77, teleport_every=4)
        sched_a.n_actions = sched_b.n_actions = 8
        a = ls.run_trace(ref, sched_a, 120)
        b = ls.run_trace(ora, sched_b, 120)
        ls.assert_traces_equal(a, b, "penalties")
        assert (a["reward"] <= -5).any() and (a["reward"] == -2).any()
    finally:
        ag.HarvestAgent.hit, ag.HarvestAgent.fire_beam = saved
