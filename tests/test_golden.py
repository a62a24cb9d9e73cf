"""The committed golden vectors (tests/golden/step_v2.npz, made by tests/golden/make_golden.py from the CPU oracle:
the reference itself cannot run here, DESIGN.md section 2) against the oracle, the host build of the kernel
arithmetic (CPU) and the CUDA kernels through the C-ABI (-m gpu)."""
import os

import numpy as np
import pytest

import golden_util as G
import oracle_lib as O
import parity_util as P

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "step_v2.npz")


@pytest.fixture(scope="module")
def gold():
    z = np.load(PATH)
    return {"z": z, "s0": G.unpack(z, "s0"), "s1": G.unpack(z, "s1"), "s2": G.unpack(z, "s2")}


def test_oracle_reproduces_the_golden_vectors_bit_exactly(gold):
    z, n = gold["z"], len(gold["s0"])
    ora = O.OracleVec(n, P.CONFIG, seed=0)
    ora.set_states(gold["s0"])
    for k, (act, obs, rew, done, goal, want) in enumerate((
            (z["act1"], z["s1_obs"], z["rew1"], z["done1"], z["goal1"], gold["s1"]),
            (z["act2"], z["s2_obs"], z["rew2"], z["done2"], z["goal2"], gold["s2"]))):
        o, r, d, g = ora.step(act, auto_reset=False)
        assert np.array_equal(o, obs) and np.array_equal(r, rew) and np.array_equal(d, done) and np.array_equal(g, goal), k
        for i, (a, b) in enumerate(zip(ora.get_states(), want)):
            for key in G.FIELDS_F:
                assert np.array_equal(a[key], b[key]), (k, i, key)
            assert a["steps"] == b["steps"] and a["score"] == b["score"] and a["cache"] == b["cache"], (k, i)


class _GoldenOracle:
    """The golden state after a step, behind the two calls parity_util.compare_all makes on an oracle."""

    def __init__(self, states):
        self._s = states

    def env(self, i):
        s = self._s[i]

        class _E:
            @staticmethod
            def get_state():
                return s
        return _E


def _check(sim_cls, gold):
    """Step 1 from the injected start states, step 2 from the golden state after step 1 (its arbiter cache, bias
    velocities and observation history included): each is an independent check against the file."""
    z, n = gold["z"], len(gold["s0"])
    for k, (first, act, obs, rew, done, goal, want) in enumerate((
            (gold["s0"], z["act1"], z["s1_obs"], z["rew1"], z["done1"], z["goal1"], gold["s1"]),
            (gold["s1"], z["act2"], z["s2_obs"], z["rew2"], z["done2"], z["goal2"], gold["s2"]))):
        sim = sim_cls(n, P.CONFIG, seed=0)
        sim.set_states(np.arange(n), [P.oracle_to_dev_state(s) for s in first])
        o_d, r_d, d_d, g_d = sim.step(act, auto_reset=False)
        assert np.array_equal(d_d, done), "done flags differ from the golden vectors"
        assert np.array_equal(g_d, goal), "goal flags differ from the golden vectors"
        worst, failing, cache_bad = P.compare_all(sim, _GoldenOracle(want), o_d, obs, r_d, rew, n)
        assert not cache_bad, f"arbiter cache / counters differ for envs {cache_bad[:10]}"
        P.record(f"golden/{getattr(sim_cls, '__name__', 'sim')}/step{k + 1}", P.summarize(failing, worst, n))
        assert len(failing) <= max(1, int(n * P.MAX_OVER_FRACTION)), f"{len(failing)} envs out of tolerance, e.g. {failing[:5]}; worst {worst}"
        assert max(worst.values()) < P.MAX_RATIO, worst


def test_host_build_of_the_kernel_arithmetic_matches_the_golden_vectors(gold):
    import hostsim_lib as H
    P.add_batch_api(H.HostSim)
    _check(H.HostSim, gold)


@pytest.mark.gpu
def test_kernels_match_the_golden_vectors(gold):
    from marl_soccer_b200.host_api import HostBufferSim

    def dev(n, config, seed=0):
        return HostBufferSim(n, config, seed=seed)
    _check(dev, gold)
