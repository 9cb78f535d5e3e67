"""CPU-only checks (no compute on a GPU): the C-ABI library loads and exports exactly what include/b200env.h declares,
host-side logic (table packing, option parsing, registration), and the no-fallback rule."""
import os
import re

import numpy as np
import pytest

from conftest import ROOT, have_cuda

import gymnasium_b200
from gymnasium_b200 import _lib
from gymnasium_b200.envs.cartpole import _parse_reset_bounds
from gymnasium_b200.envs.frozen_lake import MAPS, pack_transition_table
from oracle.frozenlake import build_table


def header_symbols():
    text = open(os.path.join(ROOT, "include", "b200env.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(b2e_[a-z0-9_]+)\s*\(", text)))


def test_library_loads_and_exports_every_declared_symbol():
    lib = _lib.load()
    declared = header_symbols()
    assert declared, "no symbols parsed from include/b200env.h"
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/b200env.h but not exported by libb200env.so"
    assert sorted(_lib.SIGNATURES) == declared, "ctypes SIGNATURES and the header disagree"
    assert lib.b2e_version() == 1


def test_struct_layouts_match_header():
    import ctypes as C

    assert C.sizeof(_lib.Batch) == 48
    assert C.sizeof(_lib.CartPoleCfg) == 24
    assert C.sizeof(_lib.FrozenLakeCfg) == 8 + 16 + 72
    assert C.sizeof(_lib.LunarLanderCfg) == 32 and C.sizeof(_lib.LunarLanderState) == 88
    assert _lib.load().b2e_lunarlander_state_words() == 12 * 16
    assert C.sizeof(_lib.HumanoidCfg) == 80 and C.sizeof(_lib.HumanoidState) == 72
    assert C.sizeof(_lib.MjPlanarCfg) == 88 and C.sizeof(_lib.PipeSlot) == 88


def test_argument_errors_do_not_need_a_gpu():
    lib = _lib.load()
    assert lib.b2e_rng_seed(None, 0, None, None, None, None) == -1
    assert b"NULL" in lib.b2e_last_error()
    b = _lib.Batch(n=-3)
    import ctypes as C

    assert lib.b2e_cartpole_step(C.byref(b), None, None, None, None, None, None, None, None, None, None, None) == -1
    assert b"n=-3" in lib.b2e_last_error()


@pytest.mark.skipif(have_cuda(), reason="checks the no-GPU behaviour")
def test_no_cpu_fallback():
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        gymnasium_b200.make_vec("CartPole-v1", num_envs=4)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        gymnasium_b200.make_vec("FrozenLake-v1", num_envs=4, map_name="8x8")


@pytest.mark.parametrize("map_name", ["4x4", "8x8"])
@pytest.mark.parametrize("slippery", [True, False])
def test_packed_table_equals_reference_P(map_name, slippery):
    sched = (1, 0, 0) if slippery else (5, -2, 3)
    table, cum3, p3, isd_cum, nS, shape = pack_transition_table(MAPS[map_name], slippery, 1.0 / 3.0, sched)
    P, isd = build_table(MAPS[map_name], slippery, 1.0 / 3.0, sched)
    table = table.reshape(nS, 4, 3)
    np.testing.assert_array_equal(np.cumsum(isd), isd_cum)
    rewards = list(sched) + [0]
    for s in range(nS):
        for a in range(4):
            tr = P[s][a]
            n_out = int(table[s, a, 0] >> 20)
            assert n_out == len(tr)
            for k, (p, s2, r, d) in enumerate(tr):
                e = int(table[s, a, k])
                assert (e & 0xFFFF) == s2 and bool((e >> 16) & 1) == d and rewards[(e >> 17) & 3] == r
                assert (p3[k] if n_out == 3 else 1.0) == p
    assert list(cum3) == list(np.cumsum([t[0] for t in P[0][1]])) if slippery else True


def test_reset_bounds_parsing():
    assert _parse_reset_bounds(None, -0.05, 0.05) == (-0.05, 0.05)
    assert _parse_reset_bounds({"low": -0.1, "high": 0.1}, -0.05, 0.05) == (-0.1, 0.1)
    assert _parse_reset_bounds({"high": 0.2}, -0.05, 0.05) == (-0.05, 0.2)
    with pytest.raises(ValueError):
        _parse_reset_bounds({"low": 0.2, "high": 0.1}, -0.05, 0.05)
    with pytest.raises(ValueError):
        _parse_reset_bounds({"low": "abc"}, -0.05, 0.05)


def test_registry_ids():
    assert set(gymnasium_b200.registration.ENVS) >= {"CartPole-v1", "FrozenLake-v1", "FrozenLake8x8-v1"}
    with pytest.raises(KeyError):
        gymnasium_b200.make_vec("NoSuchEnv-v0", 2)


def test_humanoid_compiled_model_matches_oracle_compile():
    """The product's own compile of humanoid.xml (host side of csrc/humanoid.cu) against the oracle's independent one:
    inertia-from-geoms, meaninertia and the invweight0 constants, bit for bit."""
    from oracle.humanoid import OracleHumanoid

    lib = _lib.load()
    mass = np.zeros(14); misc = np.zeros(8); inv = np.zeros(14 * 2 + 23)
    assert lib.b2e_humanoid_model_info(mass.ctypes.data, misc.ctypes.data, inv.ctypes.data) == 0
    om, omisc, oinv = OracleHumanoid(1).model_info()
    np.testing.assert_array_equal(mass, om)
    np.testing.assert_array_equal(misc[:3], omisc[:3])
    np.testing.assert_array_equal(inv, oinv)
    known = [0, 8.90746237, 2.26194671, 6.61619413, 4.75175093, 2.75569617, 1.76714587, 4.75175093, 2.75569617,
             1.76714587, 1.66108048, 1.22954019, 1.66108048, 1.22954019]  # mjModel.body_mass of the stock humanoid.xml
    np.testing.assert_allclose(mass, known, rtol=2e-8)


def test_inverted_pendulum_compiled_model_matches_oracle_compile():
    """Host side of csrc/inverted_pendulum.cu (capsule-from-fromto, slide range in metres, ctrlrange 3) against the oracle's
    compile of inverted_pendulum.xml, bit for bit, and against the closed-form capsule masses."""
    from oracle.inverted_pendulum import OracleInvertedPendulum

    lib = _lib.load()
    mass = np.zeros(3); misc = np.zeros(8); inv = np.zeros(3 * 2 + 2)
    assert lib.b2e_inverted_pendulum_model_info(mass.ctypes.data, misc.ctypes.data, inv.ctypes.data) == 0
    om, omisc, oinv = OracleInvertedPendulum(1).model_info()
    np.testing.assert_array_equal(mass, om)
    np.testing.assert_array_equal(misc[:3], omisc[:3])
    np.testing.assert_array_equal(inv, oinv)
    np.testing.assert_allclose(mass, [0.0, 10.471975511965978, 5.018591641363305], rtol=1e-13)  # rho (4/3 pi r^3 + pi r^2 h)


def test_half_cheetah_compiled_model_matches_oracle_compile():
    """Host side of csrc/half_cheetah.cu (axisangle / fromto capsules, settotalmass, radian ranges, per-joint springs and
    per-actuator gears) against the oracle's compile of half_cheetah.xml, bit for bit."""
    from oracle.half_cheetah import OracleHalfCheetah

    lib = _lib.load()
    mass = np.zeros(8); misc = np.zeros(8); inv = np.zeros(8 * 2 + 9)
    assert lib.b2e_half_cheetah_model_info(mass.ctypes.data, misc.ctypes.data, inv.ctypes.data) == 0
    om, omisc, oinv = OracleHalfCheetah(1).model_info()
    np.testing.assert_array_equal(mass, om)
    np.testing.assert_array_equal(misc[:3], omisc[:3])
    np.testing.assert_array_equal(inv, oinv)
    assert abs(mass.sum() - 14.0) < 1e-12


def test_packed_cliffwalking_and_taxi_tables_equal_reference_P():
    from gymnasium_b200.envs.toy_text import pack_cliffwalking, pack_taxi
    from oracle.toy_text import build_cliff, build_taxi, taxi_action_mask

    def check(table, cum3, p3, isd_cum, nS, nA, rewards, P, isd):
        table = table.reshape(nS, nA, 3)
        np.testing.assert_array_equal(np.cumsum(isd), isd_cum)
        for s in range(nS):
            for a in range(nA):
                tr = P[s][a]
                assert int(table[s, a, 0] >> 20) == len(tr)
                for k, (p, s2, r, d) in enumerate(tr):
                    e = int(table[s, a, k])
                    assert (e & 0xFFFF) == s2 and bool((e >> 16) & 1) == d and rewards[(e >> 17) & 3] == r
                    assert (p3[k] if len(tr) == 3 else 1.0) == p
                if len(tr) == 3:
                    assert list(cum3) == list(np.cumsum([t[0] for t in tr]))

    for slip in (False, True):
        t, c3, p3, ic, nS, nA, rw = pack_cliffwalking(slip)
        P, isd = build_cliff(slip)
        check(t, c3, p3, ic, nS, nA, rw, P, isd)
    for rainy in (False, True):  # the oracle's P is pinned to the live reference by tests/golden/taxi_*.npz
        t, c3, p3, ic, nS, nA, rw, mask = pack_taxi(rainy)
        P, isd = build_taxi(rainy)
        check(t, c3, p3, ic, nS, nA, rw, P, isd)
    for s in range(500):
        np.testing.assert_array_equal(mask[s], taxi_action_mask(s))
