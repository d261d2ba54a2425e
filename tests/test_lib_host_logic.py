"""CPU tests of the product library's host-side logic (no GPU needed).

fb_env_logic.cuh is compiled for host and device; the fb_debug_host_* hooks run the host
build of exactly the functions the kernels call (env_step, make_draw_list, obs_row_mask,
exact_obs_bit) on tables derived by fb_assets.cu.  They are pinned here against the golden
fixtures of the real reference and against the oracle.
"""
import ctypes as C
import os
import re

import numpy as np
import pytest

from dqnflappybird_b200 import _lib
from dqnflappybird_b200.assets import load_blob
from oracle import flappy_oracle as fo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def L():
    lib = _lib.lib()
    blob = load_blob()
    assert lib.fb_debug_assets_load_host(blob, len(blob)) == 0, lib.fb_last_error()
    return lib


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "flappy_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    names = set(re.findall(r"\b(fb_[a-z0-9_]+)\s*\(", hdr))
    assert len(names) >= 20
    lib = C.CDLL(_lib.SO_PATH)
    for n in sorted(names):
        assert hasattr(lib, n), f"{n} declared in include/flappy_b200.h but not exported"
    assert set(_lib.declared_symbols()) <= names


def test_resize_tables_equal_oracle(L):
    t = np.zeros((6, 80), np.int32)
    assert L.fb_resize_tables(t.ctypes.data) == 0
    np.testing.assert_array_equal(t, fo.resize_tables())


def _host_obs(L, st, mode):
    out = np.empty((80, 80), np.uint8)
    rc = L.fb_debug_host_obs(st.ctypes.data, mode, out.ctypes.data)
    assert rc == 0, L.fb_last_error()
    return out


def test_host_step_and_obs_match_reference_trajectories(L, golden_dir):
    g = np.load(os.path.join(golden_dir, "ref_env_trajectories.npz"))
    n_mixed = 0
    for ti in range(int(g["n_traj"])):
        gaps = np.ascontiguousarray(g[f"t{ti}_gaps"])
        acts = g[f"t{ti}_actions"]
        st = np.zeros(16, np.int32)
        assert L.fb_debug_host_reset(st.ctypes.data, gaps.ctypes.data, len(gaps), 0, 0) == 0
        r, t, s = C.c_float(), C.c_uint8(), C.c_int32()
        for k in range(len(acts)):
            rc = L.fb_debug_host_step(st.ctypes.data, int(acts[k]), gaps.ctypes.data, len(gaps), 0, 0,
                                      C.byref(r), C.byref(t), C.byref(s))
            assert rc == 0
            assert r.value == g[f"t{ti}_reward"][k] and t.value == g[f"t{ti}_terminal"][k] and s.value == g[f"t{ti}_score"][k], (ti, k)
            ref = g[f"t{ti}_state"][k].copy(); ref[4] = st[4]
            np.testing.assert_array_equal(st, ref, err_msg=f"traj {ti} step {k}")
            mixed = L.fb_debug_host_mixed(st.ctypes.data)
            n_mixed += mixed
            if k % 3 == 0 or mixed or t.value:
                want = np.unpackbits(g[f"t{ti}_obsbits"][k]).reshape(80, 80) * 255
                np.testing.assert_array_equal(_host_obs(L, st, 0), want, err_msg=f"table obs traj {ti} step {k}")
                if k % 30 == 0 or mixed:
                    np.testing.assert_array_equal(_host_obs(L, st, 1), want, err_msg=f"exact obs traj {ti} step {k}")
    assert n_mixed > 50          # the per-pixel fix-up path really is exercised


def _mk_state(y=244, vel=0, pidx=0, basex=0, pipes=((288, 0), (432, 0))):
    st = np.zeros(16, np.int32)
    st[0], st[1], st[2], st[5], st[7] = y, vel, pidx, basex, len(pipes)
    for k, (x, gp) in enumerate(pipes):
        st[8 + k], st[11 + k] = x, gp
    return st


def _oracle_obs(states):
    env = fo.OracleEnvs(len(states), gaps=np.zeros((len(states), 1), np.uint8))
    env.import_state(np.stack(states))
    return env.obs_all()


def test_bird_only_observations_exhaustive(L):
    """every (playery, playerIndex) with both pipes off-screen: table path == oracle"""
    states = [_mk_state(y=y, pidx=p, pipes=((420, 0), (432, 0))) for p in range(3) for y in range(380)]
    want = _oracle_obs(states)
    for st, w in zip(states, want):
        np.testing.assert_array_equal(_host_obs(L, st, 0), w, err_msg=str(st[:3]))


def test_pipe_only_observations_exhaustive(L):
    """every reachable (pipe x, gap) with the bird far from the pipe: table path == oracle"""
    states = []
    for gp in range(8):
        for x in range(-56, 300, 2):
            # park the bird where it cannot share a tap footprint with this pipe
            y = 150 + 10 * gp if -60 < x - 57 < 60 else 244
            states.append(_mk_state(y=y, pipes=((x, gp), (min(x + 144, 440), (gp + 3) % 8))))
    want = _oracle_obs(states)
    for st, w in zip(states, want):
        got = _host_obs(L, st, 0)
        np.testing.assert_array_equal(got, w, err_msg=str(st))


def test_random_states_table_and_exact_paths(L):
    rng = np.random.default_rng(3)
    states = []
    for _ in range(1500):
        x0 = int(rng.integers(-52, 140)) & ~1
        gp = int(rng.integers(0, 8))
        gapY = 100 + 10 * gp
        # inside the gap (no collision), often hugging an edge so that bird and pipe share taps
        y = int(np.clip(gapY + rng.choice([0, 1, 2, 3, 30, 73, 74, 75, 76]) + rng.integers(0, 2), 0, 379))
        states.append(_mk_state(y=y, pidx=int(rng.integers(0, 3)), basex=-int(rng.integers(0, 12)) * 4,
                                pipes=((x0, gp), (x0 + 144, int(rng.integers(0, 8))))))
    want = _oracle_obs(states)
    mixed = 0
    for st, w in zip(states, want):
        mixed += L.fb_debug_host_mixed(st.ctypes.data)
        np.testing.assert_array_equal(_host_obs(L, st, 0), w, err_msg=str(st))
        np.testing.assert_array_equal(_host_obs(L, st, 1), w, err_msg=str(st))
    assert mixed > 100


def test_philox_gap_stream_matches_oracle(L):
    """non-replay mode: gap draws from Philox(seed, env) with CPython's randint rule"""
    for env_id in (0, 1, 77, 2**33 + 5):
        seed = 42
        st = np.zeros(16, np.int32)
        assert L.fb_debug_host_reset(st.ctypes.data, None, 0, seed, env_id) == 0
        env = fo.OracleEnvs(1, seed=seed, first_env_id=env_id)
        np.testing.assert_array_equal(st, env.export_state()[0])
        rng = np.random.default_rng(env_id % 1000)
        r, t, s = C.c_float(), C.c_uint8(), C.c_int32()
        for k in range(600):
            a = int(rng.random() < 0.1)
            assert L.fb_debug_host_step(st.ctypes.data, a, None, 0, seed, env_id, C.byref(r), C.byref(t), C.byref(s)) == 0
            _, rr, tt, ss = env.step(np.array([a], np.uint8), want_obs=False)
            assert (r.value, t.value, s.value) == (rr[0], tt[0], ss[0])
            np.testing.assert_array_equal(st, env.export_state()[0])


def test_invalid_action_is_rejected(L):
    st = _mk_state()
    r, t, s = C.c_float(), C.c_uint8(), C.c_int32()
    assert L.fb_debug_host_step(st.ctypes.data, 2, None, 0, 0, 0, C.byref(r), C.byref(t), C.byref(s)) == -4
    assert b"Multiple input actions" in L.fb_last_error()


def _check_layout(mirror, out, n):
    fields = mirror._fields_
    assert n == 1 + len(fields)
    assert out[0] == C.sizeof(mirror)
    for k, (name, _) in enumerate(fields):
        assert out[1 + k] == getattr(mirror, name).offset, name


def test_step_sampling_struct_matches_the_c_layout():
    """the ctypes mirror of fb_step_sampling (the sampling descriptor handed to fb_qnet_step) against the compiled struct"""
    out = (C.c_int32 * 32)()
    _check_layout(_lib.StepSampling, out, _lib.lib().fb_debug_step_sampling_layout(out, 32))


def test_qnet_step_args_struct_matches_the_c_layout():
    """the ctypes mirror of fb_qnet_step_args (the descriptor of fb_qnet_step) against the compiled struct"""
    out = (C.c_int32 * 64)()
    _check_layout(_lib.QnetStepArgs, out, _lib.lib().fb_debug_struct_layout(1, out, 64))
