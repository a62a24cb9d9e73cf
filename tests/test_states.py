"""The msoc_env_state record formats without a GPU: the NumPy dtype and the torch field views against the ctypes struct
and the C header, and argument checks of msoc_save_states / msoc_load_states."""
import ctypes as C
import os
import subprocess

import numpy as np
import torch

from marl_soccer_b200 import _capi, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = [name for name, _ in _capi.MsocEnvState._fields_]


def test_dtype_matches_ctypes_and_c(tmp_path):
    dt = _capi.ENV_STATE_DTYPE
    assert dt.itemsize == _capi.ENV_STATE_BYTES == C.sizeof(_capi.MsocEnvState) == 808
    assert list(dt.names) == NAMES
    src = tmp_path / "off.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "msoc.h"\nint main(void){\n'
                   + "".join(f'printf("%zu %zu\\n", offsetof(msoc_env_state, {n}), '
                             f'sizeof(((msoc_env_state *)0)->{n}));\n' for n in NAMES)
                   + "return 0;}\n")
    exe = tmp_path / "off"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    c_layout = [tuple(int(v) for v in line.split())
                for line in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines()]
    for name, (off, size) in zip(NAMES, c_layout):
        field = getattr(_capi.MsocEnvState, name)
        assert (field.offset, field.size) == (off, size), name
        assert (dt.fields[name][1], dt.fields[name][0].itemsize) == (off, size), name


def random_states(n, seed=0):
    rng = np.random.default_rng(seed)
    raw = rng.integers(0, 256, (n, _capi.ENV_STATE_BYTES), dtype=np.uint8)
    return [_capi.MsocEnvState.from_buffer_copy(raw[i].tobytes()) for i in range(n)]


def as_tensor(states):
    return torch.from_numpy(np.frombuffer(b"".join(bytes(S) for S in states), np.uint8).reshape(len(states), -1).copy())


def test_state_fields_read_every_field():
    states = random_states(5)
    t = as_tensor(states)
    f = _capi.state_fields(t)
    assert set(f) == set(NAMES)
    assert f["pos"].shape == (5, 5, 2) and f["pos"].dtype == torch.float32
    assert f["hist_pos"].shape == (5, 2, 5, 2) and f["hist_ang"].shape == (5, 2, 4)
    assert f["seed"].shape == (5,) and f["seed"].dtype == torch.uint64
    assert f["cache_info"].shape == (5, 32) and f["cache_info"].dtype == torch.uint32
    arr = t.numpy().view(_capi.ENV_STATE_DTYPE).reshape(5)
    for name in NAMES:
        field = getattr(_capi.MsocEnvState, name)
        for i, S in enumerate(states):
            want = bytes(S)[field.offset:field.offset + field.size]  # random bytes: compared as bits (NaN payloads)
            assert f[name][i].numpy().tobytes() == want, (name, i)
            assert arr[name][i].tobytes() == want, (name, i)
    # values, on a state without NaNs
    S = _capi.MsocEnvState()
    S.pos[3][1], S.ang[2], S.steps, S.seed, S.cache_jt[31], S.hist_pos[1][4][0] = 2.5, -1.25, 77, 2**63 + 5, 0.75, 9.0
    g = _capi.state_fields(as_tensor([S]))
    assert g["pos"][0, 3, 1] == 2.5 and g["ang"][0, 2] == -1.25 and g["steps"][0] == 77
    assert int(g["seed"].numpy()[0]) == 2**63 + 5 and g["cache_jt"][0, 31] == 0.75 and g["hist_pos"][0, 1, 4, 0] == 9.0


def test_state_fields_write_the_right_bytes():
    states = random_states(4, seed=1)
    t = as_tensor(states)
    f = _capi.state_fields(t)
    f["pos"][2, 4] = torch.tensor([123.5, -7.25])
    f["seed"][1] = 2**62 + 11
    f["cache_count"][3] = 0
    f["hist_valid"][0] = 1
    f["hist_angvel"][2, 1, 3] = 0.5
    f["score"][1] = torch.tensor([3, -2], dtype=torch.int32)
    want = [_capi.MsocEnvState.from_buffer_copy(bytes(S)) for S in states]
    want[2].pos[4][0], want[2].pos[4][1] = 123.5, -7.25
    want[1].seed = 2**62 + 11
    want[3].cache_count = 0
    want[0].hist_valid = 1
    want[2].hist_angvel[1][3] = 0.5
    want[1].score[0], want[1].score[1] = 3, -2
    for i in range(4):
        assert t[i].numpy().tobytes() == bytes(want[i]), i


def test_state_fields_rejects_other_shapes():
    import pytest
    for bad in (torch.zeros((2, 807), dtype=torch.uint8), torch.zeros((808,), dtype=torch.uint8),
                torch.zeros((2, 808), dtype=torch.float32), torch.zeros((3, 808), dtype=torch.uint8).view(-1)[4:1620].view(2, 808)):
        with pytest.raises(ValueError):
            _capi.state_fields(bad)


def test_state_entry_points_reject_bad_arguments_without_a_device():
    L = C.CDLL(build.build())
    _capi.declare(L)
    buf = (C.c_uint64 * 256)()  # 8-byte aligned; the 16-byte aligned address inside it is found below
    base = C.addressof(buf)
    aligned = C.c_void_p(base + (-base) % 16)
    misaligned = C.c_void_p(aligned.value + 8)
    idx = (C.c_int64 * 2)(0, 1)
    for fn in (L.msoc_save_states, L.msoc_load_states):
        assert fn(None, None, 1, aligned, None) == -1  # null handle
        assert fn(None, None, 0, aligned, None) == -1
        # arguments are checked before the device is used: a zeroed stand-in handle (0 envs) is never launched on
        stand_in = (C.c_char * 4096)()
        fake = C.c_void_p(C.addressof(stand_in))
        assert fn(fake, None, -1, aligned, None) == -1  # n < 0
        assert fn(fake, idx, 1, None, None) == -1  # null state pointer
        assert fn(fake, idx, 1, misaligned, None) == -1  # misaligned state pointer
        assert b"16-byte" in L.msoc_last_error()
        assert fn(fake, None, 1, aligned, None) == -1  # NULL d_idx with n > the env count
        assert b"more entries than envs" in L.msoc_last_error()
        assert fn(fake, None, 0, aligned, None) == 0  # n = 0 is a no-op
        assert fn(fake, idx, 0, None, None) == 0
