"""CPU: pcgrl_update validates its arguments before it launches anything (no device needed)."""
import ctypes

from control_pcgrl_b200 import _lib

E_ARG = -1


def _cfg():
    c = _lib.Config()
    c.abi_version = _lib.PCGRL_ABI_VERSION
    c.problem, c.representation, c.action_kind = _lib.PROB_IDS["binary"], _lib.REP_IDS["narrow"], _lib.ACT_INT32
    c.ndim, c.dims[0], c.dims[1] = 2, 16, 16
    c.n_tiles, c.n_stats = 2, 2
    c.max_iterations, c.max_changes = 769, -1
    return c


def _state(**null):
    """A state whose update pointers are non-NULL (never dereferenced: every call below fails validation)."""
    buf = (ctypes.c_uint8 * 64)()
    p = ctypes.addressof(buf)
    st = _lib.State()
    st.n_envs = 4
    for f in ("grids", "pos", "n_step", "changed"):
        setattr(st, f, None if null.get(f) else p)
    return st, buf


def test_update_rejects_null_arguments_without_launching():
    lib = _lib.load()
    c = _cfg()
    assert lib.pcgrl_config_check(c) == 0
    n0 = lib.pcgrl_launch_count()
    dummy = ctypes.c_int32(0)
    act = ctypes.addressof(dummy)
    assert lib.pcgrl_update(c, None, act, None) == E_ARG                    # NULL state
    assert b"state" in lib.pcgrl_last_error()
    st, keep = _state()
    assert lib.pcgrl_update(c, st, None, None) == E_ARG                     # NULL actions
    assert b"actions" in lib.pcgrl_last_error()
    for f in ("grids", "pos", "n_step", "changed"):                          # each required state pointer
        st, keep = _state(**{f: True})
        assert lib.pcgrl_update(c, st, act, None) == E_ARG, f
        assert b"changed" in lib.pcgrl_last_error()
    st, keep = _state()
    st.n_envs = -1
    assert lib.pcgrl_update(c, st, act, None) == E_ARG
    bad = _cfg()
    bad.abi_version = _lib.PCGRL_ABI_VERSION + 1                            # check(cfg) runs first
    st, keep = _state()
    assert lib.pcgrl_update(bad, st, act, None) == E_ARG
    assert lib.pcgrl_launch_count() == n0
