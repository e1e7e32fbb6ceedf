"""CPU: the argument checks of pcgrl_step_envs, which return before any CUDA call, and the size of its work buffer.
The pointers below are never dereferenced on the host: the checks only compare them with NULL."""
from control_pcgrl_b200 import _lib
from tests.test_abi_cpu import _cfg, _lib_err
from tests.test_lookahead_abi_cpu import FAKE, _state


def _call(lib, c, st, n, env_idx=FAKE, actions=FAKE, work=FAKE):
    return lib.pcgrl_step_envs(c, st, actions, env_idx, n, work, None)


def test_step_envs_argument_errors():
    lib = _lib.load()
    c = _cfg()
    assert lib.pcgrl_config_check(c) == 0
    st = _state()
    E = _lib_err("PCGRL_E_ARG")
    assert _call(lib, c, st, 0) == 0                                     # nothing to do, nothing launched
    assert _call(lib, c, st, 0, env_idx=None, actions=None, work=None) == 0
    for name in ("env_idx", "actions", "work"):
        assert _call(lib, c, st, 4, **{name: None}) == E, name
    assert _call(lib, c, st, -1) == E
    assert _call(lib, c, st, 1 << 31) == E
    assert _call(lib, c, st, 9) == E                                     # 9 distinct indices of 8 envs
    assert b"n_envs" in lib.pcgrl_last_error()
    assert _call(lib, c, None, 4) == E
    for name in ("grids", "pos", "n_step", "iteration", "changes", "stats", "targets", "reward", "done"):
        bare = _state()
        setattr(bare, name, None)
        assert _call(lib, c, bare, 4) == E, name
    holey = _cfg("binary_holey", n_stats=3)
    assert lib.pcgrl_config_check(holey) == 0
    assert _call(lib, holey, st, 4) == E                                 # a holey problem needs holes
    assert b"holes" in lib.pcgrl_last_error()
    bad = _cfg()
    bad.n_stats = 5
    assert _call(lib, bad, st, 4) == E
    assert lib.pcgrl_step_envs_work_bytes(bad, 4) == -1
    assert lib.pcgrl_step_envs_work_bytes(c, -1) == -1


def test_step_envs_work_bytes_grow_with_n():
    lib = _lib.load()
    configs = [_cfg(), _cfg(dims=(32, 32)), _cfg("zelda", "turtle", (7, 11), 8, 7), _cfg("sokoban", dims=(5, 5), n_tiles=5,
                                                                                          n_stats=7)]
    for c in configs:
        assert lib.pcgrl_config_check(c) == 0
        sizes = [lib.pcgrl_step_envs_work_bytes(c, n) for n in (0, 1, 100, 10000, 1 << 20)]
        assert all(b > 0 for b in sizes)
        assert all(a < b for a, b in zip(sizes, sizes[1:])), sizes
        # at least the generic sub-shard's grids, and its outputs beside them
        n = 1 << 20
        assert sizes[-1] >= n * (c.row_stride + 4 * c.n_stats + 4 + 2)
