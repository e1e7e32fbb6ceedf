"""CPU: the argument checks of pcgrl_lookahead_obs, which return before any CUDA call, and the size of its work buffer.
The pointers below are never dereferenced on the host: the checks only compare them with NULL."""
from control_pcgrl_b200 import _lib
from tests.test_abi_cpu import _cfg, _lib_err

FAKE = 0x10000     # stands for a device pointer


def _state(n_envs=8):
    st = _lib.State()
    st.n_envs = n_envs
    for name in ("grids", "pos", "n_step", "iteration", "changes", "stats", "targets", "reward", "done", "changed"):
        setattr(st, name, FAKE)
    return st


def _obs(crop=1, dims=(32, 32), out_kind=0):
    oa = _lib.ObsArgs()
    oa.crop, oa.out_kind, oa.out = crop, out_kind, FAKE
    for i, d in enumerate(dims):
        oa.obs_dims[i] = d
    return oa


def _call(lib, c, st, n, obs, env_idx=FAKE, **null):
    args = dict(actions=FAKE, reward=FAKE, done=FAKE, changed=FAKE, stats=FAKE, work=FAKE)
    args.update(null)
    return lib.pcgrl_lookahead_obs(c, st, obs, args["actions"], env_idx, n, args["reward"], args["done"],
                                   args["changed"], args["stats"], args["work"], None)


def test_lookahead_obs_argument_errors():
    lib = _lib.load()
    c = _cfg()
    assert lib.pcgrl_config_check(c) == 0
    st = _state()
    E = _lib_err("PCGRL_E_ARG")
    oa = _obs()
    assert _call(lib, c, st, 0, oa) == 0                                 # nothing to do, nothing launched
    assert _call(lib, c, st, 0, oa, env_idx=None) == 0
    for name in ("actions", "reward", "done", "changed", "stats", "work"):
        assert _call(lib, c, st, 4, oa, **{name: None}) == E, name
    assert _call(lib, c, st, 4, None) == E
    assert _call(lib, c, st, 0, None) == E                               # obs is required even when n == 0
    assert _call(lib, c, st, -1, oa) == E
    assert _call(lib, c, st, 9, oa, env_idx=None) == E                  # candidate j is env j: n > n_envs
    assert b"n_envs" in lib.pcgrl_last_error()
    assert _call(lib, c, None, 4, oa) == E
    bare = _state()
    bare.grids = None
    assert _call(lib, c, bare, 4, oa) == E
    holey = _cfg("binary_holey", n_stats=3)
    assert lib.pcgrl_config_check(holey) == 0
    assert _call(lib, holey, st, 4, oa) == E                             # a holey problem needs holes
    bad = _cfg()
    bad.n_stats = 5
    assert _call(lib, bad, st, 4, oa) == E
    # the observation's own arguments, checked before any launch
    no_out = _obs()
    no_out.out = None
    assert _call(lib, c, st, 4, no_out) == E
    assert _call(lib, c, st, 4, _obs(out_kind=4)) == E
    assert _call(lib, c, st, 4, _obs(out_kind=-1)) == E
    ctrl_u8 = _obs(out_kind=0)
    ctrl_u8.n_ctrl, ctrl_u8.ctrl_idx[0] = 1, 0
    assert _call(lib, c, st, 4, ctrl_u8) == E                            # target planes are fractional
    assert b"target planes" in lib.pcgrl_last_error()
    for n_ctrl in (-1, _lib.MAX_STATS + 1):
        o = _obs(out_kind=1)
        o.n_ctrl = n_ctrl
        assert _call(lib, c, st, 4, o) == E
    static = _obs()
    static.static_channel = 1
    assert _call(lib, c, st, 4, static) == E                             # no static mask in the state
    assert _call(lib, c, st, 4, _obs(crop=0, dims=(15, 16))) == E       # the whole map is 16 x 16
    holey_st = _state()
    holey_st.holes = FAKE
    assert _call(lib, holey, holey_st, 4, _obs(crop=0, dims=(16, 16))) == E   # the bordered map is 18 x 18
    tile = _obs(crop=0, dims=(18, 18))
    tile.holey_border_tile = 2
    assert _call(lib, holey, holey_st, 4, tile) == E                     # binary has tiles 0 and 1
    assert lib.pcgrl_lookahead_obs_work_bytes(bad, 4) == -1
    assert lib.pcgrl_lookahead_obs_work_bytes(c, -1) == -1


def test_lookahead_obs_work_bytes_cover_the_lookahead_and_grow_with_n():
    lib = _lib.load()
    configs = [_cfg(), _cfg(dims=(14, 14), problem="minecraft_2D_maze", n_stats=2), _cfg(dims=(32, 32)),
               _cfg("zelda", "turtle", (7, 11), 8, 7), _cfg("sokoban", dims=(5, 5), n_tiles=5, n_stats=7),
               _cfg("minecraft_3D_maze", dims=(14, 14, 14), n_stats=3)]
    for c in configs:
        assert lib.pcgrl_config_check(c) == 0
        ns = (0, 1, 100, 10000, 1 << 20)
        sizes = [lib.pcgrl_lookahead_obs_work_bytes(c, n) for n in ns]
        assert all(b > 0 for b in sizes)
        assert all(a < b for a, b in zip(sizes, sizes[1:])), sizes
        for n, b in zip(ns, sizes):
            assert b >= lib.pcgrl_lookahead_work_bytes(c, n), (n, b)
        # the sub-shard's grids, behind the 256-byte work-list header
        assert sizes[-1] >= 256 + (1 << 20) * c.row_stride
    # a search cache's work-list body sits beside the sub-shard, not inside it
    c = _cfg()
    assert lib.pcgrl_config_check(c) == 0
    assert lib.pcgrl_cache_stride(c) > 0
    n = 1 << 16
    assert lib.pcgrl_lookahead_obs_work_bytes(c, n) >= 256 + n * (2 * c.row_stride + 12 + 12) + n * (2 + 2 + 1) * 4
