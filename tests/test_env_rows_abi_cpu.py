"""CPU: the packed env row (pcgrl_env_row_layout, pcgrl_save_envs / pcgrl_load_envs).  The layout query is host only,
and the argument checks return before any CUDA call; the pointers below are never dereferenced on the host."""
import ctypes
import os
import subprocess
import tempfile

from control_pcgrl_b200 import _lib
from tests.test_abi_cpu import _cfg, _lib_err
from tests.test_lookahead_abi_cpu import FAKE, _state

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OFFSETS = ("grid", "static_mask", "cache", "records", "targets", "stats", "holes", "pos", "n_step", "iteration",
           "changes", "reward", "done", "changed")
# the sections, as (first field, fields in it)
SECTIONS = (("grid",), ("static_mask",), ("cache",), ("records",), ("targets",), ("stats",), ("holes",), ("pos",),
            ("n_step", "iteration", "changes"), ("reward", "done", "changed"))


def _layout(c, st, n_pos=1):
    lay = _lib.RowLayout()
    rc = _lib.load().pcgrl_env_row_layout(c, st, n_pos, lay)
    assert rc == 0, _lib.load().pcgrl_last_error()
    return lay


def _sizes(c, lay, cache=0, rec=0, holes=0):
    """Bytes of every section, from the config (0 = absent)."""
    K = c.n_stats
    return {"grid": c.row_stride, "static_mask": c.row_stride, "cache": cache, "records": rec, "targets": 16 * K,
            "stats": 4 * K, "holes": 4 * holes, "pos": 12 * lay.n_pos, "n_step": 12,
            "reward": 6 if lay.changed >= 0 else 5}


def _check_layout(c, lay, **kw):
    sizes = _sizes(c, lay, **kw)
    spans = []
    for sec in SECTIONS:
        off = getattr(lay, sec[0])
        if off < 0:
            assert all(getattr(lay, f) == -1 for f in sec[1:]), sec
            continue
        assert off % 16 == 0, (sec, off)
        spans.append((off, off + (sizes[sec[0]] + 15) // 16 * 16))
    spans.sort()
    assert spans[0][0] == 16                                  # behind the header
    for (a0, a1), (b0, b1) in zip(spans, spans[1:]):
        assert a1 == b0, spans                                # disjoint, no gap beyond the 16-byte padding
    assert lay.row_bytes == spans[-1][1] and lay.row_bytes % 16 == 0
    assert (lay.iteration, lay.changes, lay.done) == (lay.n_step + 4, lay.n_step + 8, lay.reward + 4)
    assert lay.signature != 0


def test_layout_sections_follow_the_shard():
    lib = _lib.load()
    c = _cfg()
    assert lib.pcgrl_config_check(c) == 0
    st = _state()
    lay = _layout(c, st)
    _check_layout(c, lay)
    assert [getattr(lay, f) for f in ("static_mask", "cache", "records", "targets", "holes")] == [-1] * 5
    assert lay.row_bytes == 16 + 256 + 16 + 16 + 16 + 16

    # the cache only with work list + cache (the condition the step uses), at pcgrl_cache_stride bytes
    cs = lib.pcgrl_cache_stride(c)
    assert cs == 80
    for wl, cache in ((FAKE, None), (None, FAKE)):
        s = _state()
        s.worklist, s.cache = wl, cache
        assert _layout(c, s).cache == -1
    s = _state()
    s.worklist = s.cache = FAKE
    lay_c = _layout(c, s)
    _check_layout(c, lay_c, cache=cs)
    assert lay_c.cache > 0 and lay_c.row_bytes == lay.row_bytes + 80
    # 8x8 and 2x2 maps: cache strides 48 and 24 (not a multiple of 16)
    for dims, want in (((8, 8), 48), ((2, 2), 24)):
        c8 = _cfg(dims=dims)
        assert lib.pcgrl_config_check(c8) == 0 and lib.pcgrl_cache_stride(c8) == want
        _check_layout(c8, _layout(c8, s), cache=want)

    # records only with record_stat_bytes (and the records pointer)
    cr = _cfg()
    cr.record_stat_bytes = 1
    assert lib.pcgrl_config_check(cr) == 0
    assert _layout(cr, st).records == -1
    s = _state()
    s.records = FAKE
    assert _layout(c, s).records == -1
    lay_r = _layout(cr, s)
    _check_layout(cr, lay_r, rec=lib.pcgrl_record_stride(cr))
    assert lay_r.records > 0

    # frozen mask, per-env targets, no changed flag
    s = _state()
    s.static_mask = FAKE
    s.changed = None
    ct = _cfg()
    ct.targets_per_env = 1
    assert lib.pcgrl_config_check(ct) == 0
    lay_t = _layout(ct, s)
    _check_layout(ct, lay_t)
    assert lay_t.static_mask > 0 and lay_t.targets > 0 and lay_t.changed == -1

    # holes only for a holey problem: 4 ints in 2D, 6 in 3D
    s = _state()
    s.holes = FAKE
    assert _layout(c, s).holes == -1
    h2 = _cfg("binary_holey", n_stats=3)
    h3 = _cfg("minecraft_3D_holey_maze", dims=(8, 8, 8), n_tiles=2, n_stats=5)
    for hc, ints in ((h2, 4), (h3, 6)):
        assert lib.pcgrl_config_check(hc) == 0
        lay_h = _layout(hc, s)
        _check_layout(hc, lay_h, holes=ints)
        assert lay_h.holes > 0

    # n_pos position triples
    for n_pos in (1, 2, 3, 6):
        lay_p = _layout(c, st, n_pos)
        _check_layout(c, lay_p)
        assert lay_p.n_pos == n_pos
        assert lay_p.row_bytes == lay.row_bytes + (12 * n_pos + 15) // 16 * 16 - 16


def test_signatures():
    lib = _lib.load()
    s = _state()
    s.worklist = s.cache = FAKE
    narrow, turtle = _cfg(), _cfg(rep="turtle")
    for c in (narrow, turtle):
        assert lib.pcgrl_config_check(c) == 0
    a, b = _layout(narrow, s), _layout(turtle, s)
    assert a.row_bytes == b.row_bytes and a.signature != b.signature
    # episode and reward parameters are not part of the row's meaning
    other = _cfg()
    other.max_iterations, other.max_changes = 5, 3
    other.weights[0], other.weights[1] = 2.5, -1.0
    other.reward_mode = _lib.REWARD_RANGE
    other.init_probs[0] = 0.3
    other.static_prob = 0.5
    assert lib.pcgrl_config_check(other) == 0
    o = _layout(other, s)
    assert (o.row_bytes, o.signature) == (a.row_bytes, a.signature)
    # a different map, n_pos or section set is another layout
    for c2, s2, n_pos in ((_cfg(dims=(14, 14)), s, 1), (narrow, s, 2), (narrow, _state(), 1)):
        assert lib.pcgrl_config_check(c2) == 0
        assert _layout(c2, s2, n_pos).signature != a.signature


def test_env_rows_argument_errors():
    lib = _lib.load()
    c = _cfg()
    assert lib.pcgrl_config_check(c) == 0
    st = _state()
    E = _lib_err("PCGRL_E_ARG")
    lay = _lib.RowLayout()
    assert lib.pcgrl_env_row_layout(c, st, 0, lay) == E
    assert b"n_pos" in lib.pcgrl_last_error()
    assert lib.pcgrl_env_row_layout(c, st, 1, None) == E
    assert lib.pcgrl_env_row_layout(c, None, 1, lay) == E
    save = lambda c, st, n, env_idx=FAKE, rows=FAKE, n_pos=1: lib.pcgrl_save_envs(c, st, n_pos, env_idx, n, rows, None)  # noqa: E731
    load = lambda c, st, n, env_idx=FAKE, rows=FAKE, n_pos=1: lib.pcgrl_load_envs(c, st, n_pos, rows, env_idx, n, None)  # noqa: E731
    for call in (save, load):
        assert call(c, st, 0) == 0                                       # nothing to do, nothing launched
        assert call(c, st, 0, env_idx=None, rows=None) == 0
        assert call(c, st, 4, rows=None) == E
        assert call(c, st, 4, rows=FAKE + 8) == E                        # rows are 16-byte aligned
        assert call(c, st, -1) == E
        assert call(c, st, 1 << 31) == E
        assert call(c, st, 9, env_idx=None) == E                         # row j is env j: n > n_envs
        assert b"n_envs" in lib.pcgrl_last_error()
        assert call(c, st, 4, n_pos=0) == E
        assert call(c, None, 4) == E
        for name in ("grids", "pos", "n_step", "iteration", "changes", "stats", "targets", "reward", "done"):
            bare = _state()
            setattr(bare, name, None)
            assert call(c, bare, 4) == E, name
        holey = _cfg("binary_holey", n_stats=3)
        assert lib.pcgrl_config_check(holey) == 0
        assert call(holey, st, 4) == E                                   # a holey problem needs holes
        assert b"holes" in lib.pcgrl_last_error()
        bad = _cfg()
        bad.n_stats = 5
        assert call(bad, st, 4) == E
    assert load(c, st, 9) == E                                           # 9 distinct indices of 8 envs


def test_row_layout_struct_matches_header():
    code = ('#include "pcgrl_b200.h"\n#include <stdio.h>\n#include <stddef.h>\n'
            'int main(){printf("%zu %zu %zu %zu %zu %zu\\n", sizeof(pcgrl_row_layout), '
            'offsetof(pcgrl_row_layout, signature), offsetof(pcgrl_row_layout, n_pos), '
            'offsetof(pcgrl_row_layout, grid), offsetof(pcgrl_row_layout, holes), '
            'offsetof(pcgrl_row_layout, changed));return 0;}\n')
    with tempfile.TemporaryDirectory() as d:
        src = os.path.join(d, "s.c")
        with open(src, "w") as f:
            f.write(code)
        exe = os.path.join(d, "s")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), src, "-o", exe])
        out = subprocess.check_output([exe]).decode().split()
    R = _lib.RowLayout
    assert [int(v) for v in out] == [ctypes.sizeof(R), R.signature.offset, R.n_pos.offset, R.grid.offset,
                                     R.holes.offset, R.changed.offset]
    assert [name for name, _ in R._fields_[3:]] == list(OFFSETS)
