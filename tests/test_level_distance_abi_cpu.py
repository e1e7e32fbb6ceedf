"""CPU: the level-distance entry points (pcgrl_level_distances / pcgrl_level_knn / pcgrl_level_group_diversity /
pcgrl_level_work_bytes): ctypes argument types against the header, the argument checks that return before any CUDA
call, and the work size.  The pointers below are never dereferenced on the host: the checks only compare them with
NULL and the alignment."""
import ctypes as C
import os
import re

from control_pcgrl_b200 import _lib
from tests.test_abi_cpu import _cfg, _lib_err

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FAKE = 0x10000     # stands for a device pointer
E, U = _lib_err("PCGRL_E_ARG"), _lib_err("PCGRL_E_UNSUPPORTED")
NAMES = ("pcgrl_level_work_bytes", "pcgrl_level_distances", "pcgrl_level_knn", "pcgrl_level_group_diversity")


def _ctype(decl):
    decl = decl.strip()
    if "pcgrl_config" in decl:
        return C.POINTER(_lib.Config)
    if "*" in decl:
        return C.c_void_p
    return {"int64_t": C.c_int64, "int32_t": C.c_int32}[decl.split()[0]]


def test_argtypes_match_the_header():
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "pcgrl_b200.h")).read(), flags=re.S)
    for name in NAMES:
        m = re.search(r"\b(int64_t|int32_t)\s+" + name + r"\s*\(([^)]*)\)", src)
        assert m, name
        res, args = _lib.SYMBOLS[name]
        assert res == {"int64_t": C.c_int64, "int32_t": C.c_int32}[m.group(1)], name
        assert args == [_ctype(d) for d in m.group(2).split(",")], name


def _geom(c):
    cells = c.dims[0] * c.dims[1] * (c.dims[2] if c.ndim == 3 else 1)
    w, p = (cells + 31) // 32, max(1, (c.n_tiles - 1).bit_length())
    return cells, w * p


def _a256(x):
    return (x + 255) // 256 * 256


def test_work_bytes():
    lib = _lib.load()
    b = _cfg()                                                           # binary 16x16: 1 plane of 8 words
    assert lib.pcgrl_config_check(b) == 0 and _geom(b) == (256, 8)
    assert lib.pcgrl_level_work_bytes(b, 10, 0, 0) == _a256(320)
    assert lib.pcgrl_level_work_bytes(b, 10, 3, 0) == _a256(320) + _a256(96)
    assert lib.pcgrl_level_work_bytes(b, 0, 0, 0) == 0
    # 64 Ki queries fill the GPU alone: one archive slice, no partial lists
    assert lib.pcgrl_level_work_bytes(b, 1 << 16, 1 << 20, 15) == (1 << 16) * 32 + (1 << 20) * 32
    # 1 Ki queries (32 blocks) against 1 Mi levels (8192 trips of 128): 32 slices of 32 Ki levels, k keys of 8 bytes
    assert lib.pcgrl_level_work_bytes(b, 1024, 1 << 20, 15) == 1024 * 32 + (1 << 20) * 32 + 32 * 1024 * 15 * 8
    # ... at most 64 slices, and at least 8 trips per slice
    assert lib.pcgrl_level_work_bytes(b, 1, 1 << 20, 1) == 256 + (1 << 20) * 32 + 64 * 8
    assert lib.pcgrl_level_work_bytes(b, 1, 1919, 1) == 256 + _a256(1919 * 32)         # 15 trips: one slice
    assert lib.pcgrl_level_work_bytes(b, 1, 2048, 3) == 256 + 2048 * 32 + 2 * 3 * 8    # 16 trips: two slices
    z = _cfg("zelda", "turtle", (7, 11), 8, 7)                           # 77 cells, 8 tiles: 3 planes of 3 words
    assert lib.pcgrl_config_check(z) == 0 and _geom(z) == (77, 9)
    assert lib.pcgrl_level_work_bytes(z, 10, 20, 0) == _a256(360) + _a256(720)
    m = _cfg("minecraft_3D_maze", dims=(14, 14, 14), n_tiles=2, n_stats=3)
    assert lib.pcgrl_config_check(m) == 0 and _geom(m) == (2744, 86)
    assert lib.pcgrl_level_work_bytes(m, 7, 0, 0) == _a256(7 * 86 * 4)
    smb = _cfg("smb", dims=(116, 16), n_tiles=7, n_stats=9)             # 1856 cells, 7 tiles: 3 planes of 58 words
    assert lib.pcgrl_config_check(smb) == 0 and _geom(smb) == (1856, 174)
    assert lib.pcgrl_level_work_bytes(smb, 3, 5, 0) == _a256(3 * 174 * 4) + _a256(5 * 174 * 4)
    for bad in ((-1, 0, 0), (0, -1, 0), (1, 1, -1), (1, 1, 65)):
        assert lib.pcgrl_level_work_bytes(b, *bad) == -1, bad
    nc = _cfg()
    nc.n_stats = 5
    assert lib.pcgrl_level_work_bytes(nc, 1, 1, 1) == -1


def _dist(lib, c, a=FAKE, na=4, sa=256, b=FAKE, nb=4, sb=256, out=FAKE, work=FAKE):
    return lib.pcgrl_level_distances(c, a, na, sa, b, nb, sb, out, work, None)


def _knn(lib, c, q=FAKE, nq=4, sq=256, b=FAKE, nb=4, sb=256, k=3, off=-1, dist=FAKE, idx=FAKE, work=FAKE):
    return lib.pcgrl_level_knn(c, q, nq, sq, b, nb, sb, k, off, dist, idx, work, None)


def _div(lib, c, a=FAKE, n=6, s=256, g=3, sums=FAKE, work=FAKE):
    return lib.pcgrl_level_group_diversity(c, a, n, s, g, sums, work, None)


def test_argument_errors_before_launch():
    lib = _lib.load()
    c = _cfg()
    assert lib.pcgrl_config_check(c) == 0
    # nothing to compute: nothing launched
    assert _dist(lib, c, na=0) == 0 and _dist(lib, c, nb=0, b=None) == 0
    assert _knn(lib, c, nq=0, q=None) == 0 and _div(lib, c, n=0, a=None) == 0
    for call in (_dist, _knn, _div):
        assert call(lib, c, work=None) == E, call
        assert call(lib, c, work=FAKE + 8) == E, call                   # work must be 16-byte aligned
        assert call(lib, None) == E, call
        bad = _cfg()
        bad.n_stats = 5
        assert call(lib, bad) == E, call
    assert _dist(lib, c, sa=255) == E and b"stride" in lib.pcgrl_last_error()
    assert _dist(lib, c, sb=0) == E
    assert _dist(lib, c, na=-1) == E and _dist(lib, c, nb=1 << 31) == E
    assert _dist(lib, c, a=None) == E and _dist(lib, c, b=None) == E and _dist(lib, c, out=None) == E
    for k in (0, -1, 65):
        assert _knn(lib, c, k=k) == E and b"k must" in lib.pcgrl_last_error()
    assert _knn(lib, c, off=-2) == E
    assert _knn(lib, c, sq=100) == E and _knn(lib, c, sb=100) == E
    assert _knn(lib, c, dist=None) == E and _knn(lib, c, idx=None) == E
    assert _knn(lib, c, q=None) == E and _knn(lib, c, b=None) == E
    assert _knn(lib, c, nq=-3) == E
    for g in (0, 1, 4):
        assert _div(lib, c, g=g) == E, g                                 # 4 does not divide 6
    assert _div(lib, c, sums=None) == E and _div(lib, c, s=10) == E and _div(lib, c, a=None) == E
    big = _cfg(dims=(128, 128))                                          # 512 words: larger than the tile
    assert lib.pcgrl_config_check(big) == 0
    assert _dist(lib, big, sa=1 << 14, sb=1 << 14) == U
    assert _knn(lib, big, sq=1 << 14, sb=1 << 14) == U
    assert _div(lib, big, s=1 << 14) == U
