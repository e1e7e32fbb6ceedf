"""Level distances (pcgrl_level_distances / pcgrl_level_knn / pcgrl_level_group_diversity; level_distances, level_knn,
level_diversity, BatchedPcgrlEnv.novelty / diversity).

Every result is compared with torch.equal against plain torch: d = (a[:, None, :cells] != b[None, :, :cells]).sum(-1),
then a stable sort of each row on distance, so that equal distances keep ascending archive index.  Problems from one
bit-plane (binary) to four (zelda's 8 tiles need three, smb's 7 three); counts 1, 31, 33, primes, enough archive rows for
several trips of every block, and a few queries against a large archive, which splits the archive and merges.  Inputs
come from random grids with garbage in the row padding, from env grids and from saved env rows; duplicated levels make
ties."""
import numpy as np
import pytest
import torch

import control_pcgrl_b200 as P

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
PROBLEMS = [("binary", (16, 16)), ("binary", (64, 64)), ("zelda", (7, 11)), ("sokoban", (5, 5)), ("smb", (116, 16)),
            ("minecraft_3D_maze", (14, 14, 14)), ("binary_holey", (16, 16))]


def _cfg(problem, shape):
    return P.make_config(problem, "narrow", map_shape=shape)


def _geom(problem, shape):
    from control_pcgrl_b200.problems import get_spec
    cells = int(np.prod(shape))
    return cells, (cells + 15) // 16 * 16, get_spec(problem, shape).n_tiles


def _levels(n, problem, shape, seed, dup=True, width=None):
    """n random levels as [n, width] int8 rows (default row_stride) with garbage padding; some rows copy others."""
    cells, stride, n_tiles = _geom(problem, shape)
    g = torch.Generator(device=DEV).manual_seed(seed)
    w = stride if width is None else width
    t = torch.randint(-128, 128, (n, w), generator=g, device=DEV, dtype=torch.int32).to(torch.int8)
    t[:, :cells] = torch.randint(0, n_tiles, (n, cells), generator=g, device=DEV, dtype=torch.int32).to(torch.int8)
    if dup and n > 3:
        src = torch.randint(0, n, (n // 3,), generator=g, device=DEV)
        dst = torch.randint(0, n, (n // 3,), generator=g, device=DEV)
        t[dst, :cells] = t[src, :cells]
    return t


def _ref_dist(a, b, cells):
    out = torch.empty((a.shape[0], b.shape[0]), dtype=torch.int32, device=a.device)
    for lo in range(0, a.shape[0], 64):
        out[lo:lo + 64] = (a[lo:lo + 64, None, :cells] != b[None, :, :cells]).sum(-1).to(torch.int32)
    return out


def _ref_knn(a, b, cells, k, self_offset=None):
    d = _ref_dist(a, b, cells).to(torch.int64)
    n = b.shape[0]
    if self_offset is not None:
        i = torch.arange(a.shape[0], device=a.device)
        j = i + self_offset
        ok = j < n
        d[i[ok], j[ok]] = 1 << 40                     # excluded: sorts last, read back as -1
    sd, si = torch.sort(d, dim=1, stable=True)
    sd, si = sd[:, :k], si[:, :k]
    gone = sd >= 1 << 40
    sd[gone], si[gone] = -1, -1
    m = a.shape[0]
    dist = torch.full((m, k), -1, dtype=torch.int32, device=a.device)
    idx = torch.full((m, k), -1, dtype=torch.int32, device=a.device)
    dist[:, :sd.shape[1]], idx[:, :si.shape[1]] = sd.to(torch.int32), si.to(torch.int32)
    return dist, idx


def _ref_div(a, cells, s):
    d = _ref_dist(a, a, cells).to(torch.int64)
    g = a.shape[0] // s
    blocks = torch.stack([d[i * s:(i + 1) * s, i * s:(i + 1) * s] for i in range(g)])
    return torch.triu(blocks, diagonal=1).sum((1, 2)).double() / (s * (s - 1) // 2)


@pytest.mark.parametrize("problem,shape", PROBLEMS)
def test_distances_knn_diversity(problem, shape):
    cfg = _cfg(problem, shape)
    cells, _, _ = _geom(problem, shape)
    big = 300 if cells < 1000 else 270                # > 2 archive trips of 128
    for m, n in ((1, 1), (31, 33), (33, 31), (37, big), (97, 5)):
        a = _levels(m, problem, shape, seed=m * 7 + n)
        b = _levels(n, problem, shape, seed=m * 11 + n + 1)
        assert torch.equal(P.level_distances(a, b, cfg=cfg), _ref_dist(a, b, cells)), (m, n)
        for k in (1, 10, 64):
            got = P.level_knn(a, b, k=k, cfg=cfg)
            want = _ref_knn(a, b, cells, k)
            assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1]), (m, n, k)
    a = _levels(big, problem, shape, seed=5)
    assert torch.equal(P.level_distances(a, cfg=cfg), _ref_dist(a, a, cells))
    for k in (1, 10, 64):
        got = P.level_knn(a, k=k, cfg=cfg, exclude_self=True)
        want = _ref_knn(a, a, cells, k, self_offset=0)
        assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1]), k
        assert not bool((got[1] == torch.arange(big, device=DEV)[:, None]).any())
    for s in (2, 3, 17):
        n = s * (7 if s < 17 else 3)
        lv = _levels(n, problem, shape, seed=s)
        assert torch.equal(P.level_diversity(lv, s, cfg=cfg), _ref_div(lv, cells, s)), s


@pytest.mark.parametrize("problem,shape", [("binary", (16, 16)), ("zelda", (7, 11)), ("smb", (116, 16))])
def test_knn_split_and_merge(problem, shape):
    """A few queries against an archive of many trips: the archive is cut into slices, each slice's lists are merged."""
    cfg = _cfg(problem, shape)
    cells, _, _ = _geom(problem, shape)
    n = 5003 if cells < 1000 else 2503
    b = _levels(n, problem, shape, seed=1)
    for m in (1, 31, 67):
        a = torch.cat([b[:m // 2], _levels(m - m // 2, problem, shape, seed=m)])   # some queries are in the archive
        for k in (1, 15, 64):
            got = P.level_knn(a, b, k=k, cfg=cfg)
            want = _ref_knn(a, b, cells, k)
            assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1]), (m, k)
        got = P.level_knn(a, b, k=10, cfg=cfg, exclude_self=True, self_offset=3)
        want = _ref_knn(a, b, cells, 10, self_offset=3)
        assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1]), m


def test_ties_go_to_the_lower_index():
    cfg = _cfg("binary", (16, 16))
    base = _levels(1, "binary", (16, 16), seed=3, dup=False)
    b = base.repeat(3000, 1)                                      # every archive level is the query: all distances 0
    flip = torch.arange(0, 3000, 7, device=DEV)
    b[flip, 5] ^= 1                                               # ... except every 7th, at distance 1
    for m in (1, 40):
        dist, idx = P.level_knn(base.repeat(m, 1), b, k=64, cfg=cfg)
        keep = torch.tensor([i for i in range(3000) if i % 7][:64], dtype=torch.int32, device=DEV)
        assert torch.equal(idx, keep.repeat(m, 1)) and int(dist.abs().sum()) == 0


def test_k_larger_than_the_archive():
    cfg = _cfg("zelda", (7, 11))
    a, b = _levels(33, "zelda", (7, 11), seed=1), _levels(5, "zelda", (7, 11), seed=2)
    for k in (6, 64):
        dist, idx = P.level_knn(a, b, k=k, cfg=cfg)
        want = _ref_knn(a, b, 77, k)
        assert torch.equal(dist, want[0]) and torch.equal(idx, want[1])
        assert bool((dist[:, 5:] == -1).all() and (idx[:, 5:] == -1).all())
    dist, idx = P.level_knn(b, k=5, cfg=cfg, exclude_self=True)
    assert bool((dist[:, 4] == -1).all()) and bool((idx[:, :4] >= 0).all())
    dist, idx = P.level_knn(a, b[:0], k=3, cfg=cfg)
    assert bool((dist == -1).all() and (idx == -1).all())


def test_padding_never_counts_and_widths():
    """[M, cells] maps, [M, row_stride] rows with different garbage padding, and a wider row: all the same distances."""
    cfg = _cfg("zelda", (7, 11))
    a = _levels(40, "zelda", (7, 11), seed=4)
    b = a.clone()
    b[:, 77:] = ~b[:, 77:]                                        # only the padding differs
    assert int(P.level_distances(a, b, cfg=cfg).diagonal().abs().sum()) == 0
    wide = torch.randint(0, 256, (40, 203), device=DEV, dtype=torch.int32).to(torch.uint8)
    wide[:, :77] = a[:, :77].to(torch.uint8)
    want = _ref_dist(a, a, 77)
    assert torch.equal(P.level_distances(a[:, :77].contiguous(), wide, cfg=cfg), want)
    wide[:, 3:80] = a[:, :77].to(torch.uint8)                   # odd stride, levels at an unaligned offset
    assert torch.equal(P.level_distances(wide[:, 3:], a, cfg=cfg), want)
    assert torch.equal(P.level_knn(wide[:, 3:], k=7, cfg=cfg)[1], _ref_knn(a, a, 77, 7)[1])


@pytest.mark.parametrize("problem,shape", [("binary", (16, 16)), ("binary_holey", (16, 16)),
                                           ("minecraft_3D_maze", (14, 14, 14))])
def test_env_grids_saved_rows_novelty_diversity(problem, shape):
    cfg = _cfg(problem, shape)
    cells, _, _ = _geom(problem, shape)
    env = P.BatchedPcgrlEnv(cfg, 96, device=DEV, seed=2)
    env.reset()
    archive = P.BatchedPcgrlEnv(cfg, 200, device=DEV, seed=9)
    archive.reset()
    rows = archive.save_envs()
    arch = archive.grids
    want = _ref_knn(env.grids, arch, cells, 12)
    for b in (rows, env.row_fields(rows)["grids"]):
        got = P.level_knn(env.grids, b, k=12, cfg=env)
        assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])
    nov = env.novelty(rows, 12)
    assert torch.equal(nov, want[0].double().mean(1).float())
    ids = [5, 0, 95, 5]
    assert torch.equal(env.novelty(rows, 12, env_ids=ids), nov[ids])
    with pytest.raises(IndexError):
        env.novelty(rows, 12, env_ids=[96])
    assert torch.equal(env.diversity(16), _ref_div(env.grids, cells, 16))
    assert torch.equal(P.level_distances(env.save_envs(), rows, cfg=env), _ref_dist(env.grids, arch, cells))
    few = env.novelty(rows[:3], 12)
    assert torch.equal(few, _ref_dist(env.grids, arch[:3], cells).double().mean(1).float())


def test_argument_errors_raise_before_launch():
    cfg = _cfg("binary", (16, 16))
    a = _levels(8, "binary", (16, 16), seed=0)
    for k in (0, 65):
        with pytest.raises(ValueError):
            P.level_knn(a, k=k, cfg=cfg)
    with pytest.raises(ValueError):
        P.level_diversity(a, 3, cfg=cfg)
    with pytest.raises(ValueError):
        P.level_diversity(a, 1, cfg=cfg)
    with pytest.raises(ValueError):
        P.level_distances(a[:, :200], cfg=cfg)                  # fewer than cells bytes per level
    with pytest.raises(ValueError):
        P.level_distances(a.cpu(), cfg=cfg)
    with pytest.raises(ValueError):
        P.level_distances(a.to(torch.int32), cfg=cfg)
