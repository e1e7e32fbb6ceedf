"""Packed env rows (pcgrl_save_envs / pcgrl_load_envs; BatchedPcgrlEnv.save_envs / load_envs / fork_envs / row_fields).

For every config of the lookahead suite: a round trip (save in a random order with repeats, scramble, load back) must
restore every state tensor and output byte for byte, after which the env and a twin restored from a snapshot agree
step for step and on lookahead_all (a stale cache row would show there); a fork must equal the torch-index reference
t[dst] = t[src] over every per-env tensor, before and after identical steps.  Then: random sequences with auto_reset,
rows moved between env objects (and devices), row_fields, rejection of foreign rows and bad indices, the device-side
guards, the README's beam search, and a fork over a 1 Mi-env shard."""
import numpy as np
import pytest
import torch

import control_pcgrl_b200 as P
from tests.test_gpu_lookahead import CASES, _actions, _make, _prepare
from tests.test_gpu_step_envs import STATE, _assert_same, _bits, _distinct, _env, _snapshot, _twin_of

pytestmark = pytest.mark.gpu


def _ids(a, dev):
    return torch.as_tensor(np.asarray(a, dtype=np.int32)).to(dev)


def _ref_fork(env, src, dst):
    """The torch-index workaround: every per-env tensor's rows dst take the rows src had before."""
    s, d = src.long(), dst.long()
    for k in STATE:
        t = getattr(env, k)
        if t is None:
            continue
        if k == "agent_pos":
            t[:, d] = t[:, s]
        elif t.shape[0] == env.n_envs:      # not the shared [1, K, 2] targets
            t[d] = t[s]


def _full_steps(env, twin, g, rounds, what):
    for _ in range(rounds):
        for a in range(max(env.n_agents, 1)):
            acts = _actions(env, env.n_envs, g)
            r1, d1 = env.step(acts, agent=a)
            r2, d2 = twin.step(acts, agent=a)
            assert torch.equal(r1.view(torch.int32), r2.view(torch.int32)) and torch.equal(d1, d2), what
            _assert_same(env, twin, what)


def _assert_lookahead_all_equal(env, twin, agent, what):
    if env.action_kind in ("int32", "wide_flat") and not (
            env.action_kind == "wide_flat" and (env._cc.act_w > env.map_shape[0] or env._cc.act_h > env.map_shape[1])):
        for x, y in zip(env.lookahead_all(agent=agent), twin.lookahead_all(agent=agent)):
            assert torch.equal(_bits(x), _bits(y)), what


@pytest.mark.parametrize("case", CASES, ids=[c.id for c in CASES])
def test_round_trip(case):
    env = _make(case)
    g = torch.Generator(device=env.device).manual_seed(17)
    _prepare(env, case, g)
    n, dev = env.n_envs, env.device
    snap = _snapshot(env)
    twin = _twin_of(env, case)
    rng = np.random.default_rng(5)
    order = rng.permutation(np.concatenate([np.arange(n), rng.integers(0, n, n // 2)]))
    rows = env.save_envs(_ids(order, dev))
    assert rows.shape == (len(order), env.env_row_bytes) and rows.dtype == torch.uint8 and env.env_row_bytes % 16 == 0
    _assert_same(env, twin, "save changes nothing")
    first = {}
    for j, e in enumerate(order.tolist()):
        first.setdefault(e, j)
    for j, e in enumerate(order.tolist()):          # a repeated env saves the same bytes, padding included
        assert torch.equal(rows[j], rows[first[e]])

    # row_fields: typed views equal the env's tensors at the saved ids
    fields = env.row_fields(rows)
    per_env = {k for k in STATE if getattr(env, k) is not None and (k != "targets" or env.targets.shape[0] == n)}
    assert set(fields) == per_env, (set(fields), per_env)
    sel = torch.from_numpy(order).long().to(dev)
    for name, v in fields.items():
        t = getattr(env, name)
        want = t[:, sel].permute(1, 0, 2) if name == "agent_pos" else t[sel]
        assert v.shape == want.shape and v.dtype == want.dtype, name
        assert torch.equal(_bits(v.contiguous()), _bits(want.contiguous())), name

    # scramble: steps, a masked reset, more steps
    for t in range(3):
        for a in range(max(env.n_agents, 1)):
            env.step(_actions(env, n, g), agent=a)
        if t == 0:
            env.reset(mask=(torch.arange(n, device=dev) % 2 == 0).to(torch.uint8))
    env.check_status()
    back = rng.permutation(n)
    env.load_envs(rows[[first[e] for e in back.tolist()]].contiguous(), env_ids=back)
    for k, v in snap.items():
        assert torch.equal(_bits(getattr(env, k)), _bits(v)), (case.id, k)
    env.check_status()

    # the restored env and the twin agree at every later step, and on every lookahead
    _full_steps(env, twin, g, 3, case.id + " after load")
    _assert_lookahead_all_equal(env, twin, case.agent, case.id)
    env.check_status()


@pytest.mark.parametrize("case", CASES, ids=[c.id for c in CASES])
def test_fork_matches_reference(case):
    env = _make(case)
    g = torch.Generator(device=env.device).manual_seed(19)
    _prepare(env, case, g)
    n, dev = env.n_envs, env.device
    rng = np.random.default_rng(7)
    m = max(2, 2 * n // 3)
    dst = rng.permutation(n)[:m]
    src = rng.integers(0, n, m)
    src[:2] = dst[1], dst[0]                         # overlapping: a dst read as a src, and repeats
    src[2:4] = src[0]
    twin = _twin_of(env, case)
    lib = P._lib.load()
    torch.cuda.synchronize()
    l0 = lib.pcgrl_launch_count()
    env.fork_envs(_ids(src, dev), _ids(dst, dev))
    torch.cuda.synchronize()
    assert lib.pcgrl_launch_count() - l0 == 2
    assert env._synced_steps is None
    _ref_fork(twin, _ids(src, dev), _ids(dst, dev))
    _assert_same(env, twin, case.id + " fork")

    _full_steps(env, twin, g, 2, case.id + " full steps")
    sub = _ids(dst[: max(1, m // 2)], dev)
    acts = _actions(env, sub.numel(), g)
    r1, d1 = env.step(acts, env_ids=sub, agent=case.agent)
    r2, d2 = twin.step(acts, env_ids=sub, agent=case.agent)
    assert torch.equal(r1.view(torch.int32), r2.view(torch.int32)) and torch.equal(d1, d2)
    _assert_same(env, twin, case.id + " subset step")
    assert torch.equal(env.observe(env_ids=dst, agent=case.agent), twin.observe(env_ids=dst, agent=case.agent))
    env.check_status()


SEQ_CASES = [c for c in CASES if c.id in ("binary_narrow16", "binary_wide16", "binary_narrow16_fused", "zelda_turtle",
                                          "binary_holey", "binary_static", "binary_cellular", "sokoban_narrow",
                                          "smb_small", "minecraft_3D_holey_maze", "zelda_turtle_2agents",
                                          "binary_budget", "binary_controls", "binary_u8")]


@pytest.mark.parametrize("case", SEQ_CASES, ids=[c.id for c in SEQ_CASES])
def test_sequence_with_auto_reset(case):
    """Full steps, subset steps, forks, save / load and lookahead in a random order across episode ends, with
    auto_reset; the twin runs without it, resets the same envs by hand and forks with torch indexing.  Every full step
    starts with a quarter of the envs one iteration from the end, so the sequence crosses episode ends."""
    env = _env(case, auto_reset=True)
    env.reset()
    if env.ctrl_metrics:
        env.sample_uniform_targets(torch.Generator(device=env.device).manual_seed(3))
    g = torch.Generator(device=env.device).manual_seed(29)
    _prepare(env, case, g, steps=3)
    twin = _twin_of(env, case, auto_reset=False)
    n, dev = env.n_envs, env.device
    rng = np.random.default_rng(13)
    agents = max(env.n_agents, 1)
    ops = ["full"] * 6 + ["sub"] * 4 + ["fork"] * 4 + ["saveload"] * 3 + ["look"] * 2
    finished = 0
    for i in rng.permutation(len(ops)):
        op = ops[i]
        a = int(rng.integers(0, agents))
        if op == "full":
            # some envs one iteration from the end, on both: forks may have overwritten the ones _prepare left there,
            # and long episodes (smb) would otherwise never end within the sequence
            for e in (env, twin):
                e.iteration[int(i) % 4::4] = e.max_iterations
            acts = _actions(env, n, g)
            env.step(acts, agent=a)
            twin.step(acts, agent=a)
            finished += int(twin.done.sum())
            twin.reset(mask=twin.done)
        elif op == "sub":
            ids = _distinct(n, int(rng.integers(1, n + 1)), rng, dev)
            acts = _actions(env, ids.numel(), g)
            _, done = env.step(acts, env_ids=ids, agent=a)
            twin.step(acts, env_ids=ids, agent=a)
            mask = torch.zeros(n, dtype=torch.uint8, device=dev)
            mask[ids.long()] = done
            twin.reset(mask=mask)
            finished += int(done.sum())
        elif op in ("fork", "saveload"):
            m = int(rng.integers(1, n + 1))
            dst = _distinct(n, m, rng, dev)
            src = _ids(rng.integers(0, n, m), dev)
            if op == "fork":
                env.fork_envs(src, dst)
            else:
                env.load_envs(env.save_envs(src.cpu().numpy()), env_ids=dst.cpu().numpy())
            _ref_fork(twin, src, dst)
        else:
            ids = _distinct(n, n, rng, dev)
            acts = _actions(env, n, g)
            for x, y in zip(env.lookahead(acts, env_ids=ids, agent=a), twin.lookahead(acts, env_ids=ids, agent=a)):
                assert torch.equal(_bits(x), _bits(y)), case.id
        _assert_same(env, twin, f"{case.id} {op}")
        assert env._epoch == twin._epoch
    env.check_status()
    twin.check_status()
    assert finished > 0


CROSS_CASES = [c for c in CASES if c.id in ("binary_narrow16", "binary_controls", "zelda_turtle_2agents", "binary_holey",
                                            "binary_u8", "smb_small", "minecraft_3D_holey_maze", "binary_static")]


def _cross(case, dev_b):
    a = _make(case)
    g = torch.Generator(device=a.device).manual_seed(31)
    _prepare(a, case, g)
    cfg = P.make_config(case.problem, case.rep, map_shape=case.shape, **case.cfg)
    b = P.BatchedPcgrlEnv(cfg, a.n_envs + 13, device=dev_b, seed=11, env_offset=1000, **case.env)
    b.reset()
    assert b.env_row_bytes == a.env_row_bytes
    rng = np.random.default_rng(3)
    m = a.n_envs // 2
    ids_a = _distinct(a.n_envs, m, rng, a.device)
    ids_b = _distinct(b.n_envs, m, rng, b.device)
    b.load_envs(a.save_envs(ids_a).to(b.device), env_ids=ids_b)
    ga, gb = a.row_fields(a.save_envs(ids_a)), b.row_fields(b.save_envs(ids_b))
    for k in ga:
        assert torch.equal(_bits(ga[k].contiguous()), _bits(gb[k].contiguous()).to(a.device)), (case.id, k)
    # B's loaded envs step exactly as A's
    for _ in range(3):
        for ag in range(max(a.n_agents, 1)):
            acts = _actions(a, m, g)
            ra, da = a.step(acts, env_ids=ids_a, agent=ag)
            rb, db = b.step(acts.to(b.device), env_ids=ids_b, agent=ag)
            assert torch.equal(ra.view(torch.int32), rb.view(torch.int32).to(a.device)), case.id
            assert torch.equal(da, db.to(a.device))
    ga, gb = a.row_fields(a.save_envs(ids_a)), b.row_fields(b.save_envs(ids_b))
    for k in ga:
        assert torch.equal(_bits(ga[k].contiguous()), _bits(gb[k].contiguous()).to(a.device)), (case.id, k, "after")
    a.check_status()
    b.check_status()


@pytest.mark.parametrize("case", CROSS_CASES, ids=[c.id for c in CROSS_CASES])
def test_rows_move_between_envs(case):
    """Rows of env A load into env B, another object with another n_envs, env_offset and seed."""
    _cross(case, "cuda:0")


@pytest.mark.parametrize("case", CROSS_CASES[:3], ids=[c.id for c in CROSS_CASES[:3]])
def test_rows_move_between_devices(case):
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU visible")
    _cross(case, "cuda:1")


def test_foreign_and_zero_rows_are_rejected():
    lib = P._lib.load()
    narrow, turtle = _make(CASES[0]), _make(CASES[1])
    assert narrow.env_row_bytes == turtle.env_row_bytes
    dev = narrow.device
    rows = narrow.save_envs([0, 1, 2])
    ids = _ids([0, 1, 2], dev)
    for env, bad in ((turtle, rows), (narrow, torch.zeros_like(rows))):
        snap = _snapshot(env)
        with pytest.raises(ValueError):
            env.load_envs(bad, env_ids=[0, 1, 2])
        # through the C entry point: nothing of those rows is written, status bit 1024
        P._lib.check(lib.pcgrl_load_envs(env._cc, env._st, 1, bad.data_ptr(), ids.data_ptr(), 3, env._stream()), "load")
        for k, v in snap.items():
            assert torch.equal(_bits(getattr(env, k)), _bits(v)), k
        with pytest.raises(ValueError):
            env.check_status()
    # one corrupt header among good rows: only its env is skipped
    twin = _twin_of(narrow, CASES[0])
    mixed = narrow.save_envs([5, 6])
    mixed[1, 3] ^= 1
    P._lib.check(lib.pcgrl_load_envs(narrow._cc, narrow._st, 1, mixed.data_ptr(), _ids([0, 1], dev).data_ptr(), 2,
                                     narrow._stream()), "load")
    with pytest.raises(ValueError):
        narrow.check_status()
    _ref_fork(twin, _ids([5], dev), _ids([0], dev))
    _assert_same(narrow, twin, "mixed")


def test_validation_before_launch():
    lib = P._lib.load()
    env = _make(CASES[0])
    n, dev, S = env.n_envs, env.device, env.env_row_bytes
    rows2 = env.save_envs([0, 1])
    torch.cuda.synchronize()
    l0 = lib.pcgrl_launch_count()
    for ids in ([0, n], [-1, 0], torch.tensor([3, n], device=dev), torch.tensor([-2, 0]), np.array([0.5, 1.0]),
                torch.tensor([1.0, 2.0], device=dev)):
        with pytest.raises(IndexError):
            env.save_envs(ids)
        with pytest.raises(IndexError):
            env.load_envs(rows2, env_ids=ids)
        with pytest.raises(IndexError):
            env.fork_envs(ids, [0, 1])
        with pytest.raises(IndexError):
            env.fork_envs([0, 1], ids)
    for ids in ([1, 1], np.array([2, 2]), torch.tensor([5, 5], device=dev)):
        with pytest.raises(ValueError):
            env.load_envs(rows2, env_ids=ids)
        with pytest.raises(ValueError):
            env.fork_envs([0, 1], ids)
    with pytest.raises(ValueError):
        env.fork_envs([0, 1, 2], [3, 4])
    with pytest.raises(ValueError):
        env.load_envs(rows2, env_ids=[0, 1, 2])
    with pytest.raises(ValueError):
        env.load_envs(torch.zeros((n + 1, S), dtype=torch.uint8, device=dev))
    wide = torch.cat([rows2, rows2], dim=1)
    for bad in (rows2.view(torch.int8), rows2[:, :S - 16], wide[:, :S], rows2.cpu(), rows2.view(-1), rows2.numpy(force=True)):
        with pytest.raises(ValueError):
            env.load_envs(bad, env_ids=[0, 1])
    # nothing to do, nothing launched
    assert env.save_envs([]).shape == (0, S)
    env.load_envs(torch.zeros((0, S), dtype=torch.uint8, device=dev), env_ids=[])
    env.fork_envs([], [])
    torch.cuda.synchronize()
    assert lib.pcgrl_launch_count() == l0
    env.update(torch.zeros(n, dtype=torch.int32, device=dev))
    for call in (lambda: env.save_envs(), lambda: env.load_envs(rows2, env_ids=[0, 1]), lambda: env.fork_envs([0], [1])):
        with pytest.raises(RuntimeError):
            call()
    torch.cuda.synchronize()
    assert lib.pcgrl_launch_count() == l0 + 1           # the update


@pytest.mark.parametrize("case", [CASES[0], CASES[6], CASES[19]], ids=lambda c: c.id)   # cache, generic, 2 agents
def test_device_index_guard(case):
    """Indices the host never checked (== n_envs): save writes a zero row for it, load writes nothing; status bit 512."""
    lib = P._lib.load()
    env = _make(case)
    g = torch.Generator(device=env.device).manual_seed(3)
    _prepare(env, case, g, steps=2)
    n, dev, S = env.n_envs, env.device, env.env_row_bytes
    n_pos = env.agent_pos.shape[0]
    out = torch.full((2, S), 7, dtype=torch.uint8, device=dev)
    P._lib.check(lib.pcgrl_save_envs(env._cc, env._st, n_pos, _ids([1, n], dev).data_ptr(), 2, out.data_ptr(),
                                     env._stream()), "save")
    with pytest.raises(IndexError):
        env.check_status()
    assert torch.equal(out[0], env.save_envs([1])[0]) and int(out[1].long().sum()) == 0
    twin = _twin_of(env, case)
    rows = env.save_envs([2, 3])
    P._lib.check(lib.pcgrl_load_envs(env._cc, env._st, n_pos, rows.data_ptr(), _ids([0, n], dev).data_ptr(), 2,
                                     env._stream()), "load")
    with pytest.raises(IndexError):
        env.check_status()
    _ref_fork(twin, _ids([2], dev), _ids([0], dev))
    _assert_same(env, twin, case.id)


def _beam_search(env, rounds, after_round):
    """The README's beam search, line for line (8 beams per group of 8 envs, ranked by total reward); after every round
    after_round(step rewards, lookahead rewards of the chosen children)."""
    B, G = 8, env.n_envs // 8
    score = torch.zeros(env.n_envs, device=env.device)
    for _ in range(rounds):
        reward, _, _, _ = env.lookahead_all()
        A = reward.shape[1]
        score, top = (score[:, None] + reward).view(G, B * A).topk(B, dim=1)
        parent = (torch.arange(G, device=env.device)[:, None] * B + top // A).flatten()
        env.fork_envs(parent, torch.arange(env.n_envs, device=env.device))
        r, _ = env.step((top % A).flatten().to(torch.int32))
        score = score.flatten()
        after_round(r, reward[parent, (top % A).flatten()])


@pytest.mark.parametrize("rep", ["narrow", "wide"])
def test_beam_search(rep):
    kw = dict(obs_window=(16, 16)) if rep == "wide" else {}
    env = P.BatchedPcgrlEnv(P.make_config("binary", rep, map_shape=(16, 16), **kw), 64, seed=5)
    env.reset()

    def after_round(r, chosen):
        assert torch.equal(env.stats, env.compute_stats(env.maps))
        assert torch.equal(r.view(torch.int32), chosen.view(torch.int32))   # the fork copied what lookahead scored

    _beam_search(env, 6, after_round)
    env.check_status()


def test_large_shard_fork():
    """binary narrow 16x16 at 1 Mi envs: every env forked from a random draw (with repeats) of the shard."""
    case = CASES[0]
    n = 1 << 20
    cfg = P.make_config(case.problem, case.rep, map_shape=case.shape)
    env = P.BatchedPcgrlEnv(cfg, n, seed=3)
    env.reset()
    g = torch.Generator(device=env.device).manual_seed(37)
    for _ in range(3):
        env.step(_actions(env, n, g))
    twin = P.BatchedPcgrlEnv(cfg, n, seed=3)
    twin.load_state_dict(env.state_dict())
    for k in ("reward", "done", "changed"):
        getattr(twin, k).copy_(getattr(env, k))
    src = torch.randint(0, n, (n,), generator=g, device=env.device).to(torch.int32)
    dst = torch.arange(n, dtype=torch.int32, device=env.device)
    env.fork_envs(src, dst)
    _ref_fork(twin, src, dst)
    _assert_same(env, twin, "large fork")
    acts = _actions(env, n, g)
    env.step(acts)
    twin.step(acts)
    _assert_same(env, twin, "large, full step after")
    env.check_status()
