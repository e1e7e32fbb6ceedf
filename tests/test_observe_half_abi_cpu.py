"""CPU: the float16 / bfloat16 observation kinds (pcgrl_obs_args.out_kind 5 and 6) pass the argument checks of
pcgrl_lookahead_obs, target planes included, and every other kind outside 0..3 is still refused before any CUDA call."""
from control_pcgrl_b200 import _lib
from tests.test_abi_cpu import _cfg, _lib_err
from tests.test_lookahead_obs_abi_cpu import _call, _obs, _state


def test_half_kinds_pass_the_lookahead_obs_checks():
    lib = _lib.load()
    c = _cfg()
    assert lib.pcgrl_config_check(c) == 0
    st = _state()
    for kind in (5, 6):
        assert _call(lib, c, st, 0, _obs(out_kind=kind)) == 0, kind
        ctrl = _obs(out_kind=kind)
        ctrl.n_ctrl, ctrl.ctrl_idx[0], ctrl.ctrl_range[0] = 1, 0, 128.0
        assert _call(lib, c, st, 0, ctrl) == 0, kind         # target planes are fine in half precision
        assert _call(lib, c, st, 0, _obs(crop=0, dims=(16, 16), out_kind=kind)) == 0, kind


def test_other_kinds_are_refused():
    lib = _lib.load()
    c = _cfg()
    assert lib.pcgrl_config_check(c) == 0
    st = _state()
    E = _lib_err("PCGRL_E_ARG")
    for kind in (4, 7, -1, 255):
        assert _call(lib, c, st, 0, _obs(out_kind=kind)) == E, kind
        assert b"out_kind" in lib.pcgrl_last_error()
    # uint8 one-hot and tile codes still refuse target planes
    for kind in (0, 3):
        o = _obs(out_kind=kind)
        o.n_ctrl, o.ctrl_idx[0] = 1, 0
        assert _call(lib, c, st, 0, o) == E, kind
        assert b"target planes" in lib.pcgrl_last_error()
