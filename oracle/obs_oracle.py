"""Vectorised reference observation: Cropped + OneHotEncoding + ToImage + ControlWrapper's target planes (+ the
'static_builds' plane) for a whole batch at once, in torch on any device.

It restates the per-env loop functions of pcgrl_oracle (cropped_onehot, full_onehot, static_builds_crop,
target_channels), which tests/test_obs_oracle_cpu.py pins it on, so that the observation writer (csrc/observe.cu)
can be compared with the reference semantics at the batch sizes where its grouping and trip logic matter:

- the crop reads map cell pos + o - window // 2 for window cell o (odd windows are off-centre by that rule);
- behind a crop channel 0 means out of bounds and tile t is channel t + 1; without a crop there is no extra channel;
  onehot=False writes that channel index (the tile code) as the only map channel;
- the 2 * n_ctrl control planes come first: (target, or the midpoint of a (lo, hi) target) / range, then
  metric / range, computed in float64 and cast to the output dtype;
- the static plane is the bordered frozen-tile mask (border = 1) cropped like the map, 0 beyond the border.

Index arithmetic with a validity mask, no padding, so that the off-centre odd-window case is explicit.
"""
from __future__ import annotations

import torch


def _crop_index(pos, window, shape):
    """(src [ndim] of [N, *window] long, ok [N, *window] bool): the cell window cell o reads, and whether it lies
    inside `shape`."""
    n, nd = pos.shape[0], len(window)
    dev = pos.device
    axes = torch.meshgrid(*[torch.arange(w, device=dev) for w in window], indexing="ij")
    src, ok = [], torch.ones((n, *window), dtype=torch.bool, device=dev)
    for i in range(nd):
        s = pos[:, i].long().view(n, *([1] * nd)) + axes[i] - window[i] // 2
        ok = ok & (s >= 0) & (s < shape[i])
        src.append(s)
    return src, ok


def _gather(vals, src, ok, shape):
    """vals [N, *shape] sampled at src where ok (0 elsewhere), as long."""
    n = vals.shape[0]
    flat = torch.zeros_like(src[0])
    for i, s in enumerate(src):
        flat = flat * shape[i] + s.clamp(0, shape[i] - 1)
    got = vals.reshape(n, -1).long().gather(1, flat.reshape(n, -1)).view(flat.shape)
    return torch.where(ok, got, torch.zeros_like(got))


def observe(maps, pos=None, window=None, crop=True, n_tiles=2, static_mask=None, targets=None, stats=None,
            ctrl_idx=(), ctrl_range=(), dtype=torch.float32, onehot=True):
    """[N, *window, channels] (channels last; window = the map shape without a crop).

    maps [N, *shape] tile codes; pos [N, >= ndim] crop centres (only with crop); static_mask [N, *shape] frozen
    tiles (only with crop); targets [N or 1, K, 2] float64 ((value, NaN) or (lo, hi)); stats [N, K]; ctrl_idx /
    ctrl_range: the stat column and |hi - lo| of each controlled metric."""
    maps = torch.as_tensor(maps)
    n, shape = maps.shape[0], tuple(int(d) for d in maps.shape[1:])
    nd = len(shape)
    n_ctrl = len(ctrl_idx)
    if len(ctrl_range) != n_ctrl:
        raise ValueError("one range per controlled metric")
    if n_ctrl and (dtype == torch.uint8 or not onehot):
        raise ValueError("control planes are fractional: they need a float one-hot observation")
    if static_mask is not None and not crop:
        raise ValueError("the static plane is only observed behind a crop")
    if crop:
        window = tuple(int(w) for w in window)
        if len(window) != nd:
            raise ValueError("one window extent per map axis")
        src, ok = _crop_index(torch.as_tensor(pos, device=maps.device), window, shape)
        code = _gather(maps, src, ok, shape) + ok.long()
        n_map_ch = n_tiles + 1
    else:
        window = shape
        code = maps.long()
        n_map_ch = n_tiles
    planes = []
    if n_ctrl:
        trg = torch.as_tensor(targets, device=maps.device).to(torch.float64).expand(n, -1, -1)
        st = torch.as_tensor(stats, device=maps.device)
        for k, r in zip(ctrl_idx, ctrl_range):
            lo, hi = trg[:, k, 0], trg[:, k, 1]
            t = torch.where(torch.isnan(hi), lo, (lo + hi) / 2)
            # divide by a tensor: on CUDA, torch divides by a Python scalar as a multiply by its reciprocal, which is
            # not the correctly rounded quotient the reference (and the kernel) compute
            rng = torch.full((n,), float(r), dtype=torch.float64, device=maps.device)
            for v in (t / rng, st[:, k].to(torch.float64) / rng):
                planes.append(v.view(n, *([1] * nd)).expand(n, *window).to(dtype))
    if onehot:
        planes += list(torch.nn.functional.one_hot(code, n_map_ch).to(dtype).unbind(-1))
    else:
        planes.append(code.to(dtype))
    if static_mask is not None:
        sm = torch.as_tensor(static_mask, device=maps.device) != 0
        bordered = torch.ones((n, *[d + 2 for d in shape]), dtype=torch.bool, device=maps.device)
        bordered[(slice(None),) + tuple(slice(1, -1) for _ in shape)] = sm
        bsrc, bok = _crop_index(torch.as_tensor(pos, device=maps.device), window, [d + 2 for d in shape])
        planes.append(_gather(bordered, bsrc, bok, [d + 2 for d in shape]).to(dtype))
    return torch.stack(planes, dim=-1)
