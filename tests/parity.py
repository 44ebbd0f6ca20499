"""The 1e-5 relative contract of BASELINE.json's north_star, written down once.

``close(name, got, want)`` requires  |got - want| <= RTOL * max(|want|, FLOOR * max|want|)  for every element:
a RELATIVE bound with an explicit denominator floor instead of an absolute ``atol``.  The floor exists because
gradients and losses are sums with cancellation: an element whose magnitude is below 1 % of the tensor's largest
carries the absolute rounding error of the large terms it is made of (the reference's own fp32 sums, evaluated
in another order, differ by that much), so its error is measured against FLOOR * max|want|.  ``scale=`` replaces
max|want| where the result is a DIFFERENCE of larger operands (the DQN / M-DQN gradient w * clamp(q - T): one ulp
of a target T ~ 10 is 1e-6, which is 1e-4 of a gradient of 0.01): the magnitude of those operands.  Every call also
records the worst relative error it saw; with A0_PARITY_RECORD=<file> set (profiles/parity_r02.json holds such a
record), the session writes them there."""
import json
import os

import numpy as np

RTOL = 1e-5
FLOOR = 1e-2
RECORD = {}


def _np(x):
    try:
        import torch
        if isinstance(x, torch.Tensor):
            return x.detach().cpu().numpy()
    except ImportError:
        pass
    return np.asarray(x)


def rel_err(got, want, floor=FLOOR, scale=None):
    got = _np(got).astype(np.float64)
    want = np.asarray(_np(want), dtype=np.float64)
    if scale is None:
        scale = float(np.abs(want).max()) if want.size else 0.0
    den = np.maximum(np.abs(want), max(floor * scale, 1e-30))
    return np.abs(got - want) / den, scale


def close(name, got, want, rtol=RTOL, floor=FLOOR, scale=None):
    err, scale = rel_err(got, want, floor, scale)
    worst = float(err.max()) if err.size else 0.0
    strict, _ = rel_err(got, want, 1e-3, scale)
    rec = RECORD.setdefault(name, {"max_rel_err": 0.0, "max_rel_err_floor_1e-3": 0.0, "elements": 0, "scale": 0.0})
    rec["max_rel_err"] = max(rec["max_rel_err"], worst)
    rec["max_rel_err_floor_1e-3"] = max(rec["max_rel_err_floor_1e-3"], float(strict.max()) if strict.size else 0.0)
    rec["elements"] += int(err.size)
    rec["scale"] = max(rec["scale"], scale)
    assert _np(got).shape == _np(want).shape, f"{name}: shape {_np(got).shape} vs {_np(want).shape}"
    assert np.isfinite(_np(got)).all(), f"{name}: non-finite values"
    assert worst <= rtol, f"{name}: worst relative error {worst:.3e} > {rtol:.0e} (denominator floor {floor:g} x max|ref| = {floor * scale:.3e})"


def dump(path):
    """Write the record as JSON to ``path``."""
    if not RECORD:
        return
    doc = {"contract": f"|got-ref| <= {RTOL:g} * max(|ref|, {FLOOR:g} * max|ref|) per element (tests/parity.py)",
           "note": "max_rel_err_floor_1e-3 is the same measure with a 1e-3 denominator floor, for information",
           "worst": {k: {kk: (float(f"{vv:.3e}") if isinstance(vv, float) else vv) for kk, vv in v.items()} for k, v in sorted(RECORD.items())}}
    if os.path.exists(path):      # a partial run (-k ...) keeps the other entries
        try:
            old = json.load(open(path))["worst"]
            doc["worst"] = dict(sorted({**old, **doc["worst"]}.items()))
        except Exception:
            pass
    try:
        os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
        with open(path, "w") as f:
            json.dump(doc, f, indent=1)
            f.write("\n")
    except OSError:
        pass
