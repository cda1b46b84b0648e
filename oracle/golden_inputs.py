"""Inputs of the reference fixtures (tests/golden/*.npz), regenerated from fixed torch CPU seeds.

A fixture stores the reference's outputs, and per case a JSON string `<case>/inputs` in place of the input arrays:
the recipe that made them, its arguments and the sha256 of every input.  `pack` (oracle/make_golden.py) writes that
entry, `unpack` (tests/conftest.py) puts the inputs back and fails if one of them no longer comes out bit for bit.
"""
import hashlib
import json

import numpy as np
import torch


def factors(v_shape, w_shape, h_shape, floor=0.0, offset=0.0, scale=1.0, z=False):
    """V = rand(v_shape) rounded to bf16-representable values (then clamped to `floor`, shifted by `offset`, scaled by
    `scale`) from seed 0; W0 = |randn(w_shape)|, H0 = |randn(h_shape)| and, with `z`, Z0 = rand(R) + 0.1 from seed 1."""
    torch.manual_seed(0)
    V = torch.rand(*v_shape).bfloat16().float()
    if floor > 0:
        V = V.clamp_min(floor)
    if offset:
        V = V + offset
    if scale != 1:
        V = V * scale
    torch.manual_seed(1)
    out = dict(V=V, W0=torch.randn(*w_shape).abs(), H0=torch.randn(*h_shape).abs())
    if z:
        out["Z0"] = torch.rand(w_shape[1]) + 0.1
    return out


def thresholded(shape, rank, keep_above, seeds=(0, 1), bf16=False, empty_row=None, empty_col=None):
    """A sparse-looking target: rand(shape) (optionally bf16-rounded) with every entry <= keep_above set to zero, and an
    optional empty row and column; W0, H0 = |randn| of `rank` columns from the second seed."""
    torch.manual_seed(seeds[0])
    V = torch.rand(*shape)
    if bf16:
        V = V.bfloat16().float()
    V = torch.where(V > keep_above, V, torch.zeros(()))
    if empty_row is not None:
        V[empty_row] = 0
    if empty_col is not None:
        V[:, empty_col] = 0
    torch.manual_seed(seeds[1])
    return dict(V=V, W0=torch.randn(shape[1], rank).abs(), H0=torch.randn(shape[0], rank).abs())


def proj_slices(shape, negative_row=False):
    """X = |randn(shape)| + 0.01 from seed 3, optionally with row 1 redrawn from randn (negative entries included)."""
    torch.manual_seed(3)
    X = torch.randn(*shape).abs() + 0.01
    if negative_row:
        X[1] = torch.randn(shape[1])
    return dict(X=X)


RECIPES = {f.__name__: f for f in (factors, thresholded, proj_slices)}


def digest(a):
    a = np.ascontiguousarray(a)
    return f"{a.dtype.str}{list(a.shape)}:" + hashlib.sha256(a.tobytes()).hexdigest()


def pack(flat, name, recipe, **args):
    """Replace the input arrays of case `name` in `flat` ({"<case>/<field>": array}) by the `<case>/inputs` entry.
    The recipe must reproduce every one of them exactly."""
    spec = {"recipe": recipe, "args": args, "sha256": {}}
    for k, t in RECIPES[recipe](**args).items():
        stored = flat.pop(f"{name}/{k}")
        spec["sha256"][k] = digest(t.numpy())
        assert digest(stored) == spec["sha256"][k], f"{name}/{k}: {recipe}({args}) does not reproduce the stored input"
    flat[f"{name}/inputs"] = np.array(json.dumps(spec, sort_keys=True))


def unpack(flat):
    """The inverse of `pack` over every case of a fixture: returns a new dict with the input arrays in place."""
    out = {}
    for key, v in flat.items():
        if not key.endswith("/inputs"):
            out[key] = v
            continue
        name = key[: -len("/inputs")]
        spec = json.loads(str(v))
        for k, t in RECIPES[spec["recipe"]](**spec["args"]).items():
            a = t.numpy()
            if digest(a) != spec["sha256"][k]:
                raise RuntimeError(f"{name}/{k} no longer regenerates bit for bit from {spec['recipe']}({spec['args']})")
            out[f"{name}/{k}"] = a
    return out
