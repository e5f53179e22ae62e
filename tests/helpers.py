"""Shared helpers for the parity tests: dispatch a golden case onto an implementation module."""
import json
import os
import sys
import types

import torch


def _tup(v):
    return tuple(v) if isinstance(v, list) else v


def run_case(impl, op, kwargs, ins, device=None, dtype=None):
    """Call ``impl.<op>`` (oracle or product: same signatures) on a golden case; returns the output.
    For ``*_grad`` ops returns dict(out=..., grad_<name>=...)."""
    kw = dict(kwargs)
    t = {}
    for k, v in ins.items():
        if dtype is not None and v.is_floating_point():
            v = v.to(dtype)
        t[k] = v.to(device) if device is not None else v
    base = op[:-5] if op.endswith("_grad") else op
    cot = t.pop("cot", None)

    def call(tt):
        if base in ("warp_perspective", "warp_affine"):
            return getattr(impl, base)(tt["src"], tt["M"], _tup(kw["dsize"]), mode=kw["mode"], padding_mode=kw["padding_mode"],
                                       align_corners=kw["align_corners"], fill_value=tt.get("fill_value"))
        if base == "remap":
            return impl.remap(tt["image"], tt["map_x"], tt["map_y"], **kw)
        if base == "filter2d":
            return impl.filter2d(tt["input"], tt["kernel"], **kw)
        if base == "filter2d_separable":
            return impl.filter2d_separable(tt["input"], tt["kernel_x"], tt["kernel_y"], **kw)
        if base == "gaussian_blur2d":
            sigma = tt["sigma"] if "sigma" in tt else _tup(kw["sigma"])
            return impl.gaussian_blur2d(tt["input"], _tup(kw["kernel_size"]), sigma, kw["border_type"], kw["separable"])
        raise KeyError(op)

    if not op.endswith("_grad"):
        return call(t)
    wrt = [k for k in t if k != "fill_value"]
    leaves = dict(t)
    for k in wrt:
        leaves[k] = t[k].clone().requires_grad_(True)
    out = call(leaves)
    grads = torch.autograd.grad((out * cot).sum(), [leaves[k] for k in wrt], allow_unused=True)
    res = {"out": out.detach()}
    for k, g in zip(wrt, grads):
        res[f"grad_{k}"] = g if g is not None else torch.zeros_like(t[k])
    return res


def rel_l2(a, b):
    a = a.double().flatten()
    b = b.double().flatten()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def run_family_case(impl, op, kwargs, ins, device=None, dtype=None):
    """Golden cases of tests/golden/family.npz: every tensor is passed by keyword (the names are the
    reference's parameter names), lists in ``kwargs`` become tuples.  ``*_grad`` ops return
    dict(out=..., grad_<name>=...) for sum(out * cot)."""
    kw = {k: _tup(v) for k, v in kwargs.items()}
    t = {}
    for k, v in ins.items():
        if dtype is not None and v.is_floating_point():
            v = v.to(dtype)
        t[k] = v.to(device) if device is not None else v
    fn = getattr(impl, op[:-5] if op.endswith("_grad") else op)
    if not op.endswith("_grad"):
        return fn(**t, **kw)
    return t, fn, kw


def family_grads(impl, op, kwargs, ins, outs, device=None, dtype=None):
    t, fn, kw = run_family_case(impl, op, kwargs, ins, device, dtype)
    wrt = [k[5:] for k in outs if k.startswith("grad_")]
    leaves = {k: (v.clone().requires_grad_(True) if k in wrt else v) for k, v in t.items()}
    out = fn(**leaves, **kw)
    cot = outs["cot"].to(out)
    grads = torch.autograd.grad((out * cot).sum(), [leaves[k] for k in wrt])
    res = {"out": out.detach()}
    res.update({f"grad_{k}": g for k, g in zip(wrt, grads)})
    return res


def reference_package(monkeypatch):
    """The reference's ``kornia`` package as tests/golden/install.json records it (make_golden_install.py): every module,
    its attributes that name other modules of the package, and the functions ``kornia_b200.install()`` rebinds, bound
    under the same names in the same modules as in the reference, one stand-in object per function.  The modules are in
    ``sys.modules`` until the test ends.  Returns the top-level package and the recorded (module name, function name)
    bindings."""
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "install.json")) as f:
        rec = json.load(f)

    def stand_in(name):
        def fn(*args, **kwargs):
            raise AssertionError(f"the reference's {name} was called")

        fn.__name__ = fn.__qualname__ = name
        return fn

    originals = {name: stand_in(name) for name in rec["defining"]}
    mods = {name: types.ModuleType(name) for name in rec["modules"]}
    for name, m in mods.items():
        parent, _, leaf = name.rpartition(".")
        if parent:
            setattr(mods[parent], leaf, m)
        monkeypatch.setitem(sys.modules, name, m)
    # after the submodule attributes: ``from .sobel import sobel`` leaves the function, not the module, in kornia.filters
    for name, r in rec["modules"].items():
        for attr, target in r["aliases"].items():
            setattr(mods[name], attr, mods[target])
        for fn in r["binds"]:
            setattr(mods[name], fn, originals[fn])
    return mods["kornia"], [(m, fn) for m, r in rec["modules"].items() for fn in r["binds"]]
