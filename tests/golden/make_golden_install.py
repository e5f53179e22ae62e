"""Record the import graph of the reference package that ``kornia_b200.install()`` patches: tests/golden/install.json.

    python tests/golden/make_golden_install.py <kornia 0.9.0rc1 checkout>

The reference is imported from the checkout (an empty stub stands in for the ``kornia_rs`` wheel, as in
make_golden.py) with the modules the install tests name.  For every ``kornia.*`` module the file lists which of the
functions ``install()`` rebinds it holds -- the very object its defining module exports -- and the attributes that
refer to another module of the package (``kornia.losses.ssim.metrics`` is ``kornia.metrics``).  The install tests
rebuild the package from this record, so they check ``install()`` against the reference's importers without the
checkout.
"""
from __future__ import annotations

import json
import os
import sys
import tempfile
import types

HERE = os.path.dirname(os.path.abspath(__file__))

# name -> defining module, as in kornia_b200.install()
DEFINING = {
    "warp_perspective": "geometry.transform.imgwarp",
    "warp_affine": "geometry.transform.imgwarp",
    "remap": "geometry.transform.imgwarp",
    "filter2d": "filters.filter",
    "filter2d_separable": "filters.filter",
    "gaussian_blur2d": "filters.gaussian",
    "get_perspective_transform": "geometry.transform.imgwarp",
    "spatial_gradient": "filters.sobel",
    "sobel": "filters.sobel",
    "ssim": "metrics.ssim",
}
IMPORTED = [
    "kornia.augmentation._2d.geometric.perspective",
    "kornia.augmentation._2d.intensity.gaussian_blur",
    "kornia.geometry.transform.affwarp",
    "kornia.geometry.transform.crop2d",
    "kornia.geometry.transform.pyramid",
    "kornia.geometry.calibration.undistort",
    "kornia.filters.unsharp",
]


def main(checkout: str) -> None:
    stub = tempfile.mkdtemp(prefix="kornia_rs_stub_")
    open(os.path.join(stub, "kornia_rs.py"), "w").close()
    sys.path[:0] = [stub, checkout]
    import importlib

    for name in ["kornia"] + IMPORTED:
        importlib.import_module(name)
    orig = {n: getattr(sys.modules["kornia." + m], n) for n, m in DEFINING.items()}
    record = {}
    for name in sorted(k for k, m in sys.modules.items() if m is not None and (k == "kornia" or k.startswith("kornia."))):
        attrs = vars(sys.modules[name])
        aliases = {a: v.__name__ for a, v in sorted(attrs.items())
                   if isinstance(v, types.ModuleType) and v.__name__.split(".")[0] == "kornia" and v.__name__ != f"{name}.{a}"}
        record[name] = {"binds": [n for n in DEFINING if attrs.get(n) is orig[n]], "aliases": aliases}
    path = os.path.join(HERE, "install.json")
    lines = [f"{json.dumps(k)}: {json.dumps(v, sort_keys=True)}" for k, v in record.items()]  # one module per line
    with open(path, "w") as f:
        f.write('{"defining": ' + json.dumps(DEFINING) + ',\n"modules": {\n' + ",\n".join(lines) + "\n}}\n")
    print(f"{path}: {len(record)} modules, {sum(len(r['binds']) for r in record.values())} bindings")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(sys.argv[1])
