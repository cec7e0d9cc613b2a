"""Drop-in check of the operator surface: the public functions take exactly the reference's parameters, in the
reference's order.  The reference's side (nerfstudio-project/gsplat v1.6.0, parameter lists parsed from its sources
with `ast`) is stored in tests/golden/ref_signatures.json."""
import ast
import json
import os

import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
REF = json.load(open(os.path.join(ROOT, "tests", "golden", "ref_signatures.json")))


def _params(path, fn):
    tree = ast.parse(open(path).read())
    for n in ast.walk(tree):
        if isinstance(n, ast.FunctionDef) and n.name == fn:
            a = n.args
            return [x.arg for x in a.posonlyargs + a.args + a.kwonlyargs], len(a.defaults)
    raise AssertionError(f"{fn} not found in {path}")


@pytest.mark.parametrize(
    "fn,ref_file,our_file",
    [
        ("rasterization", "rendering.py", "rendering.py"),
        ("fully_fused_projection", "cuda/_wrapper.py", "ops.py"),
        ("spherical_harmonics", "cuda/_wrapper.py", "ops.py"),
        ("isect_tiles", "cuda/_wrapper.py", "ops.py"),
        ("isect_offset_encode", "cuda/_wrapper.py", "ops.py"),
        ("rasterize_to_pixels", "cuda/_wrapper.py", "ops.py"),
        ("quat_scale_to_covar_preci", "cuda/_wrapper.py", "ops.py"),
        ("adam", "cuda/_wrapper.py", "ops.py"),
        ("compute_relocation", "relocation.py", "ops.py"),
        ("all_gather_int32", "distributed.py", "distributed.py"),
        ("all_to_all_int32", "distributed.py", "distributed.py"),
        ("all_gather_tensor_list", "distributed.py", "distributed.py"),
        ("all_to_all_tensor_list", "distributed.py", "distributed.py"),
        ("cli", "distributed.py", "distributed.py"),
    ],
)
def test_same_parameters_as_reference(fn, ref_file, our_file):
    entry = REF["functions"][fn]
    assert entry["file"] == "gsplat/" + ref_file
    ref, ref_defaults = entry["params"], entry["n_defaults"]
    ours, our_defaults = _params(os.path.join(ROOT, "gsplat_b200", our_file), fn)
    assert ours == ref, f"{fn}: parameters differ\n reference: {ref}\n ours:      {ours}"
    assert our_defaults == ref_defaults, f"{fn}: number of defaulted parameters differs"


def test_rasterization_defaults_match_reference():
    def defaults(path):
        tree = ast.parse(open(path).read())
        for n in ast.walk(tree):
            if isinstance(n, ast.FunctionDef) and n.name == "rasterization":
                names = [x.arg for x in n.args.args]
                d = n.args.defaults
                return {k: ast.unparse(v) for k, v in zip(names[len(names) - len(d):], d)}

    ref = REF["rasterization_defaults"]
    ours = defaults(os.path.join(ROOT, "gsplat_b200", "rendering.py"))
    # rolling_shutter: the reference's default is its RollingShutterType.GLOBAL enum member; ours is None (= global)
    diff = {k: (ref[k], ours.get(k)) for k in ref if ref[k] != ours.get(k) and k != "rolling_shutter"}
    assert not diff, diff
