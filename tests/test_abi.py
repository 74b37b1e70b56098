"""CPU tests of the boundary: the C-ABI library loads without a GPU and exports exactly the symbols
include/tmf.h declares; the Python surface mirrors the reference's classes and signatures."""
import ast
import ctypes
import importlib
import inspect
import json
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "tmf.h")
# a checkout of the original TeAMOFlow project (not part of this repository): the surface checks against its source run
# only where one is given
REF_ROOT = os.environ.get("TMF_REFERENCE_ROOT")
REF = os.path.join(REF_ROOT, "src", "teamoflow", "mf") if REF_ROOT else None
SURFACE = os.path.join(ROOT, "tests", "golden", "plugin_surface.json")
MODULES = ["matrix_factorization", "loss_graphs", "embedding_graphs", "initializer_graphs", "input_utils", "predict_graphs", "utils"]


def _header_symbols():
    src = open(HEADER).read()
    return sorted(set(re.findall(r"^TMF_API [a-z_ *0-9]+?(tmf_[a-z0-9_]+)\(", src, flags=re.M)))


def test_library_loads_and_exports_every_declared_symbol():
    from teamoflow_b200 import _abi
    syms = _header_symbols()
    assert len(syms) >= 30
    h = ctypes.CDLL(_abi.LIB_PATH)
    for s in syms:
        assert hasattr(h, s), f"{s} declared in tmf.h but not exported"
    assert sorted(_abi.SIGNATURES) == syms, "ctypes SIGNATURES out of sync with include/tmf.h"
    assert _abi.lib().tmf_abi_version() == 1


def test_size_queries_need_no_gpu():
    from teamoflow_b200 import _abi
    assert _abi.query("tmf_reduce_ws_bytes") > 0
    assert _abi.query("tmf_spmm_ws_bytes", 1000, 64) > 0
    assert _abi.query("tmf_transpose_ws_bytes", 1000) > 0
    assert _abi.query("tmf_score_topk_ws_bytes", 1000, 1000, 32, 10) > 0


def test_compute_without_gpu_fails_loudly():
    import torch
    from teamoflow_b200 import _abi
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from teamoflow_b200.mf.initializer_graphs import NormalInitializer
    with pytest.raises(_abi.TmfError):
        NormalInitializer().initialize_weights(4, 2)


def _ref_signatures(path):
    """{class: {method: [arg names]}} and {function: [arg names]} parsed from reference source (no import: TF absent)."""
    tree = ast.parse(open(path).read())
    classes, funcs = {}, {}
    for node in tree.body:
        if isinstance(node, ast.ClassDef):
            classes[node.name] = {f.name: ([a.arg for a in f.args.args], len(f.args.defaults))
                                  for f in node.body if isinstance(f, ast.FunctionDef)}
        elif isinstance(node, ast.FunctionDef):
            funcs[node.name] = ([a.arg for a in node.args.args], len(node.args.defaults))
    return classes, funcs


def _surface(module):
    """``_ref_signatures`` of teamoflow_b200/mf/<module>.py in JSON form: every class, method and function the file
    defines (private ones included), each with its parameter names and number of defaults."""
    classes, funcs = _ref_signatures(os.path.join(ROOT, "teamoflow_b200", "mf", f"{module}.py"))
    return json.loads(json.dumps({"classes": classes, "functions": funcs}))


@pytest.mark.parametrize("module", MODULES)
def test_plugin_surface_is_the_recorded_one(module):
    """This package's own surface, extracted exactly as test_plugin_surface_matches_reference extracts the reference's,
    against tests/golden/plugin_surface.json.  It pins the package against unintended change, not against the reference;
    a deliberate change of the surface rewrites the file (``python tests/test_abi.py``), which then shows in the diff."""
    assert _surface(module) == json.load(open(SURFACE))[module]


@pytest.mark.skipif(not (REF and os.path.isdir(REF)), reason="needs TMF_REFERENCE_ROOT: a checkout of the original TeAMOFlow source")
@pytest.mark.parametrize("module", MODULES)
def test_plugin_surface_matches_reference(module):
    ours = importlib.import_module(f"teamoflow_b200.mf.{module}")
    classes, funcs = _ref_signatures(os.path.join(REF, f"{module}.py"))
    for cname, methods in classes.items():
        cls = getattr(ours, cname)
        for mname, (args, _) in methods.items():
            sig = inspect.signature(getattr(cls, mname))
            names = [p for p in sig.parameters if p not in ("self", "cls")]
            args = [a for a in args if a not in ("self", "cls")]
            assert names[:len(args)] == args, f"{module}.{cname}.{mname}: {names} vs reference {args}"
    for fname, (args, _) in funcs.items():
        names = list(inspect.signature(getattr(ours, fname)).parameters)
        assert names[:len(args)] == args, f"{module}.{fname}: {names} vs reference {args}"


def test_constructor_defaults_match_reference():
    from teamoflow_b200.mf.matrix_factorization import MatrixFactorization
    from teamoflow_b200.mf import embedding_graphs as e, loss_graphs as l, initializer_graphs as i
    m = MatrixFactorization(3)
    assert isinstance(m.user_repr_graph, e.LinearEmbedding) and isinstance(m.loss_graph, l.MSELoss)
    assert isinstance(m.user_weight_graph, i.NormalInitializer)
    assert m.random_ind is None and m.n_samples is None
    m2 = MatrixFactorization(3, n_items=101)
    assert m2.n_samples == 50  # n_items // 2, ref:68-69
    sig = inspect.signature(MatrixFactorization.fit)
    assert sig.parameters["lr"].default == 1e-2
    assert inspect.signature(MatrixFactorization.recall_at_k).parameters["k"].default == 10


if __name__ == "__main__":
    with open(SURFACE, "w") as f:
        json.dump({m: _surface(m) for m in MODULES}, f, indent=1, sort_keys=True)
        f.write("\n")
    print("wrote", SURFACE)
