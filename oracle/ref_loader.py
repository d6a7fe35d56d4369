"""Import the UNMODIFIED reference modules from the original project's ``src/``
directory, named by the environment variable ``TM_REFERENCE_SRC``.

Oracle / test infrastructure only, used by ``make_golden.py`` alone: the
reference is not part of this repository, and the tests compare against the
fixtures it generated.  ``available()`` says whether it is there.

* ``ref_model()`` -> the reference ``model.py`` module (needs the inert
  ``dgl.function`` stub under ``oracle/dgl_stub``);
* ``ref_unet()``  -> the reference ``Unet.py`` module;
* ``ref_parser_funcs()`` -> ``cal_topo_level`` and ``find_critical_path``
  compiled from the reference's own source text
  (``verilog_parser_asap7.py:1433-1517``).  The file cannot be imported
  (pyverilog + ``../rawdata/*.json`` at import time), so the two ``def``s are
  cut out of its AST at run time and executed as is; nothing is copied into
  this repository.
"""
import ast
import importlib.util
import os
import sys

REF_SRC = os.environ.get("TM_REFERENCE_SRC", "")
_HERE = os.path.dirname(os.path.abspath(__file__))
_cache = {}


def available():
    return bool(REF_SRC) and os.path.isfile(os.path.join(REF_SRC, "model.py"))


def _load(name, filename):
    if name in _cache:
        return _cache[name]
    stub = os.path.join(_HERE, "dgl_stub")
    had_dgl = sys.modules.get("dgl")
    sys.path.insert(0, stub)
    try:
        spec = importlib.util.spec_from_file_location(name, os.path.join(REF_SRC, filename))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        sys.path.remove(stub)
        if had_dgl is None:                      # do not leave the stub importable as `dgl`
            for k in [k for k in sys.modules if k == "dgl" or k.startswith("dgl.")]:
                del sys.modules[k]
    _cache[name] = mod
    return mod


def ref_model():
    return _load("_reference_model", "model.py")


def ref_unet():
    return _load("_reference_unet", "Unet.py")


def ref_parser_funcs():
    if "parser" in _cache:
        return _cache["parser"]
    path = os.path.join(REF_SRC, "verilog_parser_asap7.py")
    tree = ast.parse(open(path).read(), path)
    wanted = {"cal_topo_level", "find_critical_path"}
    defs = [n for n in ast.walk(tree) if isinstance(n, ast.FunctionDef) and n.name in wanted]
    assert {d.name for d in defs} == wanted
    ns = {}
    exec(compile(ast.Module(body=defs, type_ignores=[]), path, "exec"), ns)
    _cache["parser"] = (ns["cal_topo_level"], ns["find_critical_path"])
    return _cache["parser"]
