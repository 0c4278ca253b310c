"""The compiled pybind11 module `libgraphvite` over the C ABI (graphvite_b200/csrc/pybind/libgraphvite.cpp ->
graphvite_b200/pybind/libgraphvite.so): the surface a reference maintainer gets when `src/graphvite.cu`'s classes are
swapped for libgv_b200.  Checked on CPU against what tests/pybind_probe.py printed for the UNMODIFIED reference
module (recorded in tests/golden/reference_pybind_probe.json): same submodules and class names, the same argument
names / order / defaults of every solver method (parsed from both modules' docstrings), the same optimizer objects,
and a Graph that loads, maps and saves the same bytes.  Training through this module runs on the GPU box
(tests/test_gpu_x_pybind.py)."""
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUR_PATH = os.path.join(ROOT, "graphvite_b200", "pybind", "libgraphvite.so")
RECORDED = os.path.join(ROOT, "tests", "golden", "reference_pybind_probe.json")
TOY = os.path.join(ROOT, "tests", "golden", "toy_graph.txt")


def probe(path):
    """tests/pybind_probe.py in its own interpreter (two modules called `libgraphvite` cannot share one)"""
    done = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "pybind_probe.py"), path],
                          stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert done.returncode == 0, done.stderr[-3000:]
    return json.loads(done.stdout.strip().splitlines()[-1])


@pytest.fixture(scope="module")
def ours():
    """make sure OUR module is built (it is only ever loaded in a child interpreter, tests/pybind_probe.py: another
    test of the same session may already have imported the reference's module under the same name)"""
    if not os.path.exists(OUR_PATH):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "graphvite_b200", "csrc"), "pybind"],
                              stdout=subprocess.DEVNULL)
    return OUR_PATH


@pytest.fixture(scope="module")
def mine(ours):
    return probe(OUR_PATH)


@pytest.fixture(scope="module")
def theirs():
    """tests/pybind_probe.py's output for the reference's module (python tests/pybind_probe.py
    oracle/_ref/libgraphvite.so, built by `make -C oracle ref`)"""
    with open(RECORDED) as fin:
        return json.load(fin)


def public(obj):
    return {name for name in dir(obj) if not name.startswith("_")}


def same_default(theirs, mine):
    if theirs is None or mine is None:
        return theirs is None and mine is None
    if theirs == "auto":
        return mine.startswith("0") or "optimizer Default" in mine  # kAuto, or the default Optimizer(auto) object
    if theirs in ("True", "False"):
        return mine == theirs
    if theirs[0] in "'\"":
        return mine.strip("'\"") == theirs[1:-1]
    return float(theirs) == float(mine)


def test_module_layout(mine):
    assert mine["backend"] == "libgv_b200"
    for dim in (32, 64, 96, 128, 256, 512):
        assert "GraphSolver_%d_f_j" % dim in mine["solver"]  # src/graphvite.cu:52-59
    for dim in (32, 64, 96, 128, 256, 512, 1024, 2048):
        assert "KnowledgeGraphSolver_%d_f_j" % dim in mine["solver"]  # src/graphvite.cu:61-70
    assert {"Graph_j", "WordGraph_j", "KnowledgeGraph_j"} <= set(mine["graph"])
    assert {"LRSchedule", "Optimizer", "SGD", "Momentum", "AdaGrad", "RMSprop", "Adam"} <= set(mine["optimizer"])
    assert mine["auto"] == 0 and mine["gib2"] == 2 << 30 and mine["dtype2name"]["uint32"] == "j"


def test_same_names_as_the_reference_module(mine, theirs):
    skip = {"VisualizationSolver_2_f_j", "VisualizationSolver_3_f_j", "KNNGraph_j"}  # LargeVis: out of scope
    for sub in ("solver", "graph", "optimizer"):
        missing = set(theirs[sub]) - set(mine[sub]) - skip
        assert not missing, (sub, missing)
    assert set(theirs["top"]) - set(mine["top"]) - {"io"} == set()
    assert mine["auto"] == theirs["auto"] and mine["units"] == theirs["units"]
    assert mine["dtype2name"] == theirs["dtype2name"]


def signature_of(doc, generated):
    head = doc.strip().split("\n")[0]
    if not generated:  # the line the reference hands to pybind11 (bind.h): name(arg, arg=default, ...)
        inside = re.match(r"\w+\((.*)\)$", head).group(1)
        out = []
        for item in filter(None, (x.strip() for x in inside.split(","))):
            name, _, default = item.partition("=")
            out.append((name, default if default else None))
        return out
    inside = head[head.index("(") + 1:head.rindex(")")]
    out, depth, item = [], 0, ""
    for ch in inside + ",":
        depth += ch in "[(<"
        depth -= ch in "])>"
        if ch == "," and depth == 0:
            if item.strip():
                name, _, rest = item.strip().partition(":")
                out.append((name.strip(), rest.partition("=")[2].strip() if "=" in rest else None))
            item = ""
        else:
            item += ch
    return out[1:]  # drop self


@pytest.mark.parametrize("method", ["GraphSolver_128_f_j.build", "GraphSolver_128_f_j.train",
                                    "GraphSolver_128_f_j.predict", "GraphSolver_128_f_j.clear",
                                    "KnowledgeGraphSolver_2048_f_j.build", "KnowledgeGraphSolver_2048_f_j.train",
                                    "KnowledgeGraphSolver_2048_f_j.predict"])
def test_solver_method_signatures(mine, theirs, method):
    reference = signature_of(theirs["docs"][method], generated=False)
    ours_ = signature_of(mine["docs"][method], generated=True)
    assert [n for n, _ in reference] == [n for n, _ in ours_]
    for (name, a), (_, b) in zip(reference, ours_):
        assert same_default(a, b), (method, name, a, b)


@pytest.mark.parametrize("cls", ["GraphSolver_128_f_j", "KnowledgeGraphSolver_2048_f_j"])
def test_solver_attributes_are_all_present(mine, theirs, cls):
    missing = set(theirs["attributes"][cls]) - set(mine["attributes"][cls])
    assert not missing, missing


def test_graph_loads_maps_and_saves_like_the_reference(mine, theirs):
    assert mine["graphs"] == theirs["graphs"]  # counts, id2name, name2id, and the bytes save() writes


def test_optimizer_objects(mine, theirs):
    assert set(mine["optimizers"]) == set(theirs["optimizers"])
    for name, reference in theirs["optimizers"].items():
        assert mine["optimizers"][name] == reference, name


def test_implicit_conversions_and_error_behaviour(mine):
    """bind.h:793-794,837-838: int (auto) / float (lr) -> Optimizer, str / callable -> LRSchedule; errors are Python
    exceptions where the reference abort()s"""
    assert mine["optimizers"]["Optimizer(auto)"] == "Default"
    assert mine["optimizers"]["Optimizer(0.5)"] == 0.5
    assert mine["optimizers"]["LRSchedule"] == "linear"
    assert mine["bad_schedule"] in ("ValueError", "RuntimeError")
    assert mine.get("solver_without_gpu", "RuntimeError") == "RuntimeError"
    assert mine["two_devices"] != "constructed"  # one process drives one GPU: refused with instructions, not truncated
