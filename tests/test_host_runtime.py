"""CPU-side checks of the product library: the C ABI exports every symbol include/gv_b200.h
declares, and the host-side Graph / AliasTable builders agree with the oracle and the goldens.
No compute entry point is called here (there is no GPU in this container)."""
import ctypes
import os
import re

import numpy as np
import pytest

import oracle_lib as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_abi_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "gv_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(gv_[a-z0-9_]+)\s*\(", header))
    declared -= {"gv_exchange_fn"}
    from graphvite_b200 import _lib
    library = ctypes.CDLL(_lib.LIB_PATH)
    missing = [name for name in sorted(declared) if not hasattr(library, name)]
    assert not missing, "declared in gv_b200.h but not exported: %s" % missing
    unbound = sorted(declared - set(_lib.SIGNATURES))
    assert not unbound, "declared but not bound in graphvite_b200/_lib.py: %s" % unbound
    assert len(declared) >= 40


def test_ctypes_signatures_have_the_arity_of_the_header():
    """every prototype of include/gv_b200.h against graphvite_b200/_lib.py: the same number of parameters (a wrong
    count is a silent stack bug with ctypes)"""
    header = open(os.path.join(ROOT, "include", "gv_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    header = re.sub(r"typedef[^;{]*\(\s*\*\s*\w+\s*\)\s*\([^;]*\);", "", header)  # function-pointer typedefs
    from graphvite_b200 import _lib
    checked = 0
    for name, parameters in re.findall(r"\b(gv_[a-z0-9_]+)\s*\(([^()]*(?:\([^()]*\)[^()]*)*)\)\s*;", header):
        if name not in _lib.SIGNATURES:
            continue
        parameters = parameters.strip()
        count = 0 if parameters in ("", "void") else parameters.count(",") + 1
        assert len(_lib.SIGNATURES[name][1]) == count, "%s: %d parameters in the header, %d in _lib.py" % (
            name, count, len(_lib.SIGNATURES[name][1]))
        checked += 1
    assert checked >= 100


def test_ctypes_structures_have_the_layout_of_the_header(tmp_path):
    """sizeof and the offset of every member, as gcc lays out include/gv_b200.h, against the ctypes mirrors"""
    import subprocess
    from graphvite_b200 import _lib
    pairs = {"gv_optimizer_t": _lib.OptimizerDesc, "gv_device_optimizer_t": _lib.DeviceOptimizer,
             "gv_matrices_t": _lib.Matrices, "gv_device_graph_t": _lib.DeviceGraph, "gv_kg_matrices_t": _lib.KgMatrices,
             "gv_device_kgraph_t": _lib.DeviceKGraph, "gv_table_shards_t": _lib.TableShards,
             "gv_fill_params_t": _lib.FillParams}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "gv_b200.h"', 'int main(void) {']
    for c_name, mirror in pairs.items():
        lines.append('printf("%s sizeof %%zu\\n", sizeof(%s));' % (c_name, c_name))
        for field in mirror._fields_:
            lines.append('printf("%s %s %%zu\\n", offsetof(%s, %s));' % (c_name, field[0], c_name, field[0]))
    lines += ['return 0;', '}']
    source = tmp_path / "layout.c"
    source.write_text("\n".join(lines))
    binary = str(tmp_path / "layout")
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(source), "-o", binary])
    for line in subprocess.check_output([binary], text=True).splitlines():
        c_name, member, value = line.split()
        mirror = pairs[c_name]
        expected = ctypes.sizeof(mirror) if member == "sizeof" else getattr(mirror, member).offset
        assert int(value) == expected, "%s.%s: %s in C, %d in ctypes" % (c_name, member, value, expected)


def test_missing_extension_fails_loudly(tmp_path, monkeypatch):
    """the product never falls back to CPU / PyTorch code when the .so is absent"""
    import importlib.util
    source = os.path.join(ROOT, "graphvite_b200", "_lib.py")
    fake = tmp_path / "_lib.py"
    fake.write_text(open(source).read())
    spec = importlib.util.spec_from_file_location("gv_fake_lib", str(fake))
    module = importlib.util.module_from_spec(spec)
    with pytest.raises(ImportError, match="mandatory"):
        spec.loader.exec_module(module)


def test_solver_without_gpu_reports_an_error():
    import graphvite_b200 as gv
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("a GPU is present")
    except ImportError:
        pass
    with pytest.raises(gv.GVError, match="CUDA"):
        gv.solver.GraphSolver(128)


@pytest.mark.parametrize("undirected", [True, False])
@pytest.mark.parametrize("normalization", [False, True])
def test_graph_matches_golden_and_oracle(golden_dir, toy_graph_file, undirected, normalization):
    import graphvite_b200 as gv
    from graphvite_b200 import _lib
    golden = np.load("%s/graph_u%d_n%d.npz" % (golden_dir, undirected, normalization))
    graph = gv.graph.Graph()
    graph.load(toy_graph_file, as_undirected=undirected, normalization=normalization)
    assert graph.num_vertex == golden["num_vertex"] and graph.num_edge == golden["num_edge"]
    assert graph.as_undirected == undirected and graph.normalization == normalization
    m = _lib.lib.gv_graph_flatten(graph._handle, None, None, None, None, None)
    u, v = np.zeros(m, dtype=np.uint32), np.zeros(m, dtype=np.uint32)
    w, offsets = np.zeros(m, dtype=np.float32), np.zeros(graph.num_vertex, dtype=np.uint64)
    weights = np.zeros(graph.num_vertex, dtype=np.float32)
    _lib.lib.gv_graph_flatten(graph._handle, u.ctypes.data, v.ctypes.data, w.ctypes.data, offsets.ctypes.data,
                              weights.ctypes.data)
    np.testing.assert_array_equal(u, golden["u"])
    np.testing.assert_array_equal(v, golden["v"])
    np.testing.assert_array_equal(w, golden["w"])
    np.testing.assert_array_equal(weights, golden["vertex_weights"])
    oracle = O.OracleGraph(toy_graph_file, undirected, normalization)
    np.testing.assert_array_equal(offsets, oracle.flat()[3])
    assert graph.id2name == oracle.id2name()
    assert graph.name2id["n65"] == 0 and "nope" not in graph.name2id
    assert "#vertex: %d, #edge: %d" % (graph.num_vertex, graph.num_edge) in repr(graph)


def test_graph_edge_list_overloads_and_save(tmp_path):
    import graphvite_b200 as gv
    edges = [("a", "b"), ("b", "c"), ("c", "a"), ("c", "c"), ("a", "b")]
    graph = gv.graph.Graph()
    graph.load(edges)
    assert (graph.num_vertex, graph.num_edge) == (3, 5)
    weighted = gv.graph.Graph()
    weighted.load([(u, v, 0.5 + i) for i, (u, v) in enumerate(edges)], as_undirected=False)
    path = str(tmp_path / "saved.txt")
    weighted.save(path)
    lines = open(path).read().split("\n")
    assert lines[0].split("\t")[:2] == ["a", "b"] and abs(float(lines[0].split("\t")[2]) - 0.5) < 1e-6
    reloaded = gv.graph.Graph()
    reloaded.load(path, as_undirected=False)
    assert (reloaded.num_vertex, reloaded.num_edge) == (3, 5)
    weighted.save(path, weighted=False, anonymous=True)
    assert open(path).readline().strip() == "0\t1"
    with pytest.raises(gv.GVError, match="doesn't exist"):
        graph.load(str(tmp_path / "missing.txt"))
    bad = tmp_path / "bad.txt"
    bad.write_text("a b\nc\n")
    with pytest.raises(gv.GVError, match="Invalid format at line 2"):
        graph.load(str(bad))
    with pytest.raises(gv.GVError, match="Invalid format at line 1"):
        bad.write_text("a b 1 extra\n")
        graph.load(str(bad))


def test_graph_custom_delimiters_and_comments(tmp_path):
    import graphvite_b200 as gv
    path = tmp_path / "g.csv"
    path.write_text("% header\nx,y,2.5\n\ny,z % tail\n")
    graph = gv.graph.Graph()
    graph.load(str(path), delimiters=",\n ", comment="%")
    assert (graph.num_vertex, graph.num_edge) == (3, 2)
    oracle = O.OracleGraph(str(path), True, False, ",\n ", "%")
    assert graph.id2name == oracle.id2name()


@pytest.mark.parametrize("count", [1, 2, 37, 1000, 50000])
def test_alias_build_matches_oracle(count):
    from graphvite_b200 import _lib
    rng = np.random.RandomState(count)
    for weights in (rng.pareto(1.3, count) + 1e-3, np.ones(count), rng.randint(1, 4, count)):
        weights = weights.astype(np.float32)
        prob, alias = np.zeros(count, dtype=np.float32), np.zeros(count, dtype=np.uint64)
        _lib.check(_lib.lib.gv_alias_build(weights.ctypes.data, count, prob.ctypes.data, alias.ctypes.data))
        oprob, oalias = O.alias_build(weights)
        np.testing.assert_array_equal(prob, oprob)
        np.testing.assert_array_equal(alias, oalias)


def test_alias_build_matches_golden(golden_dir):
    from graphvite_b200 import _lib
    golden = np.load(golden_dir + "/alias.npz")
    weights = golden["weights"]
    prob, alias = np.zeros(len(weights), dtype=np.float32), np.zeros(len(weights), dtype=np.uint64)
    _lib.check(_lib.lib.gv_alias_build(weights.ctypes.data, len(weights), prob.ctypes.data, alias.ctypes.data))
    np.testing.assert_array_equal(prob, golden["prob"])
    np.testing.assert_array_equal(alias, golden["alias"])
    with pytest.raises(_lib.GVError, match="Invalid sampling distribution"):
        _lib.check(_lib.lib.gv_alias_build(weights.ctypes.data, 0, prob.ctypes.data, alias.ctypes.data))


def test_optimizer_surface():
    import graphvite_b200 as gv
    opt = gv.optimizer
    assert opt.Optimizer(gv.auto).type == "Default"
    assert isinstance(opt.Optimizer("Adam", lr=1e-3), opt.Adam)
    with pytest.raises(ValueError):
        opt.Optimizer("Nope")
    sgd = opt.SGD()
    assert (sgd.lr, sgd.weight_decay, sgd.schedule.type) == (1e-4, 0, "linear")
    adam = opt.Adam()
    assert (adam.beta1, adam.beta2, adam.epsilon) == (0.999, 0.99999, 1e-8)
    assert opt.Momentum().momentum == 0.999 and opt.AdaGrad().epsilon == 1e-10
    assert opt.RMSprop().alpha == 0.999 and opt.RMSprop().epsilon == 1e-8
    assert opt.LRSchedule("linear")(50, 100) == 0.5 and opt.LRSchedule("constant")(50, 100) == 1
    custom = opt.SGD(0.1, schedule=lambda batch_id, num_batch: 0.5)
    descriptor = custom._descriptor()
    assert descriptor.schedule == 2 and abs(descriptor.schedule_fn(3, 10, None) - 0.5) < 1e-7
    with pytest.raises(ValueError):
        opt.LRSchedule("cosine")
    assert "optimizer: Adam" in repr(adam) and "beta1" in repr(adam)


def test_link_prediction_auc_formula():
    from graphvite_b200.application import link_prediction_auc
    assert link_prediction_auc([0.9, 0.8, 0.1, 0.2], [1, 1, 0, 0]) == 1.0
    assert link_prediction_auc([0.1, 0.2, 0.9, 0.8], [1, 1, 0, 0]) == 0.0
    rng = np.random.RandomState(0)
    scores, labels = rng.rand(2000), rng.randint(0, 2, 2000)
    from sklearn.metrics import roc_auc_score
    assert abs(link_prediction_auc(scores, labels) - roc_auc_score(labels, scores)) < 1e-9


def test_yaml_config_loading(tmp_path):
    """the reference's quick-start configuration loads unchanged except for the dataset placeholders"""
    import yaml
    from graphvite_b200 import cmd, optimizer, auto
    # the content of the reference's config/demo/quick_start.yaml
    cfg = {"application": "graph", "resource": {"gpus": [0], "cpu_per_gpu": 8, "dim": 128},
           "format": {"delimiters": " \t\r\n", "comment": "#"},
           "graph": {"file_name": "<blogcatalog.train>", "as_undirected": True},
           "build": {"optimizer": {"type": "SGD", "lr": 0.025, "weight_decay": 0.005}, "num_partition": "auto",
                     "num_negative": 1, "batch_size": 100000, "episode_size": 500},
           "train": {"model": "LINE", "num_epoch": 2000, "negative_weight": 5, "augmentation_step": 2,
                     "random_walk_length": 40, "random_walk_batch_size": 100, "log_frequency": 1000},
           "evaluate": [{"task": "link prediction", "file_name": "<blogcatalog.test>",
                         "filter_file": "<blogcatalog.train>"},
                        {"task": "node classification", "file_name": "<blogcatalog.label>", "portions": [0.2],
                         "times": 1}],
           "save": {"file_name": "line_blogcatalog.pkl"}}
    path = tmp_path / "quick_start.yaml"
    path.write_text(yaml.safe_dump(cfg))
    with pytest.raises(ValueError, match="dataset placeholder"):
        cmd.load_config(str(path))
    cfg["graph"]["file_name"] = "graph.txt"
    cfg["evaluate"] = [{"task": "link prediction", "file_name": "test.txt", "filter_file": "graph.txt"}]
    path.write_text(yaml.safe_dump(cfg))
    loaded = cmd.load_config(str(path))
    assert isinstance(loaded["build"]["optimizer"], optimizer.SGD)
    assert loaded["build"]["optimizer"].weight_decay == 0.005
    assert loaded["build"]["num_partition"] == auto and loaded["resource"]["dim"] == 128
    args = cmd.get_parser().parse_args(["run", str(path), "--epoch", "3", "--no-eval"])
    assert args.epoch == 3 and args.eval is False


def test_node_classification_on_separable_embeddings():
    """GraphApplication.node_classification (application.py:293-351): F1 == 1 when the classes are
    linearly separable; unknown node names are dropped like name_map does"""
    from graphvite_b200.application import GraphApplication

    class FakeGraph(object):
        name2id = {str(i): i for i in range(200)}

    class FakeSolver(object):
        rng = np.random.RandomState(0)
        centers = rng.randn(4, 16) * 3
        cls = rng.randint(0, 4, 200)
        vertex_embeddings = (centers[cls] + 0.3 * rng.randn(200, 16)).astype(np.float32)

    app = GraphApplication.__new__(GraphApplication)
    app.graph, app.solver = FakeGraph(), FakeSolver()
    X = [str(i) for i in range(200)] + ["unknown"]
    Y = ["c%d" % c for c in FakeSolver.cls] + ["c0"]
    result = app.node_classification(X=X, Y=Y, portions=(0.2,), times=2, patience=20)
    assert result["macro-F1@20%"] > 0.95 and result["micro-F1@20%"] > 0.95


@pytest.mark.parametrize("seed,bulk", [(5489, 1000003), (1, 4097), (20260922, 624 * 5)])
def test_bulk_engine_is_std_mt19937(seed, bulk):
    """init_embeddings draws |V| * dim floats: gv::Mt19937 (SSE2 twist + conversion, csrc/gv_engine.h) must be
    std::mt19937 + std::uniform_real_distribution<float> bit for bit, and interchangeable with it for the seeds'
    uniform_int_distribution -- compared inside the library against libstdc++ itself."""
    from graphvite_b200 import _lib
    assert _lib.lib.gv_engine_self_check(seed, bulk) == 0


def test_binary_edge_arrays_load_like_the_equivalent_edge_list(tmp_path):
    """Graph.load_arrays (gv_graph_load_id_edges) builds what load(edge_list=[(str(u), str(v)) ...]) builds -- first-seen
    ids, edge order, counts, weights -- without materialising names: byte-identical save(), same name <-> id maps."""
    import graphvite_b200 as gv
    rng = np.random.RandomState(5)
    u = rng.randint(0, 50, 400)
    v = rng.randint(0, 50, 400)
    w = (rng.rand(400) + 0.5).astype(np.float32)
    for undirected in (True, False):
        for weights in (None, w):
            for normalization in (False, True):
                a, b = gv.graph.Graph(), gv.graph.Graph()
                a.load_arrays(u, v, weights, as_undirected=undirected, normalization=normalization)
                edges = [(str(x), str(y)) for x, y in zip(u, v)] if weights is None else \
                    [(str(x), str(y), float(z)) for x, y, z in zip(u, v, w)]
                b.load(edges, as_undirected=undirected, normalization=normalization)
                assert (a.num_vertex, a.num_edge) == (b.num_vertex, b.num_edge)
                assert a.id2name == b.id2name
                for name in ("0", "17", "49", "50", "x", "07", ""):
                    assert a.name2id.get(name) == b.name2id.get(name), name
                a.save(str(tmp_path / "a.txt"))
                b.save(str(tmp_path / "b.txt"))
                assert (tmp_path / "a.txt").read_bytes() == (tmp_path / "b.txt").read_bytes()
    empty = gv.graph.Graph()
    empty.load_arrays(np.zeros(0, dtype=np.uint32), np.zeros(0, dtype=np.uint32))
    assert empty.num_vertex == 0 and empty.num_edge == 0
    with pytest.raises(ValueError):
        empty.load_arrays(np.zeros(3), np.zeros(4))


def test_gv_sincos_accuracy(tmp_path):
    """gv_sincos (csrc/gv_device.cuh: the rotation of RotatE in the knowledge-graph train kernel) is plain C++ shared by the
    nvcc and the emulation build: compiled here for the host and compared with double precision over [-48000, 48000]
    (<= 1.6 ulp) and on the sincosf() fallback beyond."""
    import subprocess
    source = tmp_path / "probe.cpp"
    source.write_text(r'''
#include <cmath>
#include <cstdio>
#include <cstring>
#define GV_EMULATE
#define GV_DEVICE_INLINE_PROBE
static inline int __float_as_int(float x) { int i; std::memcpy(&i, &x, 4); return i; }
#include "gv_device.cuh"
static double ulp_of(double reference) { int e; std::frexp(float(reference), &e); return std::ldexp(1.0, e - 24); }
int main() {
    double worst = 0;
    const double spans[3] = {3.2, 100.0, 48000.0};
    for (double span : spans)
        for (long i = 0; i <= 4000000; i++) {
            const float x = float(-span + 2 * span * i / 4000000.0);
            float s, c;
            gv_sincos(x, &s, &c);
            const double rs = std::sin(double(x)), rc = std::cos(double(x));
            worst = std::fmax(worst, std::fabs(s - rs) / ulp_of(rs));
            worst = std::fmax(worst, std::fabs(c - rc) / ulp_of(rc));
        }
    float s, c;
    gv_sincos(1e9f, &s, &c);  // the fallback
    const double far = std::fmax(std::fabs(s - std::sin(double(1e9f))), std::fabs(c - std::cos(double(1e9f))));
    gv_sincos(NAN, &s, &c);
    std::printf("%.4f %.3g %d\n", worst, far, int(std::isnan(s) && std::isnan(c)));
    return 0;
}
''')
    binary = tmp_path / "probe"
    include = os.path.join(ROOT, "graphvite_b200", "csrc")
    subprocess.run(["g++", "-O2", "-std=c++17", "-I", include, str(source), "-o", str(binary)], check=True)
    worst, far, nan_ok = subprocess.run([str(binary)], check=True, stdout=subprocess.PIPE, text=True).stdout.split()
    assert float(worst) <= 1.6, worst
    assert float(far) < 1e-6, far
    assert nan_ok == "1"


def test_graph_file_loader_chunk_boundaries_long_names_and_odd_lines(tmp_path):
    """The file loader reads large chunks, carries incomplete lines over, hashes a batch of lines ahead of resolving it
    and keeps the first 11 bytes of a name inline in its table: a file with names of 1 .. 300 bytes (shared prefixes
    longer than 11 and than 255 bytes), blank and comment-only lines, CRLF, a weight column, no newline at the end --
    loaded with chunk sizes that cut every line -- must equal the same edges loaded as a Python list."""
    import subprocess
    import sys
    import graphvite_b200 as gv
    rng = np.random.RandomState(11)
    stem = "x" * 290
    names = ["v%d" % i for i in range(40)] + ["abcdefghijk_%d" % i for i in range(20)] + \
            ["abcdefghijkl" + "y" * int(n) for n in rng.randint(0, 40, 15)] + [stem + "%02d" % i for i in range(10)]
    names = list(dict.fromkeys(names))
    edges = [(names[a], names[b], round(float(w), 3)) for a, b, w in
             zip(rng.randint(0, len(names), 600), rng.randint(0, len(names), 600), rng.rand(600) + 0.5)]
    path = tmp_path / "odd.txt"
    with open(path, "wb") as out:
        out.write(b"# header comment\r\n\r\n   \n")
        for i, (u, v, w) in enumerate(edges):
            separator = b"\t" if i % 3 == 0 else b" "
            ending = b"\r\n" if i % 5 == 0 else b"\n"
            tail = b"  # trailing comment" if i % 7 == 0 else b""
            if i == len(edges) - 1:
                ending = b""  # no newline at the end of the file
            out.write(u.encode() + separator + v.encode() + separator + (b"%.3f" % w) + tail + ending)
            if i % 50 == 0:
                out.write(b"#only a comment\n")
    expected = gv.graph.Graph()
    expected.load([(u, v, w) for u, v, w in edges])
    reference = tmp_path / "expected.txt"
    expected.save(str(reference))
    script = ("import sys; import graphvite_b200 as gv; g = gv.graph.Graph(); g.load(sys.argv[1]); g.save(sys.argv[2]); "
              "print(g.num_vertex, g.num_edge, g.name2id[%r], g.name2id[%r])" % (names[-1], names[3]))
    for chunk in (None, 16, 37, 301, 4096):
        env = dict(os.environ)
        if chunk:
            env["GV_LOAD_CHUNK"] = str(chunk)
        saved = tmp_path / ("saved_%s.txt" % chunk)
        done = subprocess.run([sys.executable, "-c", script, str(path), str(saved)], env=env, cwd=ROOT, check=True,
                              stdout=subprocess.PIPE, text=True)
        assert done.stdout.split() == [str(expected.num_vertex), str(expected.num_edge),
                                       str(expected.name2id[names[-1]]), str(expected.name2id[names[3]])], chunk
        assert saved.read_bytes() == reference.read_bytes(), chunk
