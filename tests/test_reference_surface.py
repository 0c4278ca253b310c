"""Drop-in surface checks against the UNMODIFIED reference module.  The pybind module imports without a GPU: its
classes, docstring signatures, optimizer objects and the host-side Graph are all usable on CPU, so the mirror in
graphvite_b200/ is compared with what the real thing did rather than with a reading of it.

What the reference did is recorded in tests/golden/reference_surface.json by oracle/record_reference_surface.py (run
where the reference module is built, `make -C oracle ref`): its public names and docstrings, its optimizer objects and
learning-rate schedules, and for every loader scenario below the counts, the id maps and SHA-256 digests of the files
its save() wrote.  The scenarios themselves (seeded inputs, `observe_*`) are defined here once and run on both.
"""
import hashlib
import inspect
import json
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RECORDED = os.path.join(ROOT, "tests", "golden", "reference_surface.json")
TOY = os.path.join(ROOT, "tests", "golden", "toy_graph.txt")


@pytest.fixture(scope="module")
def ref():
    with open(RECORDED) as fin:
        return json.load(fin)


@pytest.fixture(scope="module")
def gv():
    import graphvite_b200
    return graphvite_b200


def public(obj):
    return {name for name in dir(obj) if not name.startswith("_")}


def doc_signature(doc):
    """[(name, default-or-None)] from the first docstring line pybind11 was given (bind.h)."""
    head = doc.strip().split("\n")[0]
    inside = re.match(r"\w+\((.*)\)$", head).group(1)
    out = []
    for item in filter(None, (s.strip() for s in inside.split(","))):
        name, _, default = item.partition("=")
        out.append((name, default if default else None))
    return out


def our_signature(function):
    out = []
    for name, p in list(inspect.signature(function).parameters.items())[1:]:
        out.append((name, None if p.default is inspect.Parameter.empty else p.default))
    return out


def same_default(ref_text, ours, gv):
    if ref_text is None or ours is None:
        return ref_text is None and ours is None
    if ref_text == "auto":
        return ours == gv.auto
    if ref_text in ("True", "False"):
        return ours is (ref_text == "True")
    if ref_text[0] in "'\"":
        return ours == ref_text[1:-1]
    return float(ref_text) == float(ours)


def digest(data):
    return hashlib.sha256(data).hexdigest()


def file_digest(path):
    with open(path, "rb") as fin:
        return digest(fin.read())


def names_digest(names):
    return digest("\n".join(names).encode())


def int_digest(values):
    return digest(np.ascontiguousarray(values, dtype="<i8").tobytes())


@pytest.mark.parametrize("method", ["build", "train", "predict", "clear"])
def test_solver_method_signatures(ref, gv, method):
    theirs = doc_signature(ref["docs"]["GraphSolver_128_f_j." + method])
    ours = our_signature(getattr(gv.solver.GraphSolver, method))
    assert [n for n, _ in theirs] == [n for n, _ in ours]
    for (name, a), (_, b) in zip(theirs, ours):
        assert same_default(a, b, gv), (method, name, a, b)


def test_solver_attributes_are_all_present(ref, gv):
    from graphvite_b200 import solver as S
    ours = public(gv.solver.GraphSolver) | set(S._INT_ATTRIBUTES) | set(S._FLOAT_ATTRIBUTES)
    missing = set(ref["public"]["GraphSolver_128_f_j"]) - ours
    assert not missing, missing


def test_graph_surface(ref, gv):
    assert set(ref["public"]["Graph_j"]) <= public(gv.graph.Graph)
    theirs = doc_signature(ref["docs"]["Graph_j.save"])
    ours = our_signature(gv.graph.Graph.save)
    assert [n for n, _ in theirs] == [n for n, _ in ours]
    for (name, a), (_, b) in zip(theirs, ours):
        assert same_default(a, b, gv), (name, a, b)
    assert gv.auto == ref["auto"]
    for unit in ("KiB", "MiB", "GiB"):
        assert getattr(gv, unit)(3) == ref["units"][unit]


OPTIMIZERS = {
    "SGD": ("lr", "weight_decay"),
    "Momentum": ("lr", "weight_decay", "momentum"),
    "AdaGrad": ("lr", "weight_decay", "epsilon"),
    "RMSprop": ("lr", "weight_decay", "alpha", "epsilon"),
    "Adam": ("lr", "weight_decay", "beta1", "beta2", "epsilon"),
}
POSITIONAL = [0.5, 0.25, 0.75, 0.875, 0.125]


def observe_optimizer(optimizer_module, name):
    """what test_optimizer_defaults_and_positional_order compares, for either module's `optimizer`"""
    fields = OPTIMIZERS[name]
    default = getattr(optimizer_module, name)()
    positional = getattr(optimizer_module, name)(*POSITIONAL[:len(fields)])
    constant = getattr(optimizer_module, name)(schedule="constant")
    return {"public": sorted(public(default)), "type": default.type,
            "default": [float(np.float32(getattr(default, field))) for field in fields],
            "positional": [float(getattr(positional, field)) for field in fields],
            "schedule": default.schedule.type, "constant_schedule": constant.schedule.type}


@pytest.mark.parametrize("name", sorted(OPTIMIZERS))
def test_optimizer_defaults_and_positional_order(ref, gv, name):
    theirs, ours = ref["optimizers"][name], observe_optimizer(gv.optimizer, name)
    assert set(theirs["public"]) <= set(ours["public"]) | {"lr", "weight_decay", "schedule"}
    assert theirs["type"] == ours["type"]
    for field, a, b in zip(OPTIMIZERS[name], theirs["default"], ours["default"]):
        assert a == b, field
    assert theirs["schedule"] == ours["schedule"] == "linear"
    # positional construction assigns the same fields in the same order
    assert theirs["positional"] == ours["positional"] == POSITIONAL[:len(OPTIMIZERS[name])]
    assert theirs["constant_schedule"] == ours["constant_schedule"] == "constant"


LR_POINTS = ((0, 10), (3, 10), (9, 10), (10, 10), (1978, 1978), (12, 7))


def observe_lr_schedules(optimizer_module):
    return {kind: [float(np.float32(optimizer_module.LRSchedule(kind).schedule_function(batch_id, num_batch)))
                   for batch_id, num_batch in LR_POINTS] for kind in ("constant", "linear")}


def test_lr_schedules_agree(ref, gv):
    assert observe_lr_schedules(gv.optimizer) == ref["lr_schedules"]
    with pytest.raises(ValueError):  # the reference CHECK-fails (aborts the process) on the same input
        gv.optimizer.LRSchedule("cosine")


def write_graph(path, rng, num_vertex, num_edge, weighted, comment):
    with open(path, "w") as out:
        if comment:
            out.write("# header line\n")
        for i in range(num_edge):
            u, v = rng.integers(0, num_vertex, 2)
            line = "n%d\tn%d" % (u, v) if i % 3 else "n%d n%d" % (u, v)
            if weighted:
                line += " %g" % (0.25 + 0.25 * rng.integers(0, 12))
            if comment and i % 17 == 0:
                line += " # trailing comment"
            out.write(line + "\n")


def observe_graph(graph, tmp_path, save_modes=((True, False),), sample=None):
    """counts, flags, the id map and digests of what save(weighted, anonymous) writes in each mode"""
    out = {"counts": [graph.num_vertex, graph.num_edge], "flags": [graph.as_undirected, graph.normalization],
           "id2name": names_digest(list(graph.id2name)), "saved": []}
    if sample:
        out["name2id"] = [graph.name2id[name] for name in list(graph.id2name)[::sample]]
    for mode, (weighted, anonymous) in enumerate(save_modes):
        path = str(tmp_path / ("saved%d.txt" % mode))
        graph.save(path, weighted, anonymous)
        out["saved"].append(file_digest(path))
    return out


LOADER_MODES = ((True, False), (False, False), (True, True), (False, True))
LOADER_CASES = [(u, n, w) for w in (False, True) for n in (False, True) for u in (True, False)]


def observe_graph_loader(graph_class, tmp_path, as_undirected, normalization, weighted):
    """Same edge list through both loaders: ids in order of first appearance, edge counts, and a
    byte-identical save() in every mode (instance/graph.cuh:137-277)."""
    rng = np.random.default_rng(7 + 2 * as_undirected + normalization)
    source = str(tmp_path / "edges.txt")
    write_graph(source, rng, 300, 2500, weighted, comment=True)
    graph = graph_class()
    graph.load(source, as_undirected, normalization)
    return observe_graph(graph, tmp_path, LOADER_MODES, sample=37)


def loader_key(as_undirected, normalization, weighted):
    return "u%d_n%d_w%d" % (as_undirected, normalization, weighted)


@pytest.mark.parametrize("as_undirected", [True, False])
@pytest.mark.parametrize("normalization", [False, True])
@pytest.mark.parametrize("weighted", [False, True])
def test_graph_loader_matches_the_reference_object(ref, gv, tmp_path, as_undirected, normalization, weighted):
    ours = observe_graph_loader(gv.graph.Graph, tmp_path, as_undirected, normalization, weighted)
    assert ours == ref["graph_loader"][loader_key(as_undirected, normalization, weighted)]


def observe_edge_list_overloads(graph_class, tmp_path):
    rng = np.random.default_rng(11)
    pairs = [("v%d" % u, "v%d" % v) for u, v in rng.integers(0, 50, (400, 2))]
    triples = [(u, v, float(0.5 + 0.5 * (i % 5))) for i, (u, v) in enumerate(pairs)]
    out = []
    for edges in (pairs, triples):
        for as_undirected in (True, False):
            graph = graph_class()
            graph.load(edges, as_undirected, False)
            out.append(observe_graph(graph, tmp_path))
    return out


def test_edge_list_overloads_match_the_reference_object(ref, gv, tmp_path):
    assert observe_edge_list_overloads(gv.graph.Graph, tmp_path) == ref["edge_list_overloads"]


def observe_custom_delimiters(graph_class, tmp_path):
    source = str(tmp_path / "csv.txt")
    with open(source, "w") as out:
        out.write("% matrix market style comment\n")
        out.write("a,b,2\nb,c,1.5 % note\nc,a,0.5\na,d,1\n")
    graph = graph_class()
    graph.load(source, True, False, ",\r\n", "%")
    return observe_graph(graph, tmp_path)


def test_custom_delimiters_and_comment_prefix(ref, gv, tmp_path):
    ours = observe_custom_delimiters(gv.graph.Graph, tmp_path)
    assert ours["counts"] == [4, 4]
    assert ours == ref["custom_delimiters"]


def observe_toy_graph(graph_class):
    graph = graph_class()
    graph.load(TOY, True, False)
    return {"counts": [graph.num_vertex, graph.num_edge], "id2name": list(graph.id2name)}


def test_toy_graph_golden_is_what_the_reference_loads(ref, gv):
    assert observe_toy_graph(gv.graph.Graph) == ref["toy_graph"]


# ---- KnowledgeGraph (instance/knowledge_graph.cuh:67-284) ------------------------------------------
def write_triplets(path, rng, num_entity, num_relation, num_triplet, weighted):
    with open(path, "w") as out:
        out.write("# knowledge graph\n")
        for i in range(num_triplet):
            h, t = rng.integers(0, num_entity, 2)
            r = rng.integers(0, num_relation)
            line = "/m/%d\t/rel/%d\t/m/%d" % (h, r, t) if i % 2 else "/m/%d /rel/%d /m/%d" % (h, r, t)
            if weighted:
                line += " %g" % (0.5 + 0.5 * rng.integers(0, 6))
            out.write(line + ("  # note\n" if i % 23 == 0 else "\n"))


def kg_flatten(gv, graph):
    from graphvite_b200 import _lib
    m = _lib.lib.gv_kgraph_flatten(graph._handle, None, None, None, None, None, None)
    h, t, r = (np.zeros(m, dtype=np.uint32) for _ in range(3))
    w, vw = np.zeros(m, dtype=np.float32), np.zeros(graph.num_vertex, dtype=np.float32)
    _lib.lib.gv_kgraph_flatten(graph._handle, h.ctypes.data, t.ctypes.data, r.ctypes.data, w.ctypes.data, None,
                               vw.ctypes.data)
    return h, t, r, w, vw


def test_knowledge_graph_surface(ref, gv):
    assert set(ref["public"]["KnowledgeGraph_j"]) <= public(gv.graph.KnowledgeGraph)
    theirs = doc_signature(ref["docs"]["KnowledgeGraph_j.save"])
    ours = our_signature(gv.graph.KnowledgeGraph.save)
    assert [n for n, _ in theirs] == [n for n, _ in ours]
    for (name, a), (_, b) in zip(theirs, ours):
        assert same_default(a, b, gv), (name, a, b)


def load_kg_loader_case(kg_class, tmp_path, normalization, weighted):
    rng = np.random.default_rng(3 + normalization)
    source = str(tmp_path / "triplets.txt")
    write_triplets(source, rng, 120, 9, 1500, weighted)
    graph = kg_class()
    graph.load(source, normalization)
    return graph


def observe_kg(graph):
    return {"counts": [graph.num_vertex, graph.num_edge, graph.num_relation], "normalization": graph.normalization,
            "id2entity": names_digest(list(graph.id2entity)), "id2relation": list(graph.id2relation),
            "entity2id": [graph.entity2id[name] for name in list(graph.id2entity)[::17]],
            "relation2id": [graph.relation2id[name] for name in graph.id2relation],
            "repr_tail": repr(graph).splitlines()[-2:]}


@pytest.mark.parametrize("normalization", [False, True])
@pytest.mark.parametrize("weighted", [False, True])
def test_knowledge_graph_loader_matches_the_reference_object(ref, gv, tmp_path, normalization, weighted):
    theirs = ref["kg_loader"]["n%d_w%d" % (normalization, weighted)]
    ours = load_kg_loader_case(gv.graph.KnowledgeGraph, tmp_path, normalization, weighted)
    assert observe_kg(ours) == theirs["graph"]
    # anonymous save of the reference = head, tail, int(weight) in flatten order: pins heads, tails and order;
    # (its third column is the weight by mistake, knowledge_graph.cuh:275)
    h, t, r, w, _ = kg_flatten(gv, ours)
    assert [int_digest(h), int_digest(t), int_digest(w.astype(np.int64))] == theirs["anonymous_columns"]
    assert "#entity: %d, #relation: %d" % (ours.num_vertex, ours.num_relation) in repr(ours)


def observe_kg_save(kg_class, tmp_path):
    """weights equal to the relation ids make the reference's `relation = weight` slip invisible"""
    rng = np.random.default_rng(9)
    relations = ["r%d" % i for i in range(6)]
    triplets = [("e0", "r0", "e1", 0.0)]  # r0 first so that relation ids follow the numbering
    for r in range(1, 6):
        triplets.append(("e1", relations[r], "e0", float(r)))
    for _ in range(300):
        r = int(rng.integers(0, 6))
        triplets.append(("e%d" % rng.integers(0, 40), relations[r], "e%d" % rng.integers(0, 40), float(r)))
    graph = kg_class()
    graph.load(triplets, False)
    out = {"id2relation": list(graph.id2relation), "saved": []}
    for anonymous in (False, True):
        path = str(tmp_path / "saved.txt")
        graph.save(path, anonymous)
        out["saved"].append(file_digest(path))
    return out


def test_knowledge_graph_save_is_byte_identical_where_the_reference_is_well_defined(ref, gv, tmp_path):
    ours = observe_kg_save(gv.graph.KnowledgeGraph, tmp_path)
    assert ours["id2relation"] == ["r%d" % i for i in range(6)]
    assert ours == ref["kg_save"]


def test_knowledge_graph_normalization_weights(ref, gv, tmp_path):
    """normalized weights are not exposed by the reference's Python surface except through save()'s
    integer column; compare against a float32 restatement of normalize() (knowledge_graph.cuh:95-121)"""
    rng = np.random.default_rng(21)
    triplets = [("e%d" % rng.integers(0, 30), "r%d" % rng.integers(0, 4), "e%d" % rng.integers(0, 30),
                 float(0.5 + 0.25 * rng.integers(0, 8))) for _ in range(400)]
    plain, normalized = gv.graph.KnowledgeGraph(), gv.graph.KnowledgeGraph()
    plain.load(triplets, False)
    normalized.load(triplets, True)
    h, t, r, w, vw = kg_flatten(gv, plain)
    head_w, tail_w = {}, {}
    for i in range(len(h)):
        head_w[(h[i], r[i])] = np.float32(head_w.get((h[i], r[i]), np.float32(0)) + w[i])
        tail_w[(t[i], r[i])] = np.float32(tail_w.get((t[i], r[i]), np.float32(0)) + w[i])
    expected = np.array([w[i] / np.sqrt(np.float32(head_w[(h[i], r[i])] * tail_w[(t[i], r[i])]))
                         for i in range(len(h))], dtype=np.float32)
    h2, t2, r2, w2, vw2 = kg_flatten(gv, normalized)
    np.testing.assert_array_equal(h2, h)
    np.testing.assert_array_equal(r2, r)
    np.testing.assert_allclose(w2, expected, rtol=1e-6)
    sums = np.zeros(plain.num_vertex, dtype=np.float64)
    np.add.at(sums, h2, w2.astype(np.float64))
    np.testing.assert_allclose(vw2, sums, rtol=1e-5)


def test_knowledge_graph_rejects_malformed_lines(gv, tmp_path):
    from graphvite_b200 import _lib
    source = str(tmp_path / "bad.txt")
    with open(source, "w") as out:
        out.write("a r b\nc r\n")
    with pytest.raises(_lib.GVError, match="Invalid format at line 2"):
        gv.graph.KnowledgeGraph().load(source)
    with open(source, "w") as out:
        out.write("a r b 1 extra\n")
    with pytest.raises(_lib.GVError, match="Invalid format at line 1"):
        gv.graph.KnowledgeGraph().load(source)


# ---- WordGraph (bind.h:190-234, instance/word_graph.cuh) ------------------------------------------------------------
def write_corpus(path, rng, vocabulary, lines):
    words = ["w%d" % i for i in range(vocabulary)]
    weights = np.arange(1, vocabulary + 1) ** -1.0
    weights /= weights.sum()
    with open(path, "w") as out:
        out.write("# a corpus\n\n")
        for i in range(lines):
            sentence = rng.choice(words, size=int(rng.integers(1, 25)), p=weights)
            text = " ".join(sentence)
            if i % 13 == 0:
                text = text.replace(" ", "\t", 2) + "   # trailing comment with words w1 w2"
            out.write(text + "\n")


WORD_CASES = [(5, 5, False), (2, 1, False), (7, 3, True)]


def observe_word_graph(word_class, tmp_path, window, min_count, normalization):
    """Vocabulary (ids by first appearance, min_count filter), co-occurrence counts and -- because the out-edges of
    a vertex are emitted in the iteration order of an unordered_map -- the edge ORDER: save() must be byte-identical."""
    rng = np.random.default_rng(11 + window)
    corpus = str(tmp_path / "corpus.txt")
    write_corpus(corpus, rng, 150, 400)
    graph = word_class()
    graph.load(corpus, window, min_count, normalization)
    return dict(observe_graph(graph, tmp_path, ((True, False), (False, True))),
                repr_head=repr(graph).splitlines()[0])


@pytest.mark.parametrize("window,min_count,normalization", WORD_CASES)
def test_word_graph_loader_matches_the_reference_object(ref, gv, tmp_path, window, min_count, normalization):
    theirs = ref["word_graph"]["%d_%d_%d" % (window, min_count, normalization)]
    assert [n for n, _ in doc_signature(ref["docs"]["WordGraph_j.load"])] == \
        [n for n, _ in our_signature(gv.graph.WordGraph.load)]
    ours = observe_word_graph(gv.graph.WordGraph, tmp_path, window, min_count, normalization)
    assert ours["counts"][0] > 20 and ours["counts"][1] > 100
    assert ours["flags"] == [True, normalization]
    assert ours["repr_head"] == "WordGraph<uint32>"
    assert ours == theirs
