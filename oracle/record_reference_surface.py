#!/usr/bin/env python
"""Records what tests/test_reference_surface.py (and the loader test of tests/test_oracle_kg.py) compares with: the UNMODIFIED reference module
(oracle/_ref/libgraphvite.so, `make -C oracle ref`; imports and runs on CPU) put through the test's own scenarios.

    python oracle/record_reference_surface.py tests/golden/reference_surface.json
"""
import importlib.util
import json
import os
import pathlib
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import test_oracle_kg  # noqa: E402
import test_reference_surface as T  # noqa: E402


def load_reference():
    spec = importlib.util.spec_from_file_location("libgraphvite", os.path.join(ROOT, "oracle", "_ref", "libgraphvite.so"))
    module = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(module)
    module.init_logging(module.ERROR, "", False)
    return module


def main(out_path):
    ref = load_reference()
    solver, graph = ref.solver.GraphSolver_128_f_j, ref.graph
    record = {
        "docs": dict([("GraphSolver_128_f_j." + m, getattr(solver, m).__doc__) for m in ("build", "train", "predict",
                                                                                         "clear")] +
                     [("Graph_j.save", graph.Graph_j.save.__doc__),
                      ("KnowledgeGraph_j.save", graph.KnowledgeGraph_j.save.__doc__),
                      ("WordGraph_j.load", graph.WordGraph_j.load.__doc__)]),
        "public": {"GraphSolver_128_f_j": sorted(T.public(solver)), "Graph_j": sorted(T.public(graph.Graph_j)),
                   "KnowledgeGraph_j": sorted(T.public(graph.KnowledgeGraph_j))},
        "auto": ref.auto,
        "units": {unit: getattr(ref, unit)(3) for unit in ("KiB", "MiB", "GiB")},
        "optimizers": {name: T.observe_optimizer(ref.optimizer, name) for name in sorted(T.OPTIMIZERS)},
        "lr_schedules": T.observe_lr_schedules(ref.optimizer),
        "graph_loader": {}, "kg_loader": {}, "word_graph": {},
        "toy_graph": T.observe_toy_graph(graph.Graph_j),
    }
    with tempfile.TemporaryDirectory() as tmp:
        tmp = pathlib.Path(tmp)
        for case in T.LOADER_CASES:
            record["graph_loader"][T.loader_key(*case)] = T.observe_graph_loader(graph.Graph_j, tmp, *case)
        record["edge_list_overloads"] = T.observe_edge_list_overloads(graph.Graph_j, tmp)
        record["custom_delimiters"] = T.observe_custom_delimiters(graph.Graph_j, tmp)
        for normalization in (False, True):
            for weighted in (False, True):
                kg = T.load_kg_loader_case(graph.KnowledgeGraph_j, tmp, normalization, weighted)
                kg.save(str(tmp / "anonymous.txt"), True)  # head, tail, int(weight) in flatten order
                columns = np.loadtxt(str(tmp / "anonymous.txt"), dtype=np.int64, ndmin=2)
                record["kg_loader"]["n%d_w%d" % (normalization, weighted)] = {
                    "graph": T.observe_kg(kg), "anonymous_columns": [T.int_digest(columns[:, i]) for i in range(3)]}
        record["kg_save"] = T.observe_kg_save(graph.KnowledgeGraph_j, tmp)
        record["kg_toy_triplets"] = test_oracle_kg.observe_toy_knowledge_graph(graph.KnowledgeGraph_j, tmp)
        for window, min_count, normalization in T.WORD_CASES:
            record["word_graph"]["%d_%d_%d" % (window, min_count, normalization)] = T.observe_word_graph(
                graph.WordGraph_j, tmp, window, min_count, normalization)
    with open(out_path, "w") as fout:
        fout.write(json.dumps(record, sort_keys=True, separators=(",", ":")) + "\n")


if __name__ == "__main__":
    main(sys.argv[1])
