#!/usr/bin/env python
"""Writes what tests/test_gpu_zzzzz_parity.py compares with: Hogwild training runs of the UNMODIFIED reference
(oracle/_ref/libgraphvite.so, `make -C oracle ref`), reduced to embedding L2 norms and link-prediction AUC, as
tests/golden/parity_reference.json -- so that the parity tests run without the reference.

The runs themselves are the reference's B200 runs committed under profiles/ (tools/parity_sweep.py wrote them on the
same seeded inputs the tests train on):
  * profiles/r02_parity_sweep1_{blogcatalog,youtube}.jsonl: three runs per workload, 2000 / 100 epochs;
  * profiles/r02_hogwild_probe_20k.txt: three runs of the 20k-vertex race probe, norms only.  Their link-prediction
    AUC was not recorded per run; the range measured with them, 0.8288-0.8292, is stored as its midpoint 0.829 and
    marked as such in the file.
The id order of the probe graph is taken from the reference's own loader, which runs on the CPU.

    python oracle/record_parity_reference.py tests/golden/parity_reference.json
"""
import hashlib
import importlib.util
import json
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import test_gpu_zzzzz_parity as parity  # noqa: E402

PROBE_AUC = 0.829
PROBE_AUC_NOTE = "not recorded per run: midpoint of the range 0.8288-0.8292 measured with these runs"


def reference_runs(path):
    rows = [json.loads(line) for line in open(path) if line.strip()]
    header = rows[0]
    runs = [{key: row[key] for key in ("vertex_norm", "context_norm", "auc")} for row in rows
            if row.get("impl") == "reference"]
    return header["epochs"], runs


def probe_runs(path):
    out = []
    for line in open(path):
        words = line.split()
        if words and words[0] == "reference":
            out.append({"vertex": float(words[1]), "context": float(words[2])})
    return out


def main(out_path):
    from graphvite_b200 import datasets
    spec = importlib.util.spec_from_file_location("libgraphvite", os.path.join(ROOT, "oracle", "_ref",
                                                                               "libgraphvite.so"))
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    ref.init_logging(ref.ERROR, "", False)
    record = {"workloads": {}}
    for workload in parity.RUNS:
        epochs, runs = reference_runs(os.path.join(ROOT, "profiles", "r02_parity_sweep1_%s.jsonl" % workload))
        record["workloads"][workload] = {"epochs": epochs, "runs": runs}
    u, v = datasets.power_law_edges(20000, 200000, seed=5)
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "mid.txt")
        datasets.write_edge_list(path, u, v)
        graph = ref.graph.Graph_j()
        graph.load(path, True, False)
    record["probe"] = {"runs": probe_runs(os.path.join(ROOT, "profiles", "r02_hogwild_probe_20k.txt")),
                       "auc": PROBE_AUC, "auc_note": PROBE_AUC_NOTE,
                       "id2name_sha256": hashlib.sha256("\n".join(graph.id2name).encode()).hexdigest()}
    with open(out_path, "w") as fout:
        json.dump(record, fout, indent=1, sort_keys=True)
        fout.write("\n")


if __name__ == "__main__":
    main(sys.argv[1])
