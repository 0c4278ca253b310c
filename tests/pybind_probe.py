"""Loads ONE pybind11 module named `libgraphvite` from the path in argv[1] and prints what tests/test_pybind_module.py
compares, as JSON.  A separate process per module: two extension modules with the same name (the reference's and
ours) cannot live in one interpreter -- their `libgraphvite.solver` submodules would share one sys.modules entry."""
import hashlib
import importlib.util
import json
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOY = os.path.join(ROOT, "tests", "golden", "toy_graph.txt")


def file_digest(path):
    with open(path, "rb") as fin:
        return hashlib.sha256(fin.read()).hexdigest()


def public(obj):
    return sorted(name for name in dir(obj) if not name.startswith("_"))


def main():
    spec = importlib.util.spec_from_file_location("libgraphvite", sys.argv[1])
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    m.init_logging(m.ERROR, "", False)
    out = {"top": public(m), "solver": public(m.solver), "graph": public(m.graph), "optimizer": public(m.optimizer),
           "auto": m.auto, "units": [m.KiB(3), m.MiB(3), m.GiB(3)],
           "dtype2name": {k.name: v for k, v in m.dtype2name.items()}, "docs": {}, "attributes": {}}
    for cls in ("GraphSolver_128_f_j", "KnowledgeGraphSolver_2048_f_j"):
        out["attributes"][cls] = public(getattr(m.solver, cls))
        for method in ("build", "train", "predict", "clear"):
            out["docs"]["%s.%s" % (cls, method)] = getattr(getattr(m.solver, cls), method).__doc__
    # graph: load / map / save
    graphs = {}
    with tempfile.TemporaryDirectory() as tmp:
        g = m.graph.Graph_j()
        g.load(TOY, True, False)
        g.save(os.path.join(tmp, "toy.txt"), True, False)
        graphs["file"] = {"num_vertex": g.num_vertex, "num_edge": g.num_edge, "as_undirected": g.as_undirected,
                          "normalization": g.normalization, "id2name": list(g.id2name), "name2id": dict(g.name2id),
                          "saved_sha256": file_digest(os.path.join(tmp, "toy.txt"))}
        g.load([("a", "b"), ("b", "c"), ("c", "a"), ("a", "a")], as_undirected=False)
        graphs["edge_list"] = {"num_vertex": g.num_vertex, "num_edge": g.num_edge, "name2id": dict(g.name2id)}
        g.load([("x", "y", 2.0), ("y", "z", 0.5)], normalization=True)
        g.save(os.path.join(tmp, "w.txt"))
        graphs["weighted"] = {"saved": open(os.path.join(tmp, "w.txt")).read()}
    out["graphs"] = graphs
    fields = {"SGD": ("lr", "weight_decay"), "Momentum": ("lr", "weight_decay", "momentum"),
              "AdaGrad": ("lr", "weight_decay", "epsilon"), "RMSprop": ("lr", "weight_decay", "alpha", "epsilon"),
              "Adam": ("lr", "weight_decay", "beta1", "beta2", "epsilon")}
    optimizers = {}
    for name, names in fields.items():
        default = getattr(m.optimizer, name)()
        values = [0.5, 0.25, 0.75, 0.875, 0.125][:len(names)]
        positional = getattr(m.optimizer, name)(*values)
        constant = getattr(m.optimizer, name)(schedule="constant")
        custom = getattr(m.optimizer, name)(schedule=lambda batch_id, num_batch: 0.5)
        optimizers[name] = {"type": default.type, "default": [float(getattr(default, f)) for f in names],
                            "positional": [float(getattr(positional, f)) for f in names],
                            "schedules": [default.schedule.type, constant.schedule.type, custom.schedule.type],
                            "custom_value": custom.schedule.schedule_function(3, 10)}
    optimizers["Optimizer(auto)"] = m.optimizer.Optimizer(m.auto).type
    optimizers["Optimizer(0.5)"] = m.optimizer.Optimizer(0.5).lr
    optimizers["LRSchedule"] = m.optimizer.LRSchedule("linear").type
    out["optimizers"] = optimizers
    out["backend"] = getattr(m, "__backend__", "reference")
    out["gib2"] = m.GiB(2)
    if out["backend"] != "reference":  # errors are exceptions in our module (the reference abort()s the process)
        try:
            m.optimizer.LRSchedule("cosine")
            out["bad_schedule"] = "accepted"
        except (ValueError, RuntimeError) as error:
            out["bad_schedule"] = type(error).__name__
        try:
            import torch
            have_gpu = torch.cuda.is_available()
        except Exception:
            have_gpu = False
        if not have_gpu:
            try:
                m.solver.GraphSolver_128_f_j([0], 0, 0)
                out["solver_without_gpu"] = "constructed"
            except RuntimeError as error:
                out["solver_without_gpu"] = "RuntimeError"
        try:
            m.solver.GraphSolver_128_f_j([0, 1], 0, 0)
            out["two_devices"] = "constructed"
        except RuntimeError as error:
            out["two_devices"] = str(error)[:200]
    print(json.dumps(out))


if __name__ == "__main__":
    main()
