"""Child interpreter of tests/test_gpu_x_pybind.py: trains through the compiled pybind11 module `libgraphvite` (ours).
Its own process because the reference's module has the same name and may already live in the test session."""
import importlib.util
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
PATH = os.path.join(ROOT, "graphvite_b200", "pybind", "libgraphvite.so")
TOY = os.path.join(ROOT, "tests", "golden", "toy_graph.txt")
TOY_KG = os.path.join(ROOT, "tests", "golden", "toy_kg.txt")


def load():
    spec = importlib.util.spec_from_file_location("libgraphvite", PATH)
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    assert m.__backend__ == "libgv_b200"
    return m


def graph_solver_matches_the_ctypes_mirror(module, repeat=4):
    """Hogwild training on the toy graph loses a varying share of racing updates, and which share follows the state
    of the GPU (single runs spread by several percent, drifting over a process's first runs), so the two front ends
    train alternately and their embedding norms are compared as means over `repeat` runs of each."""
    import graphvite_b200 as gv
    from graphvite_b200 import _lib
    train = dict(model="LINE", num_epoch=40, augmentation_step=2, random_walk_length=5, random_walk_batch_size=10)

    norms, mirror_norms = [], []
    for _ in range(repeat):
        _lib.lib.gv_reset_global_engine(5489)
        graph = module.graph.Graph_j()
        graph.load(TOY)
        solver = module.solver.GraphSolver_32_f_j([0], 1, 0)
        solver.build(graph, module.optimizer.SGD(0.025, 0.005), 1, 1, 500, 4)
        assert (solver.num_partition, solver.batch_size, solver.episode_size, solver.num_negative) == (1, 500, 4, 1)
        solver.train(**train)
        assert solver.model == "LINE" and solver.augmentation_step == 2
        vertex, context = solver.vertex_embeddings, solver.context_embeddings
        assert vertex.shape == (graph.num_vertex, 32) and vertex.dtype == np.float32 and not vertex.flags.owndata
        norms.append((float(np.linalg.norm(vertex)), float(np.linalg.norm(context))))

        _lib.lib.gv_reset_global_engine(5489)
        graph2 = gv.graph.Graph()
        graph2.load(TOY)
        mirror = gv.solver.GraphSolver(32, device_ids=[0], num_sampler_per_worker=1)
        mirror.build(graph2, gv.optimizer.SGD(0.025, 0.005), 1, 1, 500, 4)
        mirror.train(**train)
        mirror_norms.append((float(np.linalg.norm(mirror.vertex_embeddings)),
                             float(np.linalg.norm(mirror.context_embeddings))))
        mirror.close()
    for a, b in zip(np.mean(norms, axis=0), np.mean(mirror_norms, axis=0)):
        assert np.isfinite(a) and abs(a - b) <= 0.05 * b, (norms, mirror_norms)
    # the views alias the solver's memory: predict sees an edit made through them
    pairs = np.array([[0, 1], [2, 3]], dtype=np.uint32)
    before = solver.predict(pairs)
    np.testing.assert_allclose(before, np.einsum("ij,ij->i", vertex[pairs[:, 0]], context[pairs[:, 1]]), rtol=1e-4,
                               atol=1e-6)
    solver.vertex_embeddings[0] *= 2
    np.testing.assert_allclose(solver.predict(pairs)[0], 2 * before[0], rtol=1e-4, atol=1e-6)
    solver.clear()


def custom_schedule_and_knowledge_graph_solver(module):
    calls = []

    def schedule(batch_id, num_batch):
        calls.append((batch_id, num_batch))
        return 1.0 - batch_id / num_batch

    graph = module.graph.Graph_j()
    graph.load(TOY)
    solver = module.solver.GraphSolver_64_f_j([0])
    solver.build(graph, module.optimizer.SGD(0.025, 0.005, schedule), num_negative=2, batch_size=300, episode_size=2)
    solver.train("DeepWalk", num_epoch=10, augmentation_step=3, random_walk_length=6, random_walk_batch_size=8)
    assert calls and all(n == calls[0][1] for _, n in calls) and np.isfinite(solver.vertex_embeddings).all()

    kg = module.graph.KnowledgeGraph_j()
    kg.load(TOY_KG)
    ksolver = module.solver.KnowledgeGraphSolver_32_f_j([0])
    ksolver.build(kg, module.optimizer.Adam(1e-3), num_negative=3, batch_size=60, episode_size=2)
    ksolver.train("RotatE", num_epoch=3, margin=6, sample_batch_size=37)
    assert ksolver.entity_embeddings.shape == (kg.num_vertex, 32)
    assert ksolver.relation_embeddings.shape[0] == kg.num_relation
    triplets = np.array([[0, 1, 0], [2, 3, 1]], dtype=np.uint32)
    assert np.isfinite(ksolver.predict(triplets)).all()


if __name__ == "__main__":
    {"graph": graph_solver_matches_the_ctypes_mirror, "schedule_kg": custom_schedule_and_knowledge_graph_solver}[
        sys.argv[1]](load())
    print("ok")
