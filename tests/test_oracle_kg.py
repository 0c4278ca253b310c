"""CPU checks of the knowledge-graph oracle (oracle/gv_oracle_kg.cpp).

The loader is pinned against what the reference object loaded (tests/golden/reference_surface.json, recorded by
oracle/record_reference_surface.py) and against the product's loader.  The solver and kernels are NOT yet pinned
against reference output (their goldens need a GPU, oracle/make_golden.py kg_*): what is checked here is internal
consistency -- backward is the gradient of forward, the tied schedule covers every block exactly once without sharing
a partition inside a step, pools hold valid triplets of the right block, training lowers the loss and ranks true
triplets first -- so that a wrong restatement is caught before it is used to judge CUDA code.
"""
import hashlib
import json
import os

import numpy as np
import pytest

import oracle_kg_lib as K
import oracle_lib as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RECORDED = os.path.join(ROOT, "tests", "golden", "reference_surface.json")


def toy_triplets(seed=0, num_entity=60, num_relation=5, num_triplet=900):
    """relation r maps entity e to (e * (r + 2) + r) mod n: learnable structure, ragged degrees"""
    rng = np.random.default_rng(seed)
    heads = rng.zipf(1.6, num_triplet) % num_entity
    relations = rng.integers(0, num_relation, num_triplet)
    tails = (heads * (relations + 2) + relations) % num_entity
    return [("e%d" % h, "r%d" % r, "e%d" % t) for h, r, t in zip(heads, relations, tails)]


# ---- loader ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("normalization", [False, True])
def test_loader_matches_the_product_loader(tmp_path, normalization):
    import graphvite_b200 as gv
    from graphvite_b200 import _lib
    triplets = [(h, r, t, 0.5 + (i % 5) * 0.25) for i, (h, r, t) in enumerate(toy_triplets())]
    path = str(tmp_path / "kg.txt")
    with open(path, "w") as out:
        for h, r, t, w in triplets:
            out.write("%s\t%s\t%s\t%g\n" % (h, r, t, w))
    for source in (path, triplets):
        oracle = K.OracleKnowledgeGraph(source, normalization)
        product = gv.graph.KnowledgeGraph()
        product.load(source, normalization)
        assert (oracle.num_vertex, oracle.num_edge, oracle.num_relation) == \
            (product.num_vertex, product.num_edge, product.num_relation)
        assert oracle.id2entity() == product.id2entity and oracle.id2relation() == product.id2relation
        m = product.num_edge
        h, t, r = (np.zeros(m, dtype=np.uint32) for _ in range(3))
        w, vw = np.zeros(m, dtype=np.float32), np.zeros(product.num_vertex, dtype=np.float32)
        _lib.lib.gv_kgraph_flatten(product._handle, h.ctypes.data, t.ctypes.data, r.ctypes.data, w.ctypes.data, None,
                                   vw.ctypes.data)
        for ours, theirs in zip((h, t, r, w, vw), oracle.flat()):
            np.testing.assert_array_equal(ours, theirs)  # floats too: same accumulation order


def observe_toy_knowledge_graph(kg_class, tmp_path):
    """what the reference's KnowledgeGraph made of toy_triplets(3): counts, id maps, and digests of the head and
    tail columns of its anonymous save (head, tail, int(weight) in flatten order)"""
    graph = kg_class()
    graph.load(toy_triplets(3), False)
    path = str(tmp_path / "anonymous.txt")
    graph.save(path, True)
    columns = np.loadtxt(path, dtype=np.int64, ndmin=2)
    return {"counts": [graph.num_vertex, graph.num_edge, graph.num_relation], "id2entity": list(graph.id2entity),
            "id2relation": list(graph.id2relation), "heads": int64_digest(columns[:, 0]),
            "tails": int64_digest(columns[:, 1])}


def int64_digest(values):
    return hashlib.sha256(np.ascontiguousarray(values, dtype="<i8").tobytes()).hexdigest()


def test_loader_matches_the_live_reference():
    with open(RECORDED) as fin:
        theirs = json.load(fin)["kg_toy_triplets"]
    oracle = K.OracleKnowledgeGraph(toy_triplets(3))
    assert theirs["counts"] == [oracle.num_vertex, oracle.num_edge, oracle.num_relation]
    assert theirs["id2entity"] == oracle.id2entity() and theirs["id2relation"] == oracle.id2relation()
    h, t, r, w, _ = oracle.flat()
    assert theirs["heads"] == int64_digest(h)
    assert theirs["tails"] == int64_digest(t)


# ---- models: backward is the gradient of forward ----------------------------------------------------
def numeric_gradient(model, head, tail, relation, margin, which, epsilon=1e-3):
    base = [head.astype(np.float64), tail.astype(np.float64), relation.astype(np.float64)]
    grad = np.zeros(len(base[which]))
    for i in range(len(grad)):
        values = []
        for sign in (1, -1):
            x = [v.copy() for v in base]
            x[which][i] += sign * epsilon
            values.append(K.forward(model, x[0], x[1], x[2], margin))
        grad[i] = (values[0] - values[1]) / (2 * epsilon)
    return grad


@pytest.mark.parametrize("model", K.MODELS)
def test_backward_is_the_gradient_of_forward(model):
    """plain SGD, no weight decay, no l3: one positive sample moves every row by -lr * (prob - 1) * dlogit/drow"""
    rng = np.random.default_rng(1)
    dim = 64
    entity = rng.uniform(-0.6, 0.6, (4, dim)).astype(np.float32)
    relation = rng.uniform(-0.8, 0.8, (2, dim)).astype(np.float32)
    before_e, before_r = entity.copy(), relation.copy()
    margin_or_l3 = 3.0 if model in ("TransE", "RotatE") else 0.0
    lr = 0.01
    batch = np.array([[1, 2, 0]], dtype=np.uint32)  # relation 1, tail 2, head 0
    negatives = np.zeros((1, 0), dtype=np.uint32)
    loss = K.train_batch(model, dim, entity, relation, None, batch, negatives, (0, lr, 0.0, 0, 0, 0),
                         margin_or_l3=margin_or_l3, adversarial_temperature=0.0)
    logit = K.forward(model, before_e[0], before_e[2], before_r[1], margin_or_l3)
    prob = 1 / (1 + np.exp(-logit))
    assert loss[0] == pytest.approx(-np.log(prob + 1e-15) / 2, rel=1e-4)  # kEpsilon, util/common.h:28
    width = dim // 2 if model == "RotatE" else dim  # RotatE relations are dim/2 phases
    for which, (after, before, count) in enumerate([(entity[0], before_e[0], dim), (entity[2], before_e[2], dim),
                                                    (relation[1], before_r[1], width)]):
        if model == "QuatE" and which == 2:
            # the reference differentiates the Hamilton product only and treats the relation's norm as a constant
            # (model/knowledge_graph.h:661-664): its relation update is not the gradient of its own forward
            continue
        expected = -lr * (prob - 1) * numeric_gradient(model, before_e[0], before_e[2], before_r[1], margin_or_l3, which)
        np.testing.assert_allclose((after - before)[:count], expected[:count], rtol=2e-2, atol=2e-5)
    # rows not named by the sample are untouched
    np.testing.assert_array_equal(entity[[1, 3]], before_e[[1, 3]])
    np.testing.assert_array_equal(relation[0], before_r[0])


def test_negative_ids_corrupt_head_below_num_head_and_tail_above():
    rng = np.random.default_rng(2)
    dim, model = 32, "TransE"
    head_matrix = rng.uniform(-0.5, 0.5, (3, dim)).astype(np.float32)
    tail_matrix = rng.uniform(-0.5, 0.5, (4, dim)).astype(np.float32)
    relation = rng.uniform(-0.5, 0.5, (1, dim)).astype(np.float32)
    batch = np.array([[0, 1, 0]], dtype=np.uint32)  # relation 0, tail 1, head 0
    for negative, touched_head, touched_tail in ((2, [0, 2], [1]), (3 + 3, [0], [1, 3])):
        h, t, r = head_matrix.copy(), tail_matrix.copy(), relation.copy()
        K.train_batch(model, dim, h, r, None, batch, np.array([[negative]], dtype=np.uint32), (0, 0.05, 0.0, 0, 0, 0),
                      margin_or_l3=2.0, adversarial_temperature=0.0, tail=t)
        changed_h = [i for i in range(3) if not np.array_equal(h[i], head_matrix[i])]
        changed_t = [i for i in range(4) if not np.array_equal(t[i], tail_matrix[i])]
        assert changed_h == touched_head and changed_t == touched_tail


def test_self_adversarial_weights_follow_the_softmax_of_negative_logits():
    """with lr = 0 nothing moves, so the loss is the closed form (gpu/knowledge_graph.cuh:59-110)"""
    rng = np.random.default_rng(4)
    dim, k, temperature, margin = 32, 6, 1.5, 4.0
    entity = rng.uniform(-0.5, 0.5, (10, dim)).astype(np.float32)
    relation = rng.uniform(-3, 3, (2, dim)).astype(np.float32)
    batch = np.array([[1, 4, 2]], dtype=np.uint32)
    negatives = rng.integers(0, 20, (1, k)).astype(np.uint32)  # < 10 corrupts the head, >= 10 the tail
    loss = K.train_batch("RotatE", dim, entity, relation, None, batch, negatives, (0, 0.0, 0.0, 0, 0, 0),
                         margin_or_l3=margin, adversarial_temperature=temperature)
    logits = []
    for n in negatives[0]:
        h, t = (n, 4) if n < 10 else (2, n - 10)
        logits.append(K.forward("RotatE", entity[h], entity[t], relation[1], margin))
    logits = np.array(logits, dtype=np.float64)
    weights = np.exp((logits - logits[0]) / temperature)
    weights = np.minimum(weights / weights.sum(), 1)
    positive = K.forward("RotatE", entity[2], entity[4], relation[1], margin)
    sig = lambda x: 1 / (1 + np.exp(-x))
    expected = (-np.log(sig(positive) + 1e-15) + (weights * -np.log(1 - sig(logits) + 1e-15)).sum()) / 2
    assert loss[0] == pytest.approx(expected, rel=1e-4)
    uniform = K.train_batch("RotatE", dim, entity, relation, None, batch, negatives, (0, 0.0, 0.0, 0, 0, 0),
                            margin_or_l3=margin, adversarial_temperature=0.0)
    expected = (-np.log(sig(positive) + 1e-15) + (-np.log(1 - sig(logits) + 1e-15)).mean()) / 2
    assert uniform[0] == pytest.approx(expected, rel=1e-4)


@pytest.mark.parametrize("optimizer", list(O.OPTIMIZERS))
def test_every_optimizer_updates_rows_and_moments(optimizer):
    rng = np.random.default_rng(5)
    dim = 32
    entity = rng.uniform(-0.5, 0.5, (6, dim)).astype(np.float32)
    relation = rng.uniform(-1, 1, (2, dim)).astype(np.float32)
    otype = O.OPTIMIZERS[optimizer][0]
    num_moment = 0 if otype == 0 else (2 if otype == 4 else 1)
    moments = [np.zeros_like(entity) if num_moment >= 1 else None, np.zeros_like(relation) if num_moment >= 1 else None,
               np.zeros_like(entity) if num_moment >= 2 else None, np.zeros_like(relation) if num_moment >= 2 else None]
    before = entity.copy()
    batch = np.array([[0, 1, 0], [1, 3, 2]], dtype=np.uint32)
    negatives = np.array([[4, 7], [5, 11]], dtype=np.uint32)
    loss = K.train_batch("RotatE", dim, entity, relation, moments if num_moment else None, batch, negatives,
                         O.OPTIMIZERS[optimizer], margin_or_l3=6.0)
    assert np.isfinite(loss).all() and (loss > 0).all()
    assert not np.array_equal(entity[0], before[0]) and np.isfinite(entity).all()
    for m in moments[:2 * num_moment]:
        assert np.abs(m).max() > 0


# ---- solver ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("num_worker,num_partition", [(1, 2), (1, 4), (2, 4), (2, 8), (4, 8), (4, 16), (8, 16)])
def test_tied_schedule_covers_every_block_once_with_disjoint_partitions(num_worker, num_partition):
    graph = K.OracleKnowledgeGraph(toy_triplets())
    solver = K.OracleKGSolver(graph, 32, num_worker, 1)
    solver.build("SGD", num_partition, 2, 50, 2)
    schedule = solver.schedule(num_worker)
    seen = set()
    for step in schedule:
        used = []
        for head, tail in step:
            assert (head, tail) not in seen
            seen.add((int(head), int(tail)))
            used += [int(head)] if head == tail else [int(head), int(tail)]
        assert len(used) == len(set(used))  # tied weights: no partition in two blocks of one step
    assert len(seen) == num_partition * num_partition


def test_minimum_partitions_follow_tied_weights():
    graph = K.OracleKnowledgeGraph(toy_triplets())
    assert K.OracleKGSolver(graph, 32, 1, 1).build("SGD", 0, 2, 50, 2) is None
    solver = K.OracleKGSolver(graph, 32, 2, 1)
    solver.build("SGD", 0, 2, 50, 2)
    assert solver.info()["num_partition"] == 4
    with pytest.raises(RuntimeError, match="no less than 4"):
        K.OracleKGSolver(graph, 32, 2, 1).build("SGD", 2, 2, 50, 2)


@pytest.mark.parametrize("num_partition,num_sampler", [(1, 1), (2, 3)])
def test_pools_hold_triplets_of_their_block(num_partition, num_sampler):
    triplets = toy_triplets(7)
    graph = K.OracleKnowledgeGraph(triplets)
    solver = K.OracleKGSolver(graph, 32, 1, num_sampler)
    solver.build("Adam", num_partition, 4, 100, 3)
    solver.train_begin("RotatE", num_epoch=1, sample_batch_size=37)
    part_of, local_of = solver.locations()
    names, relations = graph.id2entity(), graph.id2relation()
    known = set(triplets)
    global_of = {(int(p), int(l)): v for v, (p, l) in enumerate(zip(part_of, local_of))}
    for head in range(num_partition):
        for tail in range(num_partition):
            pool = solver.pool(1, head, tail)  # the first fill goes to pool_id ^ 1 = 1
            assert pool.shape == (300, 3)
            for r, t, h in pool[::7]:
                assert (names[global_of[(head, int(h))]], relations[r], names[global_of[(tail, int(t))]]) in known


@pytest.mark.parametrize("model,margin", [("RotatE", 6.0), ("TransE", 6.0), ("DistMult", 0.0), ("ComplEx", 0.0),
                                          ("SimplE", 0.0)])
def test_training_learns_the_toy_relations(model, margin):
    triplets = toy_triplets(11, num_entity=40, num_relation=3, num_triplet=600)
    graph = K.OracleKnowledgeGraph(triplets)
    solver = K.OracleKGSolver(graph, 32, 1, 1)
    solver.build((4, 5e-3, 0.0, 0.9, 0.999, 1e-8), 1, 8, 100, 4, schedule=0)
    solver.train(model=model, num_epoch=60, margin=margin, l3_regularization=0.0, sample_batch_size=50,
                 log_frequency=20)
    info = solver.info()
    assert info["batch_id"] >= info["num_batch"] and info["shuffle_partition"] == 1
    losses = solver.logged_loss()
    # the first log point shows the still-empty loss buffer; later ones the batch before (also across blocks:
    # 20 is a multiple of the episode size, so every log point is a block's first batch)
    assert losses[0] == 0 and np.isfinite(losses).all() and (losses[1:] > 0).all() and losses[2:].mean() < 0.45
    negatives = solver.last_negatives()
    assert negatives.max() < 2 * graph.num_vertex and info["last_negative_count"] == 2 * graph.num_vertex
    # true tails outrank random tails
    h, t, r, _, _ = graph.flat()
    true = np.stack([h, t, r], axis=1)[:200]
    corrupted = true.copy()
    corrupted[:, 1] = (corrupted[:, 1] + 1 + np.arange(len(true)) % 7) % graph.num_vertex
    assert (solver.predict(true) > solver.predict(corrupted)).mean() > 0.9


def test_relation_deltas_are_written_back_per_block():
    """global relation matrix after an episode = initial + sum of the per-block deltas (solver.h:1413-1420):
    with lr = 0 it must not move at all, with lr > 0 it must differ from its initial value"""
    graph = K.OracleKnowledgeGraph(toy_triplets(13))
    moved = []
    for lr in (0.0, 1e-2):
        solver = K.OracleKGSolver(graph, 32, 1, 1)
        solver.build((0, lr, 0.0, 0, 0, 0), 2, 4, 60, 2, schedule=0)
        solver.train_begin("TransE", num_epoch=1, margin=4, sample_batch_size=30)
        initial = solver.relation_embeddings.copy()
        entities = solver.entity_embeddings.copy()
        while solver.train_episode():
            pass
        moved.append(not np.array_equal(initial, solver.relation_embeddings))
        if lr == 0:
            np.testing.assert_array_equal(entities, solver.entity_embeddings)
    assert moved == [False, True]
