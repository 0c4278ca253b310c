"""Generate the golden vectors under tests/golden/ by running the UNMODIFIED reference.

TEST INFRASTRUCTURE.  Runs on a GPU box (the reference's solver needs a CUDA device):
    gpurun -- 'python oracle/make_golden.py gpurun_out/golden'
then copy gpurun_out/golden/*.npz into tests/golden/ and commit them.  The reference is driven
through oracle/_ref/libref_harness.so (oracle/ref_harness.cu, built by `make -C oracle ref`
here in the authoring container; /root/reference does not exist on the GPU box).
Inputs that the tests must share (the toy graph) are committed under tests/golden/ as well.
"""
import ctypes
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN = os.path.join(ROOT, "tests", "golden")
c = ctypes


EMULATED = "--emulated" in sys.argv  # the reference executed by tests/emu's CUDA emulation (`make -C oracle ref_emu`)


def load_harness():
    if EMULATED:
        # two-pass build (oracle/Makefile, ref_emu): launches swap the host-pass kernel for its device-pass twin
        os.environ["GV_EMU_DEVICE_LIBRARY"] = os.path.join(HERE, "_ref", "libref_harness_emu_device.so")
        os.environ["GV_EMU_DEVICE_NAMESPACE"] = "graphvite=graphvite_device"
        lib = c.CDLL(os.path.join(HERE, "_ref", "libref_harness_emu.so"), mode=c.RTLD_GLOBAL)
    else:
        lib = c.CDLL(os.path.join(HERE, "_ref", "libref_harness.so"))
    lib.ref_graph_load.restype = c.c_void_p
    lib.ref_graph_load.argtypes = [c.c_char_p, c.c_int, c.c_int]
    for name in ("ref_graph_num_vertex", "ref_graph_num_edge", "ref_graph_num_directed_edge"):
        getattr(lib, name).restype = c.c_uint64
        getattr(lib, name).argtypes = [c.c_void_p]
    lib.ref_graph_flat.argtypes = [c.c_void_p] * 5
    lib.ref_solver_new.restype = c.c_void_p
    lib.ref_solver_new.argtypes = [c.c_int, c.c_int, c.c_int, c.c_uint64]
    lib.ref_solver_free.argtypes = [c.c_void_p]
    lib.ref_solver_build.argtypes = [c.c_void_p, c.c_void_p, c.c_int, c.c_int, c.c_float, c.c_float, c.c_float,
                                     c.c_float, c.c_float, c.c_int, c.c_int, c.c_int, c.c_int]
    lib.ref_solver_train.argtypes = [c.c_void_p, c.c_char_p, c.c_int, c.c_int, c.c_int, c.c_int, c.c_int, c.c_int,
                                     c.c_float, c.c_float, c.c_int, c.c_float, c.c_float, c.c_int]
    lib.ref_solver_info.argtypes = [c.c_void_p, c.c_void_p]
    lib.ref_solver_locations.argtypes = [c.c_void_p, c.c_void_p, c.c_void_p]
    lib.ref_solver_pool.argtypes = [c.c_void_p, c.c_int, c.c_int, c.c_int, c.c_void_p]
    lib.ref_solver_embeddings.argtypes = [c.c_void_p, c.c_int, c.c_void_p]
    lib.ref_solver_last_negatives.argtypes = [c.c_void_p, c.c_void_p]
    lib.ref_solver_last_loss.argtypes = [c.c_void_p, c.c_void_p]
    lib.ref_solver_edge_table.argtypes = [c.c_void_p, c.c_void_p, c.c_void_p]
    lib.ref_solver_negative_table.argtypes = [c.c_void_p, c.c_void_p, c.c_void_p]
    lib.ref_solver_predict.argtypes = [c.c_void_p, c.c_void_p, c.c_uint64, c.c_void_p]
    lib.ref_alias_build.argtypes = [c.c_void_p, c.c_uint64, c.c_void_p, c.c_void_p]
    lib.ref_alias_sample_cpu.argtypes = [c.c_void_p, c.c_uint64, c.c_void_p, c.c_uint64, c.c_void_p]
    lib.ref_alias_sample_gpu.argtypes = [c.c_void_p, c.c_uint32, c.c_void_p, c.c_int, c.c_void_p]
    lib.ref_curand.argtypes = [c.c_uint64, c.c_void_p, c.c_int, c.c_void_p]
    lib.ref_draw_seed.restype = c.c_uint64
    lib.ref_kernel_train.argtypes = [c.c_int, c.c_int, c.c_float, c.c_float, c.c_float, c.c_float, c.c_float,
                                     c.c_uint64, c.c_uint64] + [c.c_void_p] * 8 + [c.c_int, c.c_int, c.c_float,
                                                                                   c.c_void_p]
    return lib


def ptr(array):
    return array.ctypes.data if array is not None else None


OPTIMIZERS = {
    # name: (type, lr, weight_decay, a, b, epsilon)
    "SGD": (0, 0.025, 0.005, 0.0, 0.0, 0.0),
    "Momentum": (1, 0.01, 0.001, 0.9, 0.0, 0.0),
    "AdaGrad": (2, 0.05, 0.001, 0.0, 0.0, 1e-10),
    "RMSprop": (3, 0.001, 0.001, 0.99, 0.0, 1e-8),
    "Adam": (4, 0.001, 0.001, 0.9, 0.999, 1e-8),
}

# the solver cases; each is run on tests/golden/toy_graph.txt
SOLVER_CASES = {
    # name: dict(dim, P, k, B, E, S, model, epochs, aug, L, wb, shuffle_base, optimizer, undirected)
    "line_p1": dict(dim=32, P=1, k=1, B=500, E=4, S=1, model="LINE", epochs=4, aug=2, L=5, wb=10, sb=0,
                    optimizer="SGD"),
    "line_p2_s3": dict(dim=32, P=2, k=3, B=400, E=3, S=3, model="LINE", epochs=8, aug=3, L=7, wb=8, sb=0,
                       optimizer="SGD"),
    "deepwalk_p1": dict(dim=128, P=1, k=2, B=300, E=5, S=2, model="DeepWalk", epochs=3, aug=4, L=9, wb=6, sb=0,
                        optimizer="SGD"),
    "edge_p2": dict(dim=32, P=2, k=1, B=500, E=2, S=2, model="LINE", epochs=3, aug=1, L=5, wb=10, sb=0,
                    optimizer="SGD"),
    "line_p3_adam": dict(dim=32, P=3, k=2, B=300, E=2, S=1, model="LINE", epochs=4, aug=2, L=6, wb=10, sb=0,
                         optimizer="Adam"),
    "node2vec_p2": dict(dim=32, P=2, k=1, B=400, E=3, S=2, model="node2vec", epochs=5, aug=3, L=8, wb=10, sb=0,
                        optimizer="SGD", p=0.5, q=2.0),
    "node2vec_p1": dict(dim=32, P=1, k=2, B=500, E=2, S=1, model="node2vec", epochs=3, aug=2, L=5, wb=10, sb=0,
                        optimizer="SGD", p=4.0, q=0.25),
}


def make_toy_graph(path):
    """A small weighted graph with comments, blank lines, a self loop and repeated edges."""
    rng = np.random.RandomState(7)
    n, m = 300, 1500
    weights = (np.arange(1, n + 1) ** -0.9)
    cdf = np.cumsum(weights) / weights.sum()
    u = np.searchsorted(cdf, rng.rand(m))
    v = np.searchsorted(cdf, rng.rand(m))
    u[:n] = rng.permutation(n)
    lines = ["# toy graph for the golden vectors", ""]
    for i in range(m):
        a, b = int(u[i]), int(v[i])
        if i == 17:
            b = a  # one self loop (added once even when as_undirected, graph.cuh:148-151)
        elif a == b:
            b = (b + 1) % n
        if i % 5 == 0:
            lines.append("n%d\tn%d\t%.2f" % (a, b, 0.5 + 2 * rng.rand()))
        elif i % 7 == 0:
            lines.append("n%d n%d  # trailing comment" % (a, b))
        else:
            lines.append("n%d n%d" % (a, b))
    with open(path, "w") as fout:
        fout.write("\n".join(lines) + "\n")


def main(out_dir, only=None):
    os.makedirs(out_dir, exist_ok=True)
    lib = load_harness()
    toy = os.path.join(GOLDEN, "toy_graph.txt")
    if not os.path.exists(toy):
        make_toy_graph(toy)

    if not only:
        write_basics(lib, out_dir, toy)
    write_solver_cases(lib, out_dir, toy, only)


def write_basics(lib, out_dir, toy):
    # ---- process-wide engine + cuRAND stream ---------------------------------------------
    lib.ref_reset_engine()
    seeds = np.array([lib.ref_draw_seed() for _ in range(6)], dtype=np.uint64)
    chunks = np.array([1000, 7000, 12000], dtype=np.uint64)
    small = np.zeros(int(chunks.sum()), dtype=np.float64)
    lib.ref_curand(int(seeds[0]), ptr(chunks), len(chunks), ptr(small))
    big_chunks = np.array([5000000, 5000000], dtype=np.uint64)
    big = np.zeros(int(big_chunks.sum()), dtype=np.float64)
    lib.ref_curand(int(seeds[1]), ptr(big_chunks), len(big_chunks), ptr(big))
    np.savez_compressed(os.path.join(out_dir, "curand.npz"), seeds=seeds, small_chunks=chunks, small=small,
                        big_seed=seeds[1], big_head=big[:8192], big_mid=big[5000000 - 2048:5000000 + 2048],
                        big_tail=big[-4096:], big_sum=np.array([big[:5000000].sum(), big[5000000:].sum()]))

    # ---- alias tables -----------------------------------------------------------------------
    rng = np.random.RandomState(11)
    weights = (rng.pareto(1.5, 1000) + 0.01).astype(np.float32)
    prob = np.zeros(1000, dtype=np.float32)
    alias = np.zeros(1000, dtype=np.uint64)
    lib.ref_alias_build(ptr(weights), 1000, ptr(prob), ptr(alias))
    random = rng.rand(2 * 4000)
    random[random == 0] = 0.5
    cpu_samples = np.zeros(4000, dtype=np.uint64)
    lib.ref_alias_sample_cpu(ptr(weights), 1000, ptr(random), 4000, ptr(cpu_samples))
    gpu_samples = np.zeros(4000, dtype=np.uint32)
    lib.ref_alias_sample_gpu(ptr(weights), 1000, ptr(random), 4000, ptr(gpu_samples))
    uniform = np.ones(37, dtype=np.float32)
    uprob = np.zeros(37, dtype=np.float32)
    ualias = np.zeros(37, dtype=np.uint64)
    lib.ref_alias_build(ptr(uniform), 37, ptr(uprob), ptr(ualias))
    np.savez_compressed(os.path.join(out_dir, "alias.npz"), weights=weights, prob=prob, alias=alias, random=random,
                        cpu_samples=cpu_samples, gpu_samples=gpu_samples, uniform_prob=uprob, uniform_alias=ualias)

    # ---- graph loading ------------------------------------------------------------------------
    for undirected in (1, 0):
        for normalization in (0, 1):
            g = lib.ref_graph_load(toy.encode(), undirected, normalization)
            n, m = lib.ref_graph_num_vertex(g), lib.ref_graph_num_directed_edge(g)
            u = np.zeros(m, dtype=np.uint32)
            v = np.zeros(m, dtype=np.uint32)
            w = np.zeros(m, dtype=np.float32)
            vw = np.zeros(n, dtype=np.float32)
            lib.ref_graph_flat(g, ptr(u), ptr(v), ptr(w), ptr(vw))
            np.savez_compressed(os.path.join(out_dir, "graph_u%d_n%d.npz" % (undirected, normalization)),
                                num_vertex=n, num_edge=lib.ref_graph_num_edge(g), u=u, v=v, w=w, vertex_weights=vw)



def write_solver_cases(lib, out_dir, toy, only):
    # ---- solver runs ----------------------------------------------------------------------------
    graph = lib.ref_graph_load(toy.encode(), 1, 0)
    num_vertex = lib.ref_graph_num_vertex(graph)
    num_directed = lib.ref_graph_num_directed_edge(graph)
    for name, cfg in SOLVER_CASES.items():
        if only and name not in only:
            continue
        lib.ref_reset_engine()
        solver = lib.ref_solver_new(cfg["dim"], 1, cfg["S"], 4 << 30)
        otype, lr, wd, a, b, eps = OPTIMIZERS[cfg["optimizer"]]
        lib.ref_solver_build(solver, graph, otype, 1, lr, wd, a, b, eps, cfg["P"], cfg["k"], cfg["B"], cfg["E"])
        lib.ref_solver_train(solver, cfg["model"].encode(), cfg["epochs"], 0, cfg["aug"], cfg["L"], cfg["wb"],
                             cfg["sb"], cfg.get("p", 1.0), cfg.get("q", 1.0), 1, 0.75, 5.0, 1000)
        info = np.zeros(10, dtype=np.int32)
        lib.ref_solver_info(solver, ptr(info))
        P, E, B = int(info[0]), int(info[1]), int(info[2])
        part_of = np.zeros(num_vertex, dtype=np.int32)
        local_of = np.zeros(num_vertex, dtype=np.uint32)
        lib.ref_solver_locations(solver, ptr(part_of), ptr(local_of))
        pools = np.zeros((2, P, P, E * B, 2), dtype=np.uint32)
        for side in range(2):
            for h in range(P):
                for t in range(P):
                    lib.ref_solver_pool(solver, side, h, t, ptr(pools[side, h, t]))
        vertex = np.zeros((num_vertex, cfg["dim"]), dtype=np.float32)
        context = np.zeros((num_vertex, cfg["dim"]), dtype=np.float32)
        lib.ref_solver_embeddings(solver, 0, ptr(vertex))
        lib.ref_solver_embeddings(solver, 1, ptr(context))
        negatives = np.zeros(B * cfg["k"], dtype=np.uint32)
        lib.ref_solver_last_negatives(solver, ptr(negatives))
        loss = np.zeros(B, dtype=np.float32)
        lib.ref_solver_last_loss(solver, ptr(loss))
        edge_prob = np.zeros(num_directed, dtype=np.float32)
        edge_alias = np.zeros(num_directed, dtype=np.uint64)
        lib.ref_solver_edge_table(solver, ptr(edge_prob), ptr(edge_alias))
        pairs = np.random.RandomState(3).randint(0, num_vertex, (500, 2)).astype(np.uint32)
        logits = np.zeros(500, dtype=np.float32)
        lib.ref_solver_predict(solver, ptr(pairs), 500, ptr(logits))
        np.savez_compressed(os.path.join(out_dir, "solver_%s.npz" % name), info=info, part_of=part_of,
                            local_of=local_of, pools=pools, vertex=vertex, context=context, negatives=negatives,
                            loss=loss, edge_prob=edge_prob, edge_alias=edge_alias, pairs=pairs, logits=logits,
                            **{"cfg_" + k: np.array(v) for k, v in cfg.items()})
        lib.ref_solver_free(solver)
        print("solver case", name, "info", info.tolist(), flush=True)

    if not only:
        write_kernel_cases(lib, out_dir)
    print("golden vectors written to", out_dir)


# Solver runs whose embeddings tests/test_emulated_reference.py compares with the oracle's.  Only the emulated
# reference processes a batch in order, like the oracle, so these are recorded with --emulated:
#     python oracle/make_golden.py --emulated --oracle-check tests/golden
# Both embedding matrices are kept whole, and predict on the run's pairs.
ORACLE_CHECK_CASES = ("line_p1", "edge_p2", "node2vec_p1")


def write_oracle_check_cases(lib, out_dir, toy):
    import tempfile
    with tempfile.TemporaryDirectory() as tmp:
        write_solver_cases(lib, tmp, toy, set(ORACLE_CHECK_CASES))
        for name in ORACLE_CHECK_CASES:
            g = np.load(os.path.join(tmp, "solver_%s.npz" % name))
            np.savez_compressed(os.path.join(out_dir, "emu_reference_solver_%s.npz" % name), vertex=g["vertex"],
                                context=g["context"], logits=g["logits"])


def write_kernel_cases(lib, out_dir):
    # ---- the reference kernels on race-free batches ---------------------------------------------
    for dim in (32, 128):
        for oname, (otype, lr, wd, a, b, eps) in OPTIMIZERS.items():
            rng = np.random.RandomState(100 + dim + otype)
            n, k = 64, 2
            num_v, num_c = 80, 256
            vertex = (rng.rand(num_v, dim).astype(np.float32) - 0.5) * 0.6
            context = (rng.rand(num_c, dim).astype(np.float32) - 0.5) * 0.6
            moments = [np.abs(rng.randn(*shape).astype(np.float32)) * 0.01
                       for shape in ((num_v, dim), (num_c, dim), (num_v, dim), (num_c, dim))]
            heads = rng.permutation(num_v)[:n].astype(np.uint32)
            tails = rng.permutation(num_c)[:n * (k + 1)].astype(np.uint32).reshape(n, k + 1)
            batch = np.stack([tails[:, k], heads], axis=1).astype(np.uint32)  # {tail, head}
            negatives = np.ascontiguousarray(tails[:, :k])
            before = dict(vertex=vertex.copy(), context=context.copy(), vm1=moments[0].copy(), cm1=moments[1].copy(),
                          vm2=moments[2].copy(), cm2=moments[3].copy())
            loss = np.zeros(n, dtype=np.float32)
            lib.ref_kernel_train(dim, otype, lr, wd, a, b, eps, num_v, num_c, ptr(vertex), ptr(context),
                                 ptr(moments[0]), ptr(moments[1]), ptr(moments[2]), ptr(moments[3]), ptr(batch),
                                 ptr(negatives), n, k, 5.0, ptr(loss))
            np.savez_compressed(os.path.join(out_dir, "kernel_d%d_%s.npz" % (dim, oname)), batch=batch,
                                negatives=negatives, loss=loss, after_vertex=vertex, after_context=context,
                                after_vm1=moments[0], after_cm1=moments[1], after_vm2=moments[2],
                                after_cm2=moments[3], hyper=np.array([otype, lr, wd, a, b, eps, 5.0]),
                                **{"before_" + key: value for key, value in before.items()})


if __name__ == "__main__":
    arguments = [a for a in sys.argv[1:] if a not in ("--emulated", "--oracle-check")]
    if "--oracle-check" in sys.argv:
        write_oracle_check_cases(load_harness(), arguments[0], os.path.join(GOLDEN, "toy_graph.txt"))
        sys.exit(0)
    main(arguments[0] if arguments else os.path.join(ROOT, "gpurun_out", "golden"), set(arguments[1:]) or None)
