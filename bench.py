#!/usr/bin/env python
"""bench.py -- edges/sec of LINE d=128 on a Youtube-shaped synthetic graph (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # our arm
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU-sampler + CUDA path

A "step" is one sub-episode: every GPU trains one (head block, tail block) of the sample pool,
episode_size * batch_size = 5e7 positive edges per GPU at the reference's Youtube configuration
(config/graph/line_youtube.yaml), while the samplers refill the other pool.  For N > 1 the script
is launched by torchrun, one rank per GPU; the value is the whole job's edges per second with the
time taken as the max over ranks of the device time (CUDA events on the solver's work stream).

Other workloads (`--workload`): blogcatalog / toy (LINE, small graphs), node2vec_youtube (config/graph/
node2vec_youtube.yaml with p = q = 0.25 on a degree-capped Youtube-shaped graph whose per-edge tables fit),
friendster_lite (config/graph/line_friendster.yaml on a 1/16-scale Friendster-shaped graph from binary edge
arrays), rotate_fb15k237 (config/knowledge_graph/rotate_fb15k-237.yaml, KnowledgeGraphSolver).
"""
import argparse
import importlib.util
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# config/graph/line_youtube.yaml
YOUTUBE = dict(solver="graph", dim=128, lr=0.025, weight_decay=0.005, num_negative=1, batch_size=100000,
               episode_size=500, model="LINE", negative_weight=5, augmentation_step=5, random_walk_length=40,
               random_walk_batch_size=100, p=1.0, q=1.0)
WORKLOADS = {
    "youtube": dict(YOUTUBE, graph="youtube"),
    "blogcatalog": dict(YOUTUBE, graph="blogcatalog", augmentation_step=2),  # config/demo/quick_start.yaml
    "toy": dict(YOUTUBE, graph="toy", batch_size=1000, episode_size=20, augmentation_step=2, random_walk_length=10),
    # config/graph/node2vec_youtube.yaml (augmentation 5 there too) with BASELINE.json's p = q = 0.25
    "node2vec_youtube": dict(YOUTUBE, graph="youtube_capped", model="node2vec", p=0.25, q=0.25),
    # config/graph/line_friendster.yaml: d=96 in the yaml, BASELINE.json quotes d=128; augmentation 2, episode 2500
    "friendster_lite": dict(YOUTUBE, graph="friendster_lite", augmentation_step=2, episode_size=2500),
    # the two configurations that need all 8 GPUs of a box (never run: the round had no 8-GPU lease long enough):
    #   torchrun --nnodes=1 --nproc-per-node 8 ... bench.py --gpus 8 --workload friendster            (65.6 M / 1.8 G)
    #   torchrun --nnodes=1 --nproc-per-node 8 ... bench.py --gpus 8 --workload node2vec_youtube_full (209 GB of tables)
    "friendster": dict(YOUTUBE, graph="friendster", augmentation_step=2, episode_size=2500),
    "node2vec_youtube_full": dict(YOUTUBE, graph="youtube", model="node2vec", p=0.25, q=0.25),
    # config/knowledge_graph/rotate_fb15k-237.yaml
    "rotate_fb15k237": dict(solver="kg", graph="fb15k-237", dim=2048, model="RotatE", lr=2e-6, weight_decay=0,
                            num_negative=64, batch_size=100000, episode_size=1, margin=9.0, adversarial_temperature=2.0,
                            l3_regularization=2e-3, sample_batch_size=2000),
}


def bytes_per_edge(dim, k):
    """Algorithmic HBM bytes per positive edge for SGD (SURVEY.md section 8d): vertex row R+W,
    k+1 context rows R+W, the {tail, head} pair, k negative ids, the loss."""
    return 8 * dim * (k + 2) + 8 + 4 * k + 4


def graph_file(name):
    """Synthetic edge list with the published |V| / |E| (no network: real datasets are unavailable)."""
    from graphvite_b200 import datasets
    path = "/tmp/gv_b200_%s.txt" % name
    if not os.path.exists(path):
        u, v = datasets.named_edges(name)
        import pandas
        pandas.DataFrame({"u": u, "v": v}).to_csv(path + ".tmp", sep="\t", header=False, index=False)
        os.replace(path + ".tmp", path)
    return path


def heldout_pairs(name, count=50000):
    """Link-prediction evaluation set for a synthetic graph: `count` edges drawn from the SAME generative model with
    another seed (label 1; they are held out in the sense that the training graph was drawn independently) and as
    many uniformly random pairs (label 0).  Both arms are scored on it with the same function."""
    from graphvite_b200 import datasets
    u, v = datasets.named_edges(name, seed=20260923, num_edge=count)
    rng = np.random.default_rng(7)
    num_vertex = datasets.SHAPES[name][0]
    a, b = rng.integers(0, num_vertex, count), rng.integers(0, num_vertex, count)
    heads = np.concatenate([u, a])
    tails = np.concatenate([v, b])
    labels = np.concatenate([np.ones(count, dtype=np.int64), np.zeros(count, dtype=np.int64)])
    return heads, tails, labels


def quality(vertex, context, name2id, graph_name):
    """Embedding norms and link-prediction AUC (score = <vertex[h], context[t]>, the LINE link predictor,
    python/graphvite/application/network.py:45-75) of one trained model."""
    from graphvite_b200.application import link_prediction_auc
    heads, tails, labels = heldout_pairs(graph_name)
    h = np.fromiter((name2id[str(x)] for x in heads), dtype=np.int64, count=len(heads))
    t = np.fromiter((name2id[str(x)] for x in tails), dtype=np.int64, count=len(tails))
    scores = np.einsum("ij,ij->i", vertex[h], context[t])
    return {"vertex_norm": float(np.linalg.norm(vertex)), "context_norm": float(np.linalg.norm(context)),
            "auc": float(link_prediction_auc(scores, labels))}


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    QUERY = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.rows, self.process = [], None
        try:
            self.process = subprocess.Popen(
                ["nvidia-smi", "-i", str(device), "--query-gpu=" + self.QUERY, "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.process = None

    def _read(self):
        for line in self.process.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.process:
            return None
        self.process.terminate()
        self.thread.join(timeout=2)
        clocks = [int(r[0]) for r in self.rows if len(r) == 6 and r[0].isdigit()]
        if not clocks:
            return None
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) == 6 for i in range(4) if r[2 + i] == "Active"})
        maxima = [int(r[1]) for r in self.rows if len(r) == 6 and r[1].isdigit()]
        return {"sm_mhz": int(np.median(clocks)), "sm_max_mhz": max(maxima) if maxima else None, "reasons": reasons,
                "samples": len(clocks)}


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return float(json.load(open(path))["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


def workload_text(cfg, num_vertex, num_edge):
    if cfg["solver"] == "kg":
        return ("%s d=%d on %s-shaped knowledge graph (%d entities, %d triplets), Adam lr=%g, k=%d, B=%d, "
                "episode_size=%d" % (cfg["model"], cfg["dim"], cfg["graph"], num_vertex, num_edge, cfg["lr"],
                                     cfg["num_negative"], cfg["batch_size"], cfg["episode_size"]))
    return ("%s d=%d on %s-shaped power-law graph (|V|=%d, %d edge lines), SGD lr=%g wd=%g, k=%d, B=%d, "
            "episode_size=%d, augmentation_step=%d, walk length %d%s" %
            (cfg["model"], cfg["dim"], cfg["graph"], num_vertex, num_edge, cfg["lr"], cfg["weight_decay"],
             cfg["num_negative"], cfg["batch_size"], cfg["episode_size"], cfg["augmentation_step"],
             cfg["random_walk_length"], ", p=%g q=%g" % (cfg["p"], cfg["q"]) if cfg["model"] == "node2vec" else ""))


def metric_name(cfg):
    if cfg["solver"] == "kg":
        return "positive triplets/sec on FB15k-237 RotatE d=%d" % cfg["dim"]
    names = {"youtube": "Youtube", "youtube_capped": "Youtube (degree-capped)", "friendster_lite": "Friendster/16"}
    return "edges/sec on %s %s d=%d" % (names.get(cfg["graph"], cfg["graph"]), cfg["model"], cfg["dim"])


def epochs_for(steps, world, num_partition, episode_size, batch_size, num_edge):
    """num_epoch that makes train() run about `steps` sub-episodes per GPU in whole episodes (both arms use this)"""
    per_episode = num_partition * num_partition * episode_size * batch_size
    episodes = max(1, int(round(steps * world * episode_size * batch_size / per_episode)))
    return max(1, int(np.ceil(episodes * per_episode / num_edge)) - 1), episodes * per_episode


def reference_note_path(workload, gpus):
    return "/tmp/gv_b200_reference_%s_n%d.json" % (workload, gpus)


DUMP_BYTES = 64 * 10**6  # --dump-outputs writes at most this much in all


def dump_outputs(directory, arrays):
    """Writes `arrays` (name -> 2-D array of vertex / entity / relation ids) as DIR/<name>.npy in float64, which holds
    every id exactly.  Arrays that together exceed DUMP_BYTES are cut down to a fixed, seeded sample of rows (sorted,
    drawn from the row count alone), so that two builds of the project run with the same arguments can be compared
    output for output."""
    os.makedirs(directory, exist_ok=True)
    total = sum(8 * a.size for a in arrays.values())
    budget = DUMP_BYTES - 4096 * len(arrays)  # room for the .npy headers
    for name, matrix in arrays.items():
        rows = matrix.shape[0]
        keep = rows if total <= budget else max(1, int(rows * budget // total))
        if keep < rows:
            matrix = matrix[np.sort(np.random.default_rng(0).choice(rows, keep, replace=False))]
        np.save(os.path.join(directory, name + ".npy"), np.ascontiguousarray(matrix, dtype=np.float64))


def sample_pools(pool_function, handle, num_partition, pool_id, width):
    """The two sample pools after the timed steps, every (head, tail) block in order: the one the last step trained on
    and the one the samplers filled during it.  Training itself is Hogwild -- concurrent updates of a row race, as in
    the reference -- so the embeddings differ from run to run by the updates lost to races; the pools are what the
    timed path computes deterministically from its inputs."""
    from graphvite_b200 import _lib
    out = {}
    for name, pool in (("trained_pool", pool_id), ("next_pool", pool_id ^ 1)):
        blocks = []
        for head in range(num_partition):
            for tail in range(num_partition):
                count = pool_function(handle, pool, head, tail, None)  # 0: a tail partition another rank holds
                if count < 0:
                    raise _lib.GVError(_lib.last_error())
                if count == 0:
                    continue
                block = np.zeros((count, width), dtype=np.uint32)
                if pool_function(handle, pool, head, tail, block.ctypes.data) < 0:
                    raise _lib.GVError(_lib.last_error())
                blocks.append(block)
        out[name] = np.concatenate(blocks)
    return out


# --------------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------------
def load_graph(gv, cfg):
    from graphvite_b200 import datasets
    graph = gv.graph.Graph()
    if cfg["graph"] in datasets.BINARY_GRAPHS:  # no text file: integer edge arrays straight into the loader
        u, v = datasets.named_edges(cfg["graph"])
        graph.load_arrays(u, v, as_undirected=True)
    else:
        graph.load(graph_file(cfg["graph"]), as_undirected=True)
    return graph


def make_solver(cfg, graph, rank, world, local_rank, num_partition=0):
    import graphvite_b200 as gv
    solver = gv.solver.GraphSolver(cfg["dim"], device_ids=[local_rank], rank=rank, world_size=world)
    solver.build(graph, gv.optimizer.SGD(cfg["lr"], cfg["weight_decay"]), num_partition=num_partition,
                 num_negative=cfg["num_negative"], batch_size=cfg["batch_size"], episode_size=cfg["episode_size"])
    return solver


def train_kwargs(cfg, num_epoch):
    return dict(model=cfg["model"], num_epoch=num_epoch, augmentation_step=cfg["augmentation_step"],
                random_walk_length=cfg["random_walk_length"], random_walk_batch_size=cfg["random_walk_batch_size"],
                p=cfg["p"], q=cfg["q"], negative_weight=cfg["negative_weight"])


def traffic_from_capture(kernel, num_partition, per_edge):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture -- only when the
    capture is of THIS kernel at THIS partition count (profiles/r02_train_kernel.json lists its captures)."""
    path = os.path.join(ROOT, "profiles", "r02_train_kernel.json")
    if not os.path.exists(path):
        return None, "no ncu capture committed for round 2"
    for capture in json.load(open(path)).get("captures", []):
        if capture["kernel"] == kernel and capture["num_partition"] == num_partition:
            note = ("dram__bytes_read+write.sum per launch of %d edges (%.0f B/edge vs %d algorithmic), git %s, %s" %
                    (capture["edges_per_launch"], capture["dram_bytes_per_launch"] / capture["edges_per_launch"],
                     per_edge, capture.get("git", "?"), capture.get("source", "")))
            return capture["dram_bytes_per_launch"], note
    return None, "no ncu capture of %s at num_partition=%d" % (kernel, num_partition)


def parity_cases(world):
    """(name, solver kind, model, partitions): LINE at P = N always; from there on what fits the deadline -- the
    2N-partition case, node2vec with tables sharded over the ranks, the knowledge-graph solver (P = 2N)"""
    cases = [("line_P%d" % world, "graph", "LINE", world)]
    if 2 * world <= 16:
        cases.append(("rotate_adam_P%d" % (2 * world), "kg", None, 2 * world))
    cases.append(("node2vec_P%d" % world, "graph", "node2vec", world))
    if 2 * world <= 8:
        cases.append(("line_P%d" % (2 * world), "graph", "LINE", 2 * world))
    return cases


def multi_rank_parity(rank, world, local_rank, record):
    """N > 1 only: toy inputs through the N-rank solver against the oracle's N-worker emulation (tests/
    multi_rank_worker.py -- both sample pools after every episode bit-exact, embeddings rtol 1e-3): the node-embedding
    solver with LINE (block rotation over NCCL, samplers delivering into peer pools over NVLink), node2vec (per-edge
    tables sharded over the ranks) and the knowledge-graph solver (relation all-reduce).  The oracle is the checker
    here, never the thing measured.  `record(name, ok)` is called after every case with the min over ranks."""
    import torch
    import torch.distributed as dist
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import multi_rank_worker as worker
    for name, kind, model, partitions in parity_cases(world):
        ok = True
        try:
            if kind == "graph":
                os.environ["GV_TEST_MODEL"] = model
                worker.run_graph(rank, world, local_rank, partitions)
            else:
                os.environ["GV_TEST_OPTIMIZER"] = "Adam"
                worker.run_kg(rank, world, local_rank, partitions)
        except BaseException as error:  # an assertion of the worker = a parity failure; report, keep going
            ok = False
            sys.stderr.write("parity self-check %s failed on rank %d: %s\n" % (name, rank, str(error)[:2000]))
        agreed = torch.tensor([1.0 if ok else 0.0], device="cuda", dtype=torch.float64)
        dist.all_reduce(agreed, op=dist.ReduceOp.MIN)
        record(name, bool(agreed.item() > 0.5))
        if not bool(agreed.item() > 0.5):
            return  # a rank that failed mid-run has left the solvers' collectives out of step: stop here


def run_ours(args, cfg):
    import torch
    import torch.distributed as dist
    from graphvite_b200 import _lib

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    assert world == args.gpus, "--gpus must equal the number of launched ranks (torchrun --nproc-per-node)"
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(value):
        if world == 1:
            return value
        t = torch.tensor([value], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    origin = time.time()

    def progress(what):  # stderr only: if a multi-GPU run stalls, the log says in which phase
        if rank == 0 or world > 1 and os.environ.get("GV_BENCH_VERBOSE"):
            sys.stderr.write("[bench %7.2f s] rank %d: %s\n" % (time.time() - origin, rank, what))
            sys.stderr.flush()

    import graphvite_b200 as gv
    from graphvite_b200 import datasets
    if rank == 0 and cfg["graph"] not in datasets.BINARY_GRAPHS:
        graph_file(cfg["graph"])
    barrier()
    load_start = time.time()
    graph = load_graph(gv, cfg)
    load_seconds = time.time() - load_start
    progress("graph loaded, building the solver")
    solver = make_solver(cfg, graph, rank, world, local_rank, args.partitions)
    progress("solver built (%d partitions)" % solver.num_partition)
    lib, handle = _lib.lib, solver._handle
    edges_per_step = cfg["episode_size"] * cfg["batch_size"]  # per GPU
    kw = train_kwargs(cfg, 4000)  # config/graph/line_youtube.yaml; far more epochs than we will run
    _lib.check(lib.gv_solver_train_begin(handle, kw["model"].encode(), kw["num_epoch"], 0, kw["augmentation_step"],
                                         kw["random_walk_length"], kw["random_walk_batch_size"], 0, kw["p"], kw["q"], 1,
                                         0.75, float(kw["negative_weight"]), 1000))
    progress("train_begin done (tables, first pool, embeddings resident)")
    for _ in range(args.warmup):
        assert lib.gv_solver_train_step(handle) == 1, _lib.last_error()
    barrier()
    progress("%d warm-up steps done" % args.warmup)
    before = solver.stats
    sampler = ClockSampler(local_rank) if rank == 0 else None
    lib.gv_solver_device_timer(handle, 0)
    for _ in range(args.steps):
        assert lib.gv_solver_train_step(handle) == 1, _lib.last_error()
    seconds = lib.gv_solver_device_timer(handle, 1)
    barrier()
    progress("%d timed steps done" % args.steps)
    clocks = sampler.stop() if sampler else None
    after = solver.stats
    seconds = max_over_ranks(seconds)
    _lib.check(lib.gv_solver_train_end(handle))
    if args.dump_outputs and rank == 0:  # pairs {tail, head}
        dump_outputs(args.dump_outputs, sample_pools(lib.gv_solver_pool, handle, solver.num_partition,
                                                     solver.pool_id, 2))
    value = args.steps * edges_per_step * world / seconds

    # roofline of the dominant kernel (the train kernel): algorithmic bytes / CUDA-event time of its launches
    # (one event pair around the launches of a step on the solver's work stream: launch gaps count against us)
    kernel_seconds = max_over_ranks(after["kernel_seconds"] - before["kernel_seconds"])
    positives = after["positives"] - before["positives"]
    per_edge = bytes_per_edge(cfg["dim"], cfg["num_negative"])
    achieved = positives * per_edge / kernel_seconds / 1e9
    peak, peak_kind = measured_peak()
    launches = int(after["launches"] - before["launches"])
    flags = int(lib.gv_cuda_get_tunable(b"kernel_flags"))
    chunk_batches = solver.chunk_batches
    kernel = ("gv::device::train_sgd_kernel<%d, %d>" if flags & 64 else "gv::device::train_sample_per_warp_kernel<%d>") % \
        ((cfg["dim"], cfg["num_negative"]) if flags & 64 else (cfg["dim"],))
    traffic, traffic_note = traffic_from_capture(kernel, solver.num_partition, per_edge)
    num_partition = solver.num_partition

    if args.no_e2e:
        if rank == 0:
            print(json.dumps({"value": value, "ms_per_step": seconds / args.steps * 1e3, "roofline_gbs": achieved,
                              "frac": achieved / peak, "gpu_launches": launches, "kernel": kernel,
                              "num_partition": num_partition, "note": "profiling run, no e2e"}), flush=True)
        solver.close()
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return
    # end to end through the public API: host graph + host embeddings in, host embeddings out
    solver.close()  # collective teardown (IPC importers close before exporters free)
    del solver
    progress("steady-state solver closed, building the end-to-end solver")
    build_start = time.time()
    solver2 = make_solver(cfg, graph, rank, world, local_rank)
    build_seconds = time.time() - build_start
    num_epoch, _ = epochs_for(args.steps, world, solver2.num_partition, cfg["episode_size"], cfg["batch_size"],
                              graph.num_edge)
    barrier()
    start = time.time()
    solver2.train(**train_kwargs(cfg, num_epoch))
    barrier()
    e2e_seconds = max_over_ranks(time.time() - start)
    progress("end-to-end train() done")
    e2e_edges = solver2.batch_id * cfg["batch_size"]
    e2e_steps = max(1, e2e_edges // (edges_per_step * world))
    matrix_bytes = graph.num_vertex * cfg["dim"] * 4
    directed = 2 * graph.num_edge
    # what train() copies to the device: the vertex matrix (the zero context matrix is cleared there), CSR offsets and
    # targets, the negative table; an unweighted graph's source column, edge alias table and weights are built on the
    # device (gv_solver.cpp::prepare_sampling)
    h2d = matrix_bytes + directed * 4 + graph.num_vertex * (8 + 8)
    d2h = 2 * matrix_bytes
    e2e_stats = solver2.stats
    model_quality = None
    if rank == 0 and cfg["graph"] in datasets.SHAPES:
        model_quality = quality(solver2.vertex_embeddings, solver2.context_embeddings, graph.name2id, cfg["graph"])
        model_quality["num_epoch"] = num_epoch

    result = {
        "metric": metric_name(cfg), "value": value, "unit": "edges/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": seconds / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "impl": "graphvite_b200",
        "config": {"workload": workload_text(cfg, graph.num_vertex, graph.num_edge), "num_partition": num_partition},
        "parallelism": "2-D block partition, %d GPU(s), one process per GPU" % world,
        "l2": "working set (2 x %.0f MB embedding blocks + %.0f MB pool block per GPU) >> 126 MB L2, no flush needed" %
              (matrix_bytes / num_partition / 1e6, edges_per_step * 8 / 1e6),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_note": traffic_note, "peak_source": peak_kind,
                     "bytes_per_edge": per_edge, "kernel": kernel,
                     "algorithmic_bytes_per_launch": per_edge * chunk_batches * cfg["batch_size"],
                     "batches_per_launch": chunk_batches,
                     "kernel_edges_per_s": positives / kernel_seconds,
                     "timing": "CUDA events on the work stream around each step's train launches (gaps included), "
                               "max over ranks"},
        "e2e": {"value": e2e_edges / e2e_seconds, "unit": "edges/s", "h2d_bytes_per_step": h2d / e2e_steps,
                "d2h_bytes_per_step": d2h / e2e_steps, "seconds": e2e_seconds, "edges": e2e_edges,
                "num_epoch": num_epoch, "sampler_seconds": e2e_stats["sample_seconds"],
                "train_seconds": e2e_stats["train_seconds"],
                # outside the timed region in BOTH arms (the reference's "training time" is train() too,
                # application.py:99-105): what a user waits for before train() starts
                "setup_seconds": {"graph_load": load_seconds, "solver_build": build_seconds}},
        "gpu_launches": launches,
        "clocks": clocks,
        "model_quality": model_quality,
    }
    # float parity on the driver's record: the reference arm (run just before on the same box) leaves its model's
    # norms / AUC for the same num_epoch; rel_diff = (ours - reference) / reference
    note = reference_note_path(args.workload, world)
    if rank == 0 and model_quality and os.path.exists(note):
        try:
            theirs = json.load(open(note))
            if theirs.get("num_epoch") == num_epoch:
                result["vs_reference_quality"] = {
                    "reference": theirs,
                    "vertex_norm_rel": model_quality["vertex_norm"] / theirs["vertex_norm"] - 1,
                    "context_norm_rel": model_quality["context_norm"] / theirs["context_norm"] - 1,
                    "auc_diff": model_quality["auc"] - theirs["auc"],
                    "north_star": "norms within 1e-3 relative, AUC within 0.003"}
        except (OSError, ValueError, KeyError):
            pass
    solver2.close()
    del solver2
    if world > 1 and not args.no_parity:
        progress("multi-rank parity self-check against the oracle")
        # Runs on a helper thread with a deadline: a rank that fails a comparison leaves the collective calls of the
        # others unanswered, and the benchmark line must not be lost to that.  After a timeout the process prints its
        # line (parity_ok false) and leaves without the collective teardown.
        outcome = {}
        started = time.time()

        def check():
            multi_rank_parity(rank, world, 0 if os.environ.get("GV_EMULATE") == "1" else local_rank,
                              lambda name, ok: outcome.__setitem__(name, {"ok": ok, "after_s": round(time.time() - started, 1)}))

        worker = threading.Thread(target=check, daemon=True)
        worker.start()
        worker.join(timeout=args.parity_timeout)
        timed_out = worker.is_alive()
        planned = [c[0] for c in parity_cases(world)]
        result["parity"] = {name: outcome[name]["ok"] for name in planned if name in outcome}
        result["parity_seconds"] = {name: outcome[name]["after_s"] for name in planned if name in outcome}
        result["parity_not_run"] = [name for name in planned if name not in outcome]
        result["parity_ok"] = bool(result["parity"]) and all(result["parity"].values())
        result["parity_note"] = ("toy inputs, %d ranks vs the oracle's %d-worker emulation: pools bit-exact after "
                                 "every episode, embeddings rtol 1e-3 (tests/multi_rank_worker.py); min over ranks; "
                                 "parity_ok = every case that finished inside the %d s deadline passed%s" %
                                 (world, world, args.parity_timeout,
                                  " (deadline reached: %s not run)" % ", ".join(result["parity_not_run"])
                                  if timed_out else ""))
        if timed_out:
            if rank == 0:
                print(json.dumps(result), flush=True)
            sys.stderr.flush()
            os._exit(0)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        child = run_reference_child(args, max(2, min(args.steps, 10)))
        if "unavailable" in child:
            result["cpu_baseline"] = {"value": None, "unit": "edges/s", "cores": os.cpu_count(), "kind": "reference",
                                      "sample": "unavailable: %s" % child["unavailable"]}
        else:
            result["cpu_baseline"] = child["cpu_baseline"]
    if rank == 0:
        print(json.dumps(result), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# --------------------------------------------------------------------------------------------------
# knowledge-graph workload (config #4): KnowledgeGraphSolver, RotatE d=2048, Adam
# --------------------------------------------------------------------------------------------------
def kg_bytes_per_positive(dim, k, num_moment, adversarial=True):
    """DESIGN.md section 4: negative rows once for the normaliser, once read-modify-write with their moments; the
    positive head / tail / relation rows (+ moments) once each way."""
    row = dim * 4
    relation_row = row // 2  # RotatE: phases
    states = 1 + num_moment
    return ((k * row if adversarial else 0) + k * states * 2 * row + states * 2 * (2 * row + relation_row) +
            12 + 8 * k + 4)


def run_ours_kg(args, cfg):
    import torch
    import torch.distributed as dist
    import graphvite_b200 as gv
    from graphvite_b200 import _lib, datasets

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    assert world == args.gpus
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    path = "/tmp/gv_b200_fb15k237.txt"
    if rank == 0 and not os.path.exists(path):
        datasets.synthetic_knowledge_graph_file("fb15k-237", path + ".tmp")
        os.replace(path + ".tmp", path)
    if world > 1:
        dist.barrier()
    graph = gv.graph.KnowledgeGraph()
    graph.load(path)
    solver = gv.solver.KnowledgeGraphSolver(cfg["dim"], device_ids=[local_rank], rank=rank, world_size=world)
    solver.build(graph, gv.optimizer.Adam(cfg["lr"], cfg["weight_decay"]), num_partition=args.partitions,
                 num_negative=cfg["num_negative"], batch_size=cfg["batch_size"], episode_size=cfg["episode_size"])
    lib, handle = _lib.lib, solver._handle
    _lib.check(lib.gv_kg_solver_train_begin(handle, cfg["model"].encode(), 1000, 0, 1.0, cfg["margin"],
                                            cfg["l3_regularization"], cfg["sample_batch_size"], 1,
                                            cfg["adversarial_temperature"], 100))
    for _ in range(args.warmup):
        assert lib.gv_kg_solver_train_episode(handle) == 1, _lib.last_error()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    before = solver.stats
    sampler = ClockSampler(local_rank) if rank == 0 else None
    start = time.time()
    for _ in range(args.steps):
        assert lib.gv_kg_solver_train_episode(handle) == 1, _lib.last_error()
    torch.cuda.synchronize()
    seconds = time.time() - start
    after = solver.stats
    clocks = sampler.stop() if sampler else None
    positives = after["positives"] - before["positives"]
    kernel_seconds = after["kernel_seconds"] - before["kernel_seconds"]
    if world > 1:
        t = torch.tensor([seconds, kernel_seconds], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        seconds, kernel_seconds = float(t[0].item()), float(t[1].item())
    _lib.check(lib.gv_kg_solver_train_end(handle))
    if args.dump_outputs and rank == 0:  # triplets {relation, tail, head}
        dump_outputs(args.dump_outputs, sample_pools(lib.gv_kg_solver_pool, handle, solver.num_partition,
                                                     solver.pool_id, 3))
    per_positive = kg_bytes_per_positive(cfg["dim"], cfg["num_negative"], 2)
    peak, peak_kind = measured_peak()
    achieved = positives * per_positive / max(kernel_seconds, 1e-12) / 1e9
    result = {
        "metric": metric_name(cfg), "value": positives * world / seconds, "unit": "triplets/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": seconds / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "impl": "graphvite_b200",
        "config": {"workload": workload_text(cfg, graph.num_vertex, graph.num_edge),
                   "num_partition": solver.num_partition},
        "step": "one episode = every rank's blocks of the tied-weight schedule, %d positives per rank" %
                (positives // max(1, args.steps)),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": None, "peak_source": peak_kind, "bytes_per_positive": per_positive,
                     "kernel": "gv::device::kg_train_kernel",
                     "note": "algorithmic bytes; entity rows + 2 Adam moments of one rank's two blocks are %.0f MB, so "
                             "part of the negative-row traffic is served by the 126 MB L2 (frac > 1 is possible)" %
                             (2.0 * graph.num_vertex / max(1, solver.num_partition) * cfg["dim"] * 4 * 3 / 1e6)},
        "gpu_launches": int(after["launches"] - before["launches"]),
        "clocks": clocks,
        "entity_norm": float(np.linalg.norm(solver.entity_embeddings)),
    }
    if rank == 0:
        print(json.dumps(result), flush=True)
    solver.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# --------------------------------------------------------------------------------------------------
# reference arm: the UNMODIFIED reference (oracle/_ref/libgraphvite.so) through its own pybind API
# --------------------------------------------------------------------------------------------------
def load_reference():
    path = os.path.join(ROOT, "oracle", "_ref", "libgraphvite.so")
    if not os.path.exists(path):
        raise RuntimeError("oracle/_ref/libgraphvite.so is not built (make -C oracle ref)")
    spec = importlib.util.spec_from_file_location("libgraphvite", path)
    module = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(module)
    module.init_logging(module.ERROR, "", False)
    return module


def reference_train(cfg, path, num_gpu, steps):
    """Times GraphSolver.train() of the reference (its own definition of training time,
    python/graphvite/application/application.py:99-105) for about `steps` sub-episodes per GPU."""
    ref = load_reference()
    graph = ref.graph.Graph_j()
    graph.load(path, True, False)
    solver = getattr(ref.solver, "GraphSolver_%d_f_j" % cfg["dim"])(list(range(num_gpu)), 0, 0)
    solver.build(graph, ref.optimizer.SGD(cfg["lr"], cfg["weight_decay"]), 0, cfg["num_negative"],
                 cfg["batch_size"], cfg["episode_size"])
    P, E, B = solver.num_partition, solver.episode_size, solver.batch_size
    num_epoch, _ = epochs_for(steps, num_gpu, P, E, B, graph.num_edge)
    kwargs = dict(model=cfg["model"], num_epoch=num_epoch, resume=False,
                  augmentation_step=cfg["augmentation_step"], random_walk_length=cfg["random_walk_length"],
                  random_walk_batch_size=cfg["random_walk_batch_size"], p=cfg["p"], q=cfg["q"],
                  negative_weight=cfg["negative_weight"], log_frequency=1 << 30)
    start = time.time()
    solver.train(**kwargs)
    seconds = time.time() - start
    num_batch = num_epoch * graph.num_edge // B
    per_episode_batches = P * P * E
    trained = -(-num_batch // per_episode_batches) * per_episode_batches * B
    return {"edges": trained, "seconds": seconds, "num_sampler": solver.num_sampler, "num_worker": solver.num_worker,
            "num_partition": P, "num_epoch": num_epoch, "graph": graph, "solver": solver,
            "steps": trained // (E * B * num_gpu)}


def reference_child(args, cfg):
    """Runs in its own process (the reference abort()s on every error, util/debug.h:30-38): one warm-up run, one
    timed run, one JSON line."""
    path = graph_file(cfg["graph"])
    warm = reference_train(cfg, path, args.gpus, 1)  # CUDA context, page-in, first allocations
    del warm
    r = reference_train(cfg, path, args.gpus, args.steps)
    value = r["edges"] / r["seconds"]
    graph, solver = r["graph"], r["solver"]
    cores = r["num_sampler"] + r["num_worker"]
    sample = ("warmed GraphSolver.train() wall time for %d edges (%d sub-episodes per GPU, num_epoch %d), %d CPU "
              "sampler threads + %d worker thread(s), host has %d logical cores" %
              (r["edges"], r["steps"], r["num_epoch"], r["num_sampler"], r["num_worker"], os.cpu_count()))
    from graphvite_b200 import datasets
    model_quality = None
    if cfg["graph"] in datasets.SHAPES:
        model_quality = quality(np.array(solver.vertex_embeddings), np.array(solver.context_embeddings),
                                graph.name2id, cfg["graph"])
        model_quality["num_epoch"] = r["num_epoch"]
        try:
            json.dump(model_quality, open(reference_note_path(args.workload, args.gpus), "w"))
        except OSError:
            pass
    print(json.dumps({
        "metric": metric_name(cfg), "value": value, "unit": "edges/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["seconds"] / max(1, r["steps"]) * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "impl": "reference",
        "config": {"workload": workload_text(cfg, graph.num_vertex, graph.num_edge),
                   "num_partition": r["num_partition"]},
        "steps_run": int(r["steps"]),
        "warmup_note": "one untimed GraphSolver.train() of one episode in the same process (the reference has no "
                       "step API; --warmup is echoed for the driver's bookkeeping)",
        "cpu_baseline": {"value": value, "unit": "edges/s", "cores": cores, "kind": "reference", "sample": sample},
        "e2e": {"value": value, "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "model_quality": model_quality,
    }), flush=True)


def run_reference_child(args, steps):
    """Launch `bench.py --impl reference-child` and parse its line; a crash of the reference becomes
    {"unavailable": <its last words>} instead of taking this process down."""
    command = [sys.executable, os.path.abspath(__file__), "--impl", "reference-child", "--gpus", str(args.gpus),
               "--steps", str(steps), "--warmup", str(args.warmup), "--workload", args.workload, "--watchdog", "0"]
    env = dict(os.environ)
    for name in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT"):  # one process drives all GPUs
        env.pop(name, None)
    try:
        done = subprocess.run(command, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env,
                              timeout=max(300, args.watchdog - 120 if args.watchdog else 1200))
    except subprocess.TimeoutExpired:
        return {"unavailable": "the reference run did not finish in time"}
    log_dir = os.path.join(ROOT, "gpurun_out")
    if os.path.isdir(log_dir):
        with open(os.path.join(log_dir, "reference_stderr_n%d.log" % args.gpus), "w") as fout:
            fout.write(done.stderr[-20000:])
    for line in reversed(done.stdout.strip().splitlines()):
        if line.startswith("{"):
            try:
                return json.loads(line)
            except ValueError:
                continue
    words = [x for x in done.stderr.strip().splitlines() if x.strip()]
    return {"unavailable": "reference process ended with code %d: %s" %
                           (done.returncode, (words[-1] if words else "no output")[:300])}


def run_reference(args, cfg):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return  # the reference is one process driving all GPUs from threads
    if cfg["solver"] != "graph":
        print(json.dumps({"impl": "reference", "unavailable": "reference arm is wired for the node-embedding "
                          "workloads only"}), flush=True)
        return
    child = run_reference_child(args, args.steps)
    if "unavailable" in child:
        print(json.dumps({"impl": "reference", "unavailable": child["unavailable"]}), flush=True)
    else:
        print(json.dumps(child), flush=True)


def start_watchdog(seconds):
    """A hung collective must not hang the box: give up loudly after `seconds`."""
    def expire():
        sys.stderr.write("bench.py: no result after %d s, aborting\n" % seconds)
        sys.stderr.flush()
        os._exit(3)
    timer = threading.Timer(seconds, expire)
    timer.daemon = True
    timer.start()
    return timer


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument("--gpus", type=int, default=1)
    parser.add_argument("--steps", type=int, default=10)
    parser.add_argument("--warmup", type=int, default=3)
    parser.add_argument("--impl", default="graphvite_b200", choices=["graphvite_b200", "reference", "reference-child"])
    parser.add_argument("--workload", default="youtube", choices=sorted(WORKLOADS))
    parser.add_argument("--no-cpu-baseline", action="store_true")
    parser.add_argument("--no-e2e", action="store_true", help="skip the end-to-end leg (profiling runs only)")
    parser.add_argument("--no-parity", action="store_true", help="skip the multi-rank parity self-check (N > 1)")
    parser.add_argument("--parity-timeout", type=int, default=300, help="deadline of the parity self-check in seconds")
    parser.add_argument("--partitions", type=int, default=0, help="num_partition (0 = auto; diagnosis only)")
    parser.add_argument("--watchdog", type=int, default=1500, help="abort after this many seconds (0 = never)")
    parser.add_argument("--dump-outputs", default="", metavar="DIR",
                        help="write the sample pools of the last timed step as DIR/<name>.npy (float64 ids, at most "
                             "64 MB in all: a fixed, seeded sample of rows where the pools are larger)")
    args = parser.parse_args()
    if args.watchdog > 0:
        start_watchdog(args.watchdog)
    cfg = WORKLOADS[args.workload]
    if args.impl == "reference-child":
        reference_child(args, cfg)
        return
    if args.impl == "reference":
        run_reference(args, cfg)
        return
    try:
        if cfg["solver"] == "kg":
            run_ours_kg(args, cfg)
        else:
            run_ours(args, cfg)
    except BaseException:
        # leave at once: a rank that unwinds normally would first wait for its sampler thread, which may be waiting
        # for the peers -- torchrun only stops the other ranks once this process is gone
        import traceback
        traceback.print_exc()
        sys.stderr.flush()
        sys.stdout.flush()
        os._exit(1)


if __name__ == "__main__":
    main()
