"""How far can the CUDA emulation of tests/emu be trusted?  Here it executes the UNMODIFIED reference (two-pass
build, `make -C oracle ref_emu`, see oracle/emulate_reference.py) and regenerates golden vectors that were
recorded from the same reference on a real B200 (tests/golden/, oracle/make_golden.py): every integer output --
cuRAND streams, alias tables, partitions, BOTH sample pools and the last negatives of full solver runs -- must be
bit-identical to what the hardware produced, and the train kernels (race-free batches) equal up to the rounding of
libm / FMA contraction.  (Embeddings of the solver runs are not compared: the B200 run is Hogwild, the emulation
processes a batch in order.)  Skipped where the emulated reference is not built (`make -C oracle ref_emu` needs the
reference's sources).

The emulation processes a batch in order, like the oracle, so its solver runs also pin the oracle's training arithmetic
float for float.  That comparison does not need the reference at hand: what the emulated reference trained (both
embedding matrices, and predict) is stored in tests/golden/emu_reference_*.npz
(`python oracle/make_golden.py --emulated --oracle-check tests/golden`)."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
LIBRARY = os.path.join(ROOT, "oracle", "_ref", "libref_harness_emu.so")

# GV_EMU_FULL=1 regenerates all seven solver runs (+1 min)
SOLVER_CASES = ["line_p1", "edge_p2", "node2vec_p1"]
if os.environ.get("GV_EMU_FULL") == "1":
    SOLVER_CASES += ["line_p2_s3", "deepwalk_p1", "line_p3_adam", "node2vec_p2"]

needs_emulated_reference = pytest.mark.skipif(not os.path.exists(LIBRARY),
                                              reason="oracle/_ref/libref_harness_emu.so is not built")
# solver runs of the emulated reference stored for the oracle comparison (oracle/make_golden.py ORACLE_CHECK_CASES)
RECORDED_CASES = ["line_p1", "edge_p2", "node2vec_p1"]


@pytest.fixture(scope="module")
def regenerated(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("golden_emu"))
    script = ("import sys; sys.argv = ['make_golden.py', '--emulated']; sys.path.insert(0, %r)\n"
              "import make_golden as M\n"
              "lib = M.load_harness(); toy = %r\n"
              "M.write_basics(lib, %r, toy)\n"
              "M.write_kernel_cases(lib, %r)\n"
              "M.write_solver_cases(lib, %r, toy, %r)\n" %
              (os.path.join(ROOT, "oracle"), os.path.join(GOLDEN, "toy_graph.txt"), out, out, out, set(SOLVER_CASES)))
    env = dict(os.environ, GV_EMU_BACKTRACE="1")
    result = subprocess.run([sys.executable, "-c", script], cwd=ROOT, env=env, stdout=subprocess.PIPE,
                            stderr=subprocess.STDOUT, text=True, timeout=1500)
    assert result.returncode == 0, result.stdout[-4000:]
    return out


def compare(regenerated, name, float_tolerance=None, skip=()):
    ours, theirs = np.load(os.path.join(regenerated, name)), np.load(os.path.join(GOLDEN, name))
    assert set(ours.files) == set(theirs.files)
    for key in theirs.files:
        if key in skip:
            continue
        a, b = ours[key], theirs[key]
        if b.dtype.kind in "iub" or key.startswith("cfg_"):
            np.testing.assert_array_equal(a, b, err_msg="%s:%s" % (name, key))
        elif float_tolerance is None:
            np.testing.assert_array_equal(a, b, err_msg="%s:%s" % (name, key))  # host arithmetic on both sides
        else:
            np.testing.assert_allclose(a, b, err_msg="%s:%s" % (name, key), **float_tolerance)


@needs_emulated_reference
@pytest.mark.parametrize("name", ["curand.npz", "alias.npz", "graph_u0_n0.npz", "graph_u0_n1.npz", "graph_u1_n0.npz",
                                  "graph_u1_n1.npz"])
def test_host_side_fixtures_regenerate_identically(regenerated, name):
    compare(regenerated, name)


@needs_emulated_reference
@pytest.mark.parametrize("optimizer", ["SGD", "Momentum", "AdaGrad", "RMSprop", "Adam"])
@pytest.mark.parametrize("dim", [32, 128])
def test_train_kernels_match_the_b200_to_rounding(regenerated, dim, optimizer):
    compare(regenerated, "kernel_d%d_%s.npz" % (dim, optimizer), float_tolerance=dict(rtol=2e-5, atol=2e-6))


@needs_emulated_reference
@pytest.mark.parametrize("case", SOLVER_CASES)
def test_solver_runs_reproduce_the_b200s_integer_state(regenerated, case):
    # vertex / context / loss / logits: Hogwild on the B200, in order here; edge_prob is float but host-built
    compare(regenerated, "solver_%s.npz" % case, skip=("vertex", "context", "loss", "logits"))


@needs_emulated_reference
@pytest.mark.parametrize("case", RECORDED_CASES)
def test_stored_solver_runs_are_the_emulated_references(regenerated, case):
    """provenance of tests/golden/emu_reference_solver_*.npz: the emulated reference regenerates them bit for bit"""
    ours, stored = np.load(os.path.join(regenerated, "solver_%s.npz" % case)), \
        np.load(os.path.join(GOLDEN, "emu_reference_solver_%s.npz" % case))
    for key in ("vertex", "context", "logits"):
        np.testing.assert_array_equal(ours[key], stored[key], err_msg=key)


@pytest.mark.parametrize("case", RECORDED_CASES)
def test_oracle_training_arithmetic_equals_the_references_in_order(case):
    """On the B200 the reference's solver runs are Hogwild, so tests/test_oracle_golden.py can pin the oracle's
    integer state only.  The emulation processes a batch in order (one warp per sample, warps one after another) --
    the oracle's order -- so here the oracle's whole training run is compared with the reference's float for float:
    vertex / context embeddings, the last batch's losses and predict."""
    import oracle_lib as O
    g = np.load(os.path.join(GOLDEN, "solver_%s.npz" % case))  # configuration and predict pairs of the run
    recorded = np.load(os.path.join(GOLDEN, "emu_reference_solver_%s.npz" % case))
    cfg = {key[4:]: g[key].item() for key in g.files if key.startswith("cfg_")}
    graph = O.OracleGraph(os.path.join(GOLDEN, "toy_graph.txt"))
    solver = O.OracleSolver(graph, cfg["dim"], 1, cfg["S"])
    solver.build(cfg["optimizer"], cfg["P"], cfg["k"], cfg["B"], cfg["E"])
    solver.train(model=cfg["model"], num_epoch=cfg["epochs"], augmentation_step=cfg["aug"],
                 random_walk_length=cfg["L"], random_walk_batch_size=cfg["wb"], p=cfg.get("p", 1.0),
                 q=cfg.get("q", 1.0))
    tolerance = dict(rtol=1e-4, atol=1e-7)
    np.testing.assert_allclose(solver.embeddings(0), recorded["vertex"], **tolerance)
    np.testing.assert_allclose(solver.embeddings(1), recorded["context"], **tolerance)
    np.testing.assert_allclose(solver.predict(g["pairs"]), recorded["logits"], rtol=1e-4, atol=1e-6)
