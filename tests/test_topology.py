"""MXNET_KVSTORE_USETREE: the engine's restated tree solver (csrc/topology.cc) against the reference's own
(src/kvstore/gpu_topology.h) -- no GPU needed, the solver is host code and the library loads without a device.

Three pins, strongest first:
* tests/golden/tree_topology.npz: trees the reference's compiled header produced for 136 link matrices (one
  switch, the NVLink cube mesh, random 2 ... 16 GPUs; Kernighan-Lin and exhaustive search) -- always checked;
* oracle/_ref/libkvref_topo.so, the reference header compiled in place: random matrices -- a fixed draw against the
  trees it returned, stored in tests/golden/tree_draw.npz; fresh ones in soak runs, when the library is there;
* the known answers of the reference's unit test, tests/cpp/kvstore/gpu_topology_test.cc, function by function.
Then the derived add schedules: the kernel's own evaluator (csrc/tree_math.h compiled for the host) against the
oracle's level-by-level restatement of CommDeviceTree::ReduceInner on every golden tree."""
import os

import numpy as np
import pytest

import mxnet_b200 as mx
from oracle import oracle as O

T = mx.topology
HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def golden():
    return np.load(os.path.join(HERE, "golden", "tree_topology.npz"))


def test_trees_match_the_reference_solver_golden(golden):
    n_cases = int(golden["n_cases"])
    assert n_cases >= 130
    checked = failed = 0
    for i in range(n_cases):
        W, alpha, bt = golden["case_%d_W" % i], float(golden["case_%d_alpha" % i]), bool(golden["case_%d_backtrack" % i])
        if "case_%d_fails" % i in golden.files:
            with pytest.raises(mx.MXNetError, match="no balanced binary tree"):
                T.compute_trees(W, alpha, bt)
            failed += 1
            continue
        topo, scan, depth = T.compute_trees(W, alpha, bt)
        assert np.array_equal(topo, golden["case_%d_topo" % i]), (i, W.shape[0], bt)
        assert np.array_equal(scan, golden["case_%d_scan" % i]), i
        assert depth == T.depth(W.shape[0]) and topo.shape[1] == (2 << depth) - 1 and scan.shape[1] == depth + 2
        checked += 1
    assert checked >= 120 and failed >= 1


def test_kernighan_lin_pass_matches_the_reference_golden(golden):
    for i in range(int(golden["n_kl"])):
        W = golden["kl_%d_W" % i]
        stop, P, npart, pairs = T.bisect(W, np.zeros(W.shape[0], np.int32), 1, seed=int(golden["kl_%d_seed" % i]))
        assert stop == bool(golden["kl_%d_stop" % i])
        assert np.array_equal(P, golden["kl_%d_P" % i]) and npart == int(golden["kl_%d_npart" % i])
        assert [int(v) for p in pairs for v in p] == golden["kl_%d_pairs" % i].tolist()


def link_matrix_draw(rng):
    """(W, alpha, backtrack) for random link matrices of 2 ... 16 GPUs, some with missing links."""
    for n in (2, 3, 4, 5, 6, 7, 8, 9, 11, 13, 16):
        for rep in range(3):
            u = rng.uniform(0, 1, (n, n))
            W = np.where(u < 0.33, 1.0, np.where(u < 0.66, 2.0, 3.0))
            if rep % 3 == 2:
                W = np.where(rng.uniform(0, 1, (n, n)) < 0.3, 0.0, W)
            W = np.triu(W, 1)
            W = (W + W.T).astype(np.float32)
            alpha = float(rng.choice([0.7, 0.5, 0.9]))
            for bt in ((False, True) if n <= 5 else (False,)):
                yield W, alpha, bt


def test_trees_match_the_reference_header_compiled_in_place():
    """A fixed draw against tests/golden/tree_draw.npz (what oracle/_ref/libkvref_topo.so returned for it,
    make_golden.py::tree_draw); MXKV_FUZZ_SEEDS > 0 (soak runs): fresh matrices against that library itself."""
    fresh = int(os.environ.get("MXKV_FUZZ_SEEDS", "0")) > 0
    if fresh and O.ref_topology_lib() is None:
        pytest.skip("fresh matrices need oracle/_ref/libkvref_topo.so (built by oracle/Makefile from the reference tree)")
    gold = None if fresh else dict(np.load(os.path.join(HERE, "golden", "tree_draw.npz")))
    rng = np.random.default_rng(int.from_bytes(os.urandom(4), "little") if fresh else 20260921)
    at = dict.fromkeys(("W", "topo", "scan"), 0)

    def take(name, count):
        at[name] += count
        return gold[name][at[name] - count:at[name]]

    i = -1
    for i, (W, alpha, bt) in enumerate(link_matrix_draw(rng)):
        n = W.shape[0]
        if fresh:
            want = O.ref_compute_trees(W, alpha, bt)
        else:
            assert np.array_equal(W.ravel(), take("W", n * n)), i
            assert alpha == gold["alpha"][i] and bt == gold["backtrack"][i], i
            tl, sl = int(gold["topo_len"][i]), int(gold["scan_len"][i])
            want = (take("topo", n * tl).reshape(n, tl), take("scan", n * sl).reshape(n, sl)) if tl else None
        if want is None:
            with pytest.raises(mx.MXNetError):
                T.compute_trees(W, alpha, bt)
            continue
        topo, scan, _ = T.compute_trees(W, alpha, bt)
        assert np.array_equal(topo, want[0]) and np.array_equal(scan, want[1]), (i, bt, W.tolist())
    assert fresh or (i + 1 == gold["alpha"].size and at["W"] == gold["W"].size and at["topo"] == gold["topo"].size)


# ---- tests/cpp/kvstore/gpu_topology_test.cc, case by case -------------------------------------------------------
W7 = np.array([[0, 2, 2, 3, 3, 0, 0], [2, 0, 3, 2, 0, 3, 0], [2, 3, 0, 3, 0, 0, 2], [3, 2, 3, 0, 0, 0, 0],
               [3, 0, 0, 0, 0, 2, 2], [0, 3, 0, 0, 2, 0, 3], [0, 0, 2, 0, 2, 3, 0]], np.float32)
W8 = np.array([[0, 2, 2, 3, 3, 1, 1, 1], [2, 0, 3, 2, 1, 3, 1, 1], [2, 3, 0, 3, 1, 1, 2, 1], [3, 2, 3, 0, 1, 1, 1, 2],
               [3, 1, 1, 1, 0, 2, 2, 3], [1, 3, 1, 1, 2, 0, 3, 2], [1, 1, 2, 1, 2, 3, 0, 3], [1, 1, 1, 2, 3, 2, 3, 0]], np.float32)


def test_reference_unit_test_depth():                                 # TestDepth, :190-198
    for n, d in ((2, 1), (3, 2), (8, 3), (7, 3), (5, 3), (4, 2), (16, 4)):
        assert T.depth(n) == d
        assert T.compute_trees(2.0 * (np.ones((n, n)) - np.eye(n)))[2] == d


def test_reference_unit_test_postprocess():                           # TestPostprocess, :164-188
    for got, want, n, d in (([3, 0, 0, 4, 1, 2, 5, 6], [3, 3, 0, 4, 1, 2, 5, 6], 7, 3),
                            ([2, 0, 0, 4, 1, 3, 5, 1], [2, 2, 0, 4, 1, 3, 5, 5], 6, 3),
                            ([5, 4, 1, 3, 1, 0, 2, 0], [5, 4, 5, 3, 1, 0, 2, 2], 6, 3),
                            ([10, 10, 0, 0, 0, 0, 0, 1, 2, 3, 6, 4, 7, 5, 8, 9],
                             [10, 10, 10, 10, 0, 0, 0, 1, 2, 3, 6, 4, 7, 5, 8, 9], 11, 4)):
        assert T.fold_repeats(got, n, d).tolist() == want


def test_reference_unit_test_tree_weight():                           # TestComputeTreeWeight, :148-162
    assert T.tree_weight(W7, [3, 2, 1, 5, 0, 0, 4, 6], 7, 3, False) == 16
    assert T.tree_weight(W7, [3, 2, 0, 4, 1, 1, 5, 6], 7, 3, False) == 17


def test_reference_unit_test_is_valid():                              # TestIsValid, :200-236
    for state, row, want in (([3, 2, 1, 5, 0, 0, 4, 6], 7, True), ([3, 2, 0, 4, 1, 1, 5, 6], 7, True),
                             ([3, 2, 5, 1, 0, 4, 2, 5], 7, False), ([3, 7, 2, 6, 0, 1, 4, 5], 7, False),
                             ([3, -1, 2, 6, 0, 1, 4, 5], 7, True), ([3, -1, 2, 6, 0, 1, 4, -1], 8, False),
                             ([3, -1, -1, -1, -1, -1, -1, -1], 1, True)):
        assert T.admissible(W7, state, 7, row, 3) is want, state


def test_reference_unit_test_is_connected():                          # TestIsConnected1-3, :515-557
    assert not T.connected([[0, 0, 2, 0], [0, 0, 0, 2], [2, 0, 0, 0], [0, 2, 0, 0]])
    assert not T.connected([[1, 1, 2, 1], [1, 1, 1, 2], [2, 1, 1, 1], [1, 2, 1, 1]])
    assert T.connected([[1, 1, 2, 2], [1, 1, 1, 2], [2, 1, 1, 1], [2, 2, 1, 1]])


def test_reference_unit_test_kernighan_lin():                         # TestKernighanLin1/2, :602-676
    Wa = np.array([[0, 1, 2, 3, 2, 4], [1, 0, 1, 4, 2, 1], [2, 1, 0, 3, 2, 1], [3, 4, 3, 0, 4, 3], [2, 2, 2, 4, 0, 2],
                   [4, 1, 1, 3, 2, 0]], np.float32)
    Wb = np.array([[0, 1, 0, 0, 1, 1, 0, 0], [1, 0, 0, 0, 1, 1, 0, 0], [0, 0, 0, 1, 0, 1, 1, 1], [0, 0, 1, 0, 0, 0, 1, 1],
                   [1, 1, 0, 0, 0, 1, 0, 0], [1, 1, 1, 0, 1, 0, 0, 0], [0, 0, 1, 1, 0, 0, 0, 1], [0, 0, 1, 1, 0, 0, 1, 0]], np.float32)
    for W, correct in ((Wa, [0, 1, 0, 1, 1, 0]), (Wb, [0, 0, 1, 1, 0, 0, 1, 1])):
        stop, P, npart, pairs = T.bisect(W, np.zeros(W.shape[0], np.int32), 1, seed=1)
        assert stop is False and npart == 2 and pairs == [(0, 1)]
        errors = int(np.sum(P != np.array(correct)))
        assert errors in (0, len(correct))                            # either naming of the two halves


def test_reference_unit_test_trees_have_the_expected_size():          # TestComputeTreesFromRoot1, TestComputeTrees1/2
    topo, scan, d = T.compute_trees(W8, 0.7, True)
    assert topo.shape == (8, 15) and scan.shape == (8, 5) and d == 3
    rng = np.random.default_rng(1)
    for n in range(2, 17):
        for bt in ((False, True) if n <= 6 else (False,)):
            u = rng.uniform(0, 1, (n, n))
            W = np.triu(np.where(u < 0.33, 1.0, np.where(u < 0.66, 2.0, 3.0)), 1)
            topo, scan, d = T.compute_trees(W + W.T, 0.7, bt)
            assert topo.shape == (n, (2 << d) - 1) and scan.shape == (n, d + 2)
            for r in range(n):
                assert topo[r, 0] == r and set(topo[r, scan[r, d]:].tolist()) == set(range(n))


# ---- the link matrix (GetP2PWeight, gpu_topology.h:137-253) -------------------------------------------------------
def test_link_weights_follow_get_p2p_weight():
    acc8 = np.array([[c in ".v"[1:] for c in row] for row in
                     (".vvvv...", "v.vv.v..", "vv.v..v.", "vvv....v", "v....vvv", ".v..v.vv", "..v.vv.v", "...vvvv.")], np.int32)
    # CUDA 9.0 on p3.16xlarge: the attribute ranks NVLink pairs above PCI-E pairs -> trusted; the machine is
    # connected over NVLink alone -> PCI-E links (weight 1) are dropped
    W = T.link_weights(W8.astype(np.int32) - 1 + np.eye(8, dtype=np.int32), acc8)
    assert np.array_equal(W, np.where(W8 == 1, 0, W8))
    # CUDA 9.2: double NVLink pairs rank like PCI-E (gpu_topology.h:192-205) -> not trusted -> peer access = 2
    bad = np.where(W8 == 3, 1, W8)
    W = T.link_weights(bad.astype(np.int32) - 1 + np.eye(8, dtype=np.int32), acc8)
    assert np.array_equal(W, np.where(acc8 > 0, 2.0, 0.0))
    # behind one switch every pair maps each other and ranks 0: all 2s off the diagonal
    for n in (2, 4, 8):
        full = 1 - np.eye(n, dtype=np.int32)
        assert np.array_equal(T.link_weights(np.zeros((n, n), np.int32), full), 2.0 * full)
    # two NVLink islands: not connected -> PCI-E links stay, discounted to 1/n
    acc4 = np.array([[0, 1, 0, 0], [1, 0, 0, 0], [0, 0, 0, 1], [0, 0, 1, 0]], np.int32)
    W = T.link_weights(acc4.copy(), acc4)
    want = np.where(acc4 > 0, 2.0, 0.25).astype(np.float32)
    np.fill_diagonal(want, 0.0)
    assert np.array_equal(W, want)


def test_link_matrix_override_for_tests(monkeypatch):
    monkeypatch.setenv("MXKV_B200_TREE_LINKS", ",".join(str(int(v)) for v in W8.ravel()))
    assert np.array_equal(T.query_links(list(range(8))), W8)
    with pytest.raises(mx.MXNetError, match="MXKV_B200_TREE_LINKS"):
        T.query_links([0, 1, 2])


# ---- add schedules: the kernel's evaluator vs CommDeviceTree::ReduceInner restated -----------------------------------
def test_reduce_programs_reproduce_reduce_inner_on_every_golden_tree(golden):
    rng = np.random.default_rng(3)
    trees = nontrivial = 0
    for i in range(int(golden["n_cases"])):
        if "case_%d_topo" % i not in golden.files:
            continue
        topo, scan = golden["case_%d_topo" % i].astype(np.int64), golden["case_%d_scan" % i].astype(np.int64)
        n = topo.shape[0]
        if n > 8:                       # one NVSwitch domain: the kernel holds at most 3 pending partial sums
            with pytest.raises(mx.MXNetError):
                T.reduce_program(topo[0], scan[0], n)
            continue
        depth = scan.shape[1] - 2
        srcs = [rng.uniform(-1, 1, 257).astype(np.float32) * np.float32(10.0 ** rng.integers(-3, 4)) for _ in range(n)]
        plain = O.sum_device(srcs)
        for r in range(n):
            leaves, prog = T.reduce_program(topo[r], scan[r], n)
            assert sorted(leaves.tolist()) == list(range(n)) and bin(prog).count("1") == n and prog.bit_length() == 2 * n - 1
            want = O.tree_reduce(srcs, topo[r], scan[r], depth)
            got = T.run_program([srcs[l] for l in leaves], prog)
            assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), (i, r)
            trees += 1
            nontrivial += int(not np.array_equal(got.view(np.uint32), plain.view(np.uint32)))
    assert trees > 300 and nontrivial > 200


def test_oracle_sliced_reduce_cuts_rows_like_the_reference():
    """comm_tree.h:203-234: slice_size = rows // n, the last slice takes the remainder; below the bound or with fewer
    than 2n rows the key goes up tree 0 whole."""
    n = 4
    topo, scan, d = T.compute_trees(2.0 * (np.ones((n, n)) - np.eye(n)))
    rng = np.random.default_rng(9)
    srcs = [rng.uniform(-1, 1, (11, 5)).astype(np.float32) for _ in range(n)]
    whole = O.sum_tree(srcs, topo, scan, d, bound=10 ** 7)
    assert np.array_equal(whole, O.tree_reduce(srcs, topo[0], scan[0], d))
    sliced = O.sum_tree(srcs, topo, scan, d, bound=10)
    for i, (lo, hi) in enumerate(((0, 2), (2, 4), (4, 6), (6, 11))):
        assert np.array_equal(sliced[lo:hi], O.tree_reduce([s[lo:hi] for s in srcs], topo[i], scan[i], d))
    few_rows = [s[:7] for s in srcs]                                   # 7 < 2n rows: not sliced
    assert np.array_equal(O.sum_tree(few_rows, topo, scan, d, bound=10), O.tree_reduce(few_rows, topo[0], scan[0], d))
