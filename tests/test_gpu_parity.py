"""Parity of the CUDA hot path (through the C ABI) against the CPU oracle and the reference goldens.
Integer / index results are bit-exact; PageRank: EXACT mode bit-exact, JACOBI mode within 1e-6
relative of the f64-accumulating oracle (the tolerance BASELINE.json's north_star states)."""
import numpy as np
import pytest

import oracle
from conftest import LAYOUTS, edges_to_arrays

pytestmark = pytest.mark.gpu

PR_RTOL = 1e-6
# the sweep error is a sum of n |new - old| terms, each a difference of nearly equal f32 values: ranks
# that agree to 1e-6 relative (sum of ranks <= 1) move it by at most ~1e-6 absolute
ERR_ATOL = 2e-6


@pytest.fixture(scope="module")
def gb():
    import graph_b200
    return graph_b200


def f32(strings):
    return np.array([np.float32(s) for s in strings], dtype=np.float32)


def layout_of(gb, name):
    return getattr(gb.Layout, name)


def oracle_digraph(src, dst, n, layout, w=None):
    out = oracle.csr_build(src, dst, n, oracle.OUTGOING, layout, w)
    inc = oracle.csr_build(src, dst, n, oracle.INCOMING, layout)
    return out, inc


@pytest.fixture(scope="module")
def rmat16():
    src, dst = oracle.rmat_edges(16, seed=42)
    n = 1 << 16
    out, inc = oracle_digraph(src, dst, n, oracle.SORTED)
    return src, dst, n, out, inc


# ---- synthetic stream + CSR build ------------------------------------------------------------
def test_rmat_stream_bit_exact(gb):
    import ctypes as C
    from graph_b200._capi import lib, check
    for scale, first, count in ((8, 0, 4096), (17, 12345, 100000), (26, (1 << 30) - 5000, 5000)):
        src = np.empty(count, np.uint32)
        dst = np.empty(count, np.uint32)
        check(lib.gb_rmat_edges(0, scale, 42, first, count, src.ctypes.data_as(C.c_void_p),
                                dst.ctypes.data_as(C.c_void_p)))
        osrc, odst = oracle.rmat_edges(scale, 42, first, count)
        assert (src == osrc).all() and (dst == odst).all()


@pytest.mark.parametrize("layout", ["Unsorted", "Sorted", "Deduplicated"])
def test_csr_build_matches_oracle(gb, scale8_edges, layout):
    src, dst, n = scale8_edges
    g = gb.DiGraph.from_numpy(np.stack([src, dst], 1), layout=layout_of(gb, layout), node_count=n)
    for which, direction in (("out", oracle.OUTGOING), ("in", oracle.INCOMING)):
        off, tgt = g.csr(which)
        ooff, otgt = oracle.csr_build(src, dst, n, direction, LAYOUTS[layout])
        assert (off == ooff).all() and (tgt == otgt).all(), (layout, which)
    ug = gb.Graph.from_numpy(np.stack([src, dst], 1), layout=layout_of(gb, layout), node_count=n)
    off, tgt = ug.csr()
    ooff, otgt = oracle.csr_build(src, dst, n, oracle.UNDIRECTED, LAYOUTS[layout])
    assert (off == ooff).all() and (tgt == otgt).all(), layout
    assert ug.edge_count() == len(otgt) // 2


def test_csr_build_rmat_device_equals_host_edges(gb):
    g = gb.DiGraph.rmat(14, seed=7, layout=gb.Layout.Sorted)
    src, dst = oracle.rmat_edges(14, seed=7)
    for which, direction in (("out", oracle.OUTGOING), ("in", oracle.INCOMING)):
        off, tgt = g.csr(which)
        ooff, otgt = oracle.csr_build(src, dst, 1 << 14, direction, oracle.SORTED)
        assert (off == ooff).all() and (tgt == otgt).all()


def test_reference_csr_goldens(gb, goldens, scale8_edges):
    g8 = goldens["scale8_lists"]
    src, dst, n = scale8_edges
    g = gb.DiGraph.from_numpy(np.stack([src, dst], 1), layout=gb.Layout.Sorted, node_count=n)
    assert g.out_neighbors(0).tolist() == g8["out_neighbors_0"]
    assert g.in_neighbors(0).tolist() == g8["in_neighbors_0"]
    ug = g.to_undirected(gb.Layout.Sorted)
    assert ug.neighbors(0).tolist() == g8["neighbors_0"]
    tu = goldens["to_undirected"]
    e = np.array(tu["edges"], dtype=np.uint32)
    d = gb.DiGraph.from_numpy(e)
    for name, want in tu["neighbors_0"].items():
        assert d.to_undirected(layout_of(gb, name)).neighbors(0).tolist() == want, name
    sd = goldens["sort_and_deduplicate"]
    off, tg = sd["offsets"], sd["targets"]
    edges = np.array([(r, t) for r in range(len(off) - 1) for t in tg[off[r]:off[r + 1]]], dtype=np.uint32)
    dd = gb.DiGraph.from_numpy(edges, layout=gb.Layout.Deduplicated)
    o, t = dd.csr("out")
    assert o[:len(off)].tolist() == sd["new_offsets"] and t.tolist() == sd["new_targets"]


def test_weighted_csr_keeps_values_with_targets(gb):
    src, dst = oracle.rmat_edges(10, seed=3)
    w = oracle.rmat_weights(3, 0, len(src))
    g = gb.DiGraph.from_numpy(np.stack([src, dst], 1), layout=gb.Layout.Sorted, weights=w, node_count=1 << 10)
    off, tgt = g.csr("out")
    got = sorted(zip(np.repeat(np.arange(1 << 10), np.diff(off.astype(np.int64))).tolist(), tgt.tolist(),
                     g.out_weights().tolist()))
    want = sorted(zip(src.tolist(), dst.tolist(), w.tolist()))
    assert got == want


def test_make_degree_ordered_matches_oracle(gb, goldens, scale8_edges):
    rg = goldens["relabel_by_degree"]
    ug = gb.Graph.from_numpy(np.array(rg["edges"], dtype=np.uint32))
    ug.make_degree_ordered()
    assert [ug.degree(v) for v in range(4)] == rg["degrees"]
    assert [ug.neighbors(v).tolist() for v in range(4)] == rg["neighbors"]
    for layout in (oracle.SORTED, oracle.DEDUPLICATED):
        src, dst = oracle.rmat_edges(12, seed=5)
        n = 1 << 12
        off, tgt = oracle.csr_build(src, dst, n, oracle.UNDIRECTED, layout)
        noff, ntgt, _ = oracle.make_degree_ordered(off, tgt)
        h = gb.Graph.from_csr(off, tgt)
        h.make_degree_ordered()
        goff, gtgt = h.csr()
        assert (goff == noff).all() and (gtgt == ntgt).all()


def test_in_degree_partition(gb, rmat16):
    src, dst, n, out, inc = rmat16
    g = gb.DiGraph.from_csr(out[0], out[1], inc[0], inc[1])
    for parts in (1, 2, 3, 8):
        want = oracle.in_degree_partition(inc[0], parts)
        got = g.in_degree_partition(parts)
        assert [a for a, _ in got] + [got[-1][1]] == want.tolist()


# ---- PageRank --------------------------------------------------------------------------------
def test_page_rank_reference_goldens_bit_exact(gb, goldens):
    g13 = goldens["page_rank_13_nodes"]
    g = gb.DiGraph.from_numpy(np.array(g13["edges"], dtype=np.uint32), layout=layout_of(gb, g13["layout"]))
    pr = g.page_rank(**g13["config"])
    assert pr.ran_iterations == g13["iterations"]
    assert pr.scores().tobytes() == f32(g13["scores"]).tobytes()
    g2 = goldens["page_rank_two_components"]
    g = gb.DiGraph.from_numpy(np.array(g2["edges"], dtype=np.uint32), layout=layout_of(gb, g2["layout"]))
    assert g.page_rank().scores().tobytes() == f32(g2["scores"]).tobytes()


def test_page_rank_example_el_config0(gb, golden_dir):
    """BASELINE.json configs[0]: resources/example.el, 10 iterations, damping 0.85."""
    g = gb.DiGraph.load(str(golden_dir / "example.el"), layout=gb.Layout.Sorted, file_format=gb.FileFormat.EdgeList)
    src, dst = oracle.edgelist_parse((golden_dir / "example.el").read_bytes())
    out, inc = oracle_digraph(src, dst, 4, oracle.SORTED)
    want, it, err = oracle.page_rank_seq(inc[0], inc[1], out[0], 10, 1e-4, 0.85)
    pr = g.page_rank(max_iterations=10, tolerance=1e-4, damping_factor=0.85)
    assert pr.ran_iterations == it and pr.scores().tobytes() == want.tobytes() and pr.error == err


@pytest.mark.parametrize("scale", [8, 12, 14])
def test_page_rank_exact_mode_equals_single_thread_reference(gb, scale):
    src, dst = oracle.rmat_edges(scale, seed=42)
    n = 1 << scale
    out, inc = oracle_digraph(src, dst, n, oracle.SORTED)
    g = gb.DiGraph.from_csr(out[0], out[1], inc[0], inc[1])
    for cfg in ({"max_iterations": 20, "tolerance": 1e-4}, {"max_iterations": 7, "tolerance": 0.0},
                {"max_iterations": 0, "tolerance": 1e-3, "damping_factor": 0.5}):
        kw = {"max_iterations": 20, "tolerance": 1e-4, "damping_factor": 0.85, **cfg}
        want, it, err = oracle.page_rank_seq(inc[0], inc[1], out[0], kw["max_iterations"], kw["tolerance"],
                                             kw["damping_factor"])
        pr = g.page_rank(mode="exact", **kw)
        assert pr.ran_iterations == it
        assert pr.scores().tobytes() == want.tobytes()
        assert pr.error == err


@pytest.mark.parametrize("scale", [16, 18, 20])
def test_page_rank_repeated_runs_are_bit_equal(gb, scale):
    """Regression: with <= 4 hot blocks (scale 18: exactly 4) the hub rows are completed by their k_pr_sell
    lane, so the parts of their cut segments must be summed BEFORE that kernel (k_pr_fixup), not by its
    first warps — a race that showed up as run-to-run differences in the last bits."""
    g = gb.DiGraph.rmat(scale, seed=7, layout=gb.Layout.Sorted)
    first = g.page_rank(max_iterations=20, tolerance=0.0, mode="jacobi").scores().tobytes()
    for _ in range(25):
        assert g.page_rank(max_iterations=20, tolerance=0.0, mode="jacobi").scores().tobytes() == first


@pytest.mark.parametrize("scale,seed", [(8, 42), (13, 42), (16, 42), (18, 7)])
def test_page_rank_jacobi_vs_oracle(gb, scale, seed):
    src, dst = oracle.rmat_edges(scale, seed=seed)
    n = 1 << scale
    out, inc = oracle_digraph(src, dst, n, oracle.SORTED)
    g = gb.DiGraph.from_csr(out[0], out[1], inc[0], inc[1])
    want, it, err = oracle.page_rank_jacobi(inc[0], inc[1], out[0], 20, 0.0, 0.85)
    pr = g.page_rank(max_iterations=20, tolerance=0.0, mode="jacobi")
    assert pr.ran_iterations == 20
    rel = np.abs(pr.scores() - want) / want
    assert rel.max() <= PR_RTOL, rel.max()
    assert abs(pr.error - err) <= ERR_ATOL
    # deterministic: a second run gives the same bits
    assert g.page_rank(max_iterations=20, tolerance=0.0, mode="jacobi").scores().tobytes() == pr.scores().tobytes()


def test_page_rank_jacobi_stop_rule(gb, rmat16):
    src, dst, n, out, inc = rmat16
    g = gb.DiGraph.from_csr(out[0], out[1], inc[0], inc[1])
    for tol, maxit in ((1e-4, 50), (1e-2, 20), (1.0, 20), (1e-7, 13)):
        want, it, err = oracle.page_rank_jacobi(inc[0], inc[1], out[0], maxit, tol, 0.85)
        pr = g.page_rank(max_iterations=maxit, tolerance=tol, mode="jacobi")
        assert pr.ran_iterations == it, (tol, maxit)
        assert np.max(np.abs(pr.scores() - want) / want) <= PR_RTOL
        assert abs(pr.error - err) <= ERR_ATOL
    # damping 0: one sweep, every score == 1/n exactly (page_rank_test.py:27-33)
    pr = g.page_rank(damping_factor=0.0, mode="jacobi")
    assert pr.ran_iterations == 1 and (pr.scores() == np.float32(1.0) / np.float32(n)).all()


def test_page_rank_jacobi_fixed_point_is_the_references(gb, rmat16):
    """Jacobi (device) and the reference's in-place sweep share one fixed point.  The reference's own
    sequential f32 row sums carry rounding noise that grows with the in-degree (5.2e-6 relative on the
    12804-edge hub of this graph, measured against exactly rounded f64 sums), so the 1e-6 gate is held
    against the f64-accumulating oracle and the in-place f32 reference is matched to its own noise."""
    src, dst, n, out, inc = rmat16
    g = gb.DiGraph.from_csr(out[0], out[1], inc[0], inc[1])
    pr = g.page_rank(max_iterations=200, tolerance=0.0, mode="jacobi")
    j64, _, _ = oracle.page_rank_jacobi(inc[0], inc[1], out[0], 200, 0.0, 0.85, acc64=True)
    assert np.max(np.abs(pr.scores() - j64) / j64) <= PR_RTOL
    ref, _, _ = oracle.page_rank_seq(inc[0], inc[1], out[0], 200, 0.0, 0.85)
    ref_noise = np.max(np.abs(ref - j64) / j64)
    assert np.max(np.abs(pr.scores() - ref) / ref) <= ref_noise + PR_RTOL
    assert ref_noise < 2e-5


def test_page_rank_edge_cases(gb):
    # dangling nodes, isolated nodes, self loops, duplicate edges, a node that only has out-edges
    e = np.array([[0, 1], [0, 1], [1, 1], [2, 0], [5, 0], [5, 5], [3, 1]], dtype=np.uint32)
    for layout in ("Sorted", "Unsorted", "Deduplicated"):
        g = gb.DiGraph.from_numpy(e, layout=layout_of(gb, layout), node_count=8)
        src, dst, _ = edges_to_arrays(e)
        out, inc = oracle_digraph(src, dst, 8, LAYOUTS[layout])
        want, it, err = oracle.page_rank_seq(inc[0], inc[1], out[0], 20, 1e-4, 0.85)
        pr = g.page_rank(mode="exact")
        assert pr.ran_iterations == it and pr.scores().tobytes() == want.tobytes()
        wj, itj, _ = oracle.page_rank_jacobi(inc[0], inc[1], out[0], 20, 1e-4, 0.85)
        pj = g.page_rank(mode="jacobi")
        assert pj.ran_iterations == itj and np.max(np.abs(pj.scores() - wj) / wj) <= PR_RTOL
    # a graph whose nodes have no edges at all
    g = gb.DiGraph.from_numpy(np.array([[0, 1]], dtype=np.uint32), node_count=5)
    pj = g.page_rank(mode="jacobi", max_iterations=3, tolerance=0.0)
    out, inc = oracle_digraph(np.array([0], np.uint32), np.array([1], np.uint32), 5, oracle.UNSORTED)
    wj, _, ej = oracle.page_rank_jacobi(inc[0], inc[1], out[0], 3, 0.0, 0.85)
    assert pj.scores().tobytes() == wj.tobytes() and abs(pj.error - ej) < 1e-12
    with pytest.raises(ValueError):
        g.page_rank(max_iterations=0, tolerance=0.0)


def test_page_rank_scale22_matches_oracle(gb):
    """BASELINE.json configs[1]: RMAT scale-22, 20 sweeps, every rank within 1e-6 of the f64-accumulating
    oracle on the same CSR (the device CSR build is checked against the oracle's separately)."""
    g = gb.DiGraph.rmat(22, seed=42, layout=gb.Layout.Sorted)
    ooff, _ = g.csr("out")
    ioff, itgt = g.csr("in")
    want, it, err = oracle.page_rank_jacobi(ioff, itgt, ooff, 20, 0.0, 0.85, acc64=True)
    pr = g.page_rank(max_iterations=20, tolerance=0.0, mode="jacobi")
    assert pr.ran_iterations == it == 20
    rel = np.abs(pr.scores() - want) / want
    assert rel.max() <= PR_RTOL, rel.max()
    assert abs(pr.error - err) <= 4 * ERR_ATOL


def test_page_rank_full_size_properties(gb):
    """BASELINE.json configs[1] size (RMAT scale-22, 20 sweeps): size-independent properties."""
    g = gb.DiGraph.rmat(22, seed=42, layout=gb.Layout.Sorted)
    n = 1 << 22
    pr = g.page_rank(max_iterations=20, tolerance=0.0, mode="jacobi")
    s = pr.scores()
    base = (np.float32(1.0) - np.float32(0.85)) / np.float32(n)
    assert pr.ran_iterations == 20 and np.isfinite(s).all() and (s >= base).all()
    ioff, _ = g.csr("in")
    indeg = np.diff(ioff.astype(np.int64))
    assert (s[indeg == 0] == base).all()          # no in-edges -> exactly the base score
    assert 0.0 < float(s.astype(np.float64).sum()) <= 1.0 + 1e-6   # no dangling redistribution
    # one more sweep from the converged state changes nothing beyond rounding (fixed point)
    pr2 = g.page_rank(max_iterations=60, tolerance=0.0, mode="jacobi")
    pr3 = g.page_rank(max_iterations=61, tolerance=0.0, mode="jacobi")
    assert np.max(np.abs(pr2.scores() - pr3.scores()) / pr3.scores()) < 1e-5
    assert pr3.error < 1e-5
    # spot-check 64 rows against an f64 evaluation of the update rule on the returned vector
    ooff, _ = g.csr("out")
    _, itgt = g.csr("in")
    outdeg = np.diff(ooff.astype(np.int64)).astype(np.float32)
    with np.errstate(divide="ignore"):
        x = pr2.scores() / outdeg
    rng = np.random.default_rng(0)
    rows = np.concatenate([rng.integers(0, n, 60), np.argsort(indeg)[-4:]])
    for u in rows:
        tot = x[itgt[ioff[u]:ioff[u + 1]]].astype(np.float64).sum()
        want = float(base) + 0.85 * tot
        assert abs(float(pr3.scores()[u]) - want) <= 2e-5 * want


# ---- WCC ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("scale,seed", [(8, 42), (14, 1), (18, 42)])
def test_wcc_bit_exact(gb, scale, seed):
    src, dst = oracle.rmat_edges(scale, seed=seed)
    n = 1 << scale
    out, inc = oracle_digraph(src, dst, n, oracle.SORTED)
    g = gb.DiGraph.from_csr(out[0], out[1], inc[0], inc[1])
    want = oracle.wcc_min_label(out[0], out[1])
    if scale <= 14:
        assert (oracle.wcc_afforest(out[0], out[1], inc[0], inc[1]) == want).all()
    for kw in ({}, {"neighbor_rounds": 0}, {"neighbor_rounds": 1, "sampling_size": 16},
               {"neighbor_rounds": 5, "sampling_size": 0}, {"neighbor_rounds": 100}):
        assert (g.wcc(**kw).components() == want).all(), kw


def test_wcc_goldens_and_structured_graphs(gb, goldens, scale8_edges):
    src, dst, n = scale8_edges
    g = gb.DiGraph.from_numpy(np.stack([src, dst], 1), layout=gb.Layout.Sorted, node_count=n)
    comp = g.wcc().components()
    sd = goldens["survey_derived"]
    labels, counts = np.unique(comp, return_counts=True)
    assert len(labels) == sd["scale8_components"] and counts.max() == sd["scale8_largest_component"]
    au = goldens["afforest_union"]
    g = gb.DiGraph.from_numpy(np.array(au["unions"], dtype=np.uint32), node_count=au["size"])
    assert g.wcc().components()[9] == au["find_9"]
    # a long path (deep pointer chains) and a star, in adversarial id order
    k = 50000
    path = np.stack([np.arange(k - 1, 0, -1), np.arange(k - 2, -1, -1)], 1).astype(np.uint32)
    assert (gb.DiGraph.from_numpy(path).wcc().components() == 0).all()
    star = np.stack([np.full(k - 1, k - 1), np.arange(k - 1)], 1).astype(np.uint32)
    assert (gb.DiGraph.from_numpy(star).wcc().components() == 0).all()


def test_wcc_full_size_properties(gb):
    """BASELINE.json configs[2] size (RMAT scale-24): labels are roots, idempotent, edges stay inside."""
    g = gb.DiGraph.rmat(24, seed=42, layout=gb.Layout.Sorted)
    comp = g.wcc().components()
    n = 1 << 24
    assert (comp <= np.arange(n, dtype=np.uint32)).all()     # parent[x] <= x
    assert (comp[comp] == comp).all()                        # every label is its own root
    ooff, otgt = g.csr("out")
    srcs = np.repeat(np.arange(n, dtype=np.uint32), np.diff(ooff.astype(np.int64)))
    assert (comp[srcs] == comp[otgt]).all()                  # no edge crosses components
    assert (g.wcc(neighbor_rounds=1).components() == comp).all()
    # bit-exact against the oracle at the stated size (the properties above cannot see over-merging)
    assert (comp == oracle.wcc_min_label(ooff, otgt)).all()


# ---- SSSP --------------------------------------------------------------------------------------
def test_sssp_reference_golden(gb, goldens):
    gs = goldens["sssp"]
    e = np.array(gs["edges"])
    g = gb.DiGraph.from_numpy(e[:, :2].astype(np.uint32), layout=layout_of(gb, gs["layout"]),
                              weights=e[:, 2].astype(np.float32))
    d = g.delta_stepping(start_node=gs["start_node"], delta=gs["delta"]).distances()
    assert d.tolist() == gs["distances"]


@pytest.mark.parametrize("scale,delta", [(10, 0.05), (14, 0.3), (16, 1000.0), (16, 0.01)])
def test_sssp_bit_exact(gb, scale, delta):
    src, dst = oracle.rmat_edges(scale, seed=42)
    w = oracle.rmat_weights(42, 0, len(src))
    n = 1 << scale
    off, tgt, ww = oracle.csr_build(src, dst, n, oracle.OUTGOING, oracle.SORTED, w)
    g = gb.DiGraph.from_numpy(np.stack([src, dst], 1), layout=gb.Layout.Sorted, weights=w, node_count=n)
    start = int(np.argmax(np.diff(off.astype(np.int64))))
    want = oracle.sssp_delta_stepping(off, tgt, ww, start, delta)
    assert (oracle.sssp_bellman_ford(off, tgt, ww, start) == want).all()
    got = g.delta_stepping(start_node=start, delta=delta).distances()
    assert got.tobytes() == want.tobytes()
    assert (got == np.finfo(np.float32).max).sum() == (want == np.finfo(np.float32).max).sum()


def test_sssp_errors(gb):
    g = gb.DiGraph.from_numpy(np.array([[0, 1]], dtype=np.uint32), weights=np.array([1.0], np.float32))
    with pytest.raises(ValueError):
        g.delta_stepping(start_node=7, delta=1.0)
    with pytest.raises(ValueError):
        g.delta_stepping(start_node=0, delta=0.0)
    with pytest.raises(ValueError):
        gb.DiGraph.from_numpy(np.array([[0, 1]], dtype=np.uint32)).delta_stepping(start_node=0, delta=1.0)


# ---- triangle count ----------------------------------------------------------------------------
def test_triangle_count_goldens(gb, goldens, scale8_edges):
    for t in goldens["triangle_count"]:
        ug = gb.Graph.from_numpy(np.array(t["edges"], dtype=np.uint32), layout=layout_of(gb, t["layout"]))
        assert ug.global_triangle_count().triangles == t["triangles"], t["cite"]
    src, dst, n = scale8_edges
    sd = goldens["survey_derived"]
    e = np.stack([src, dst], 1)
    ug = gb.Graph.from_numpy(e, layout=gb.Layout.Sorted, node_count=n)
    assert ug.global_triangle_count().triangles == sd["scale8_triangles_sorted_unrelabelled"]
    ug.make_degree_ordered()
    assert ug.global_triangle_count().triangles == goldens["triangle_count_scale8_degree_ordered"]["triangles"]
    ud = gb.Graph.from_numpy(e, layout=gb.Layout.Deduplicated, node_count=n)
    assert ud.global_triangle_count().triangles == sd["scale8_triangles_deduplicated"]


@pytest.mark.parametrize("scale,layout", [(10, "Sorted"), (13, "Sorted"), (13, "Deduplicated"), (15, "Sorted")])
def test_triangle_count_bit_exact(gb, scale, layout):
    src, dst = oracle.rmat_edges(scale, seed=42)
    n = 1 << scale
    off, tgt = oracle.csr_build(src, dst, n, oracle.UNDIRECTED, LAYOUTS[layout])
    ug = gb.Graph.from_csr(off, tgt)
    assert ug.global_triangle_count().triangles == oracle.triangle_count(off, tgt, threads=0)
    noff, ntgt, _ = oracle.make_degree_ordered(off, tgt)
    ug.make_degree_ordered()
    assert ug.global_triangle_count().triangles == oracle.triangle_count(noff, ntgt, threads=0)


def test_triangle_count_scale22_matches_oracle(gb):
    """BASELINE.json configs[3]: undirected RMAT scale-22, CsrLayout::Sorted — the count of the raw graph
    and of the degree-ordered graph, bit-exact against the multi-threaded oracle on the same CSR."""
    ug = gb.Graph.rmat(22, seed=42, layout=gb.Layout.Sorted)
    off, tgt = (a.copy() for a in ug.csr())   # copies: live views would block the relabelling below
    if oracle.hardware_threads() >= 16:     # the raw Sorted count is ~1e11 merge steps on the CPU
        assert ug.global_triangle_count().triangles == oracle.triangle_count(off, tgt, threads=0)
    ug.make_degree_ordered()
    noff, ntgt = ug.csr()
    want_off, want_tgt, _ = oracle.make_degree_ordered(off, tgt)
    assert (noff == want_off).all() and (ntgt == want_tgt).all()
    assert ug.global_triangle_count().triangles == oracle.triangle_count(noff, ntgt, threads=0)


def test_wrong_graph_kind_is_rejected(gb):
    e = np.array([[0, 1], [1, 2]], dtype=np.uint32)
    import ctypes as C
    from graph_b200._capi import lib
    d = gb.DiGraph.from_numpy(e)
    u = gb.Graph.from_numpy(e)
    tri = C.c_uint64(0)
    assert lib.gb_triangle_count(d._g, C.byref(tri)) == 4       # GB_ERR_UNSUPPORTED
    assert lib.gb_make_degree_ordered(d._g) == 4
    assert b"undirected" in lib.gb_last_error()
    out = C.c_void_p()
    assert lib.gb_to_undirected(u._g, 0, C.byref(out)) == 4
    assert lib.gb_page_rank(u._g, None, None, None, None) == 1  # GB_ERR_INVALID (NULL arguments)


# ---- one-shot host-CSR entry point and input validation ----------------------------------------
def test_page_rank_csr_one_shot_matches_resident_twin(gb, rmat16):
    import ctypes as C
    from graph_b200 import _capi
    from graph_b200._capi import lib, check
    src, dst, n, out, inc = rmat16
    P = lambda a: a.ctypes.data_as(C.c_void_p)
    for mode, maxit in ((_capi.PR_JACOBI, 20), (_capi.PR_EXACT, 5)):
        cfg = _capi.PageRankConfig(maxit, 0.0, 0.85, mode)
        scores = np.empty(n, np.float32)
        it, err = C.c_uint64(0), C.c_double(0.0)
        check(lib.gb_page_rank_csr_u32(0, n, P(inc[0]), P(inc[1]), P(out[0]), C.byref(cfg), P(scores), C.byref(it),
                                       C.byref(err)))
        g = gb.DiGraph.from_csr(out[0], out[1], inc[0], inc[1])
        want = g.page_rank(max_iterations=maxit, tolerance=0.0, mode="jacobi" if mode == _capi.PR_JACOBI else "exact")
        assert it.value == maxit and scores.tobytes() == want.scores().tobytes() and err.value == want.error


@pytest.mark.parametrize("chunks,mega", [(1, None), (3, None), (7, "200"), (16, None)])
def test_page_rank_csr_streamed_upload_matches_resident_twin(gb, rmat16, monkeypatch, chunks, mega):
    """gb_page_rank_csr_u32 streams the targets in row-aligned chunks and classifies each chunk while the
    next one is on the bus; the layout it builds is the one the resident twin builds (bit-equal ranks)."""
    import ctypes as C
    from graph_b200 import _capi
    from graph_b200._capi import lib, check
    src, dst, n, out, inc = rmat16
    P = lambda a: a.ctypes.data_as(C.c_void_p)
    if mega:
        monkeypatch.setenv("GB_PR_MEGA", mega)
    g = gb.DiGraph.from_csr(out[0], out[1], inc[0], inc[1])
    want = g.page_rank(max_iterations=12, tolerance=0.0, mode="jacobi")
    monkeypatch.setenv("GB_PR_FEED_MIN_EDGES", "0")
    monkeypatch.setenv("GB_PR_FEED_CHUNKS", str(chunks))
    cfg = _capi.PageRankConfig(12, 0.0, 0.85, _capi.PR_JACOBI)
    scores = np.empty(n, np.float32)
    it, err = C.c_uint64(0), C.c_double(0.0)
    check(lib.gb_page_rank_csr_u32(0, n, P(inc[0]), P(inc[1]), P(out[0]), C.byref(cfg), P(scores), C.byref(it),
                                   C.byref(err)))
    assert it.value == 12 and scores.tobytes() == want.scores().tobytes() and err.value == want.error
    # the streamed path validates like the resident one
    bad_tgt = inc[1].copy()
    bad_tgt[len(bad_tgt) // 2] = n + 5
    assert lib.gb_page_rank_csr_u32(0, n, P(inc[0]), P(bad_tgt), P(out[0]), C.byref(cfg), P(scores), C.byref(it),
                                    C.byref(err)) == 1
    assert b"targets >= node_count" in lib.gb_last_error()
    bad_off = inc[0].copy()
    bad_off[5], bad_off[6] = bad_off[6] + 3, bad_off[5]
    if bad_off[5] > bad_off[6]:
        assert lib.gb_page_rank_csr_u32(0, n, P(bad_off), P(inc[1]), P(out[0]), C.byref(cfg), P(scores), C.byref(it),
                                        C.byref(err)) == 1
        assert b"monotone" in lib.gb_last_error()


def test_invalid_host_csr_is_rejected(gb):
    off = np.array([0, 2, 3], np.uint32)
    tgt = np.array([1, 7, 0], np.uint32)          # 7 >= n
    with pytest.raises(ValueError, match="targets >= node_count"):
        gb.DiGraph.from_csr(off, tgt, off, np.array([1, 0, 0], np.uint32))
    bad_off = np.array([0, 3, 2], np.uint32)      # not monotone
    with pytest.raises(ValueError):
        gb.Graph.from_csr(bad_off, np.array([1, 0], np.uint32))
    with pytest.raises(ValueError, match="out of range|>= node_count"):
        gb.DiGraph.from_numpy(np.array([[0, 9]], dtype=np.uint32), node_count=4)


# ---- shard API on one GPU: several virtual ranks, dealt slices exchanged by plain copies ----------
@pytest.mark.parametrize("world", [2, 3, 8])
def test_shard_api_virtual_ranks_match_single_gpu(gb, world):
    import torch
    from graph_b200.multigpu import CudaShardBackend, owner_of_rows
    g = gb.DiGraph.rmat(15, seed=11, layout=gb.Layout.Sorted)
    n = g.node_count()
    sweeps, damping = 6, 0.85
    want = g.page_rank(max_iterations=sweeps, tolerance=0.0, damping_factor=damping, mode="jacobi")
    ranks = [CudaShardBackend(g, r, world) for r in range(world)]
    n_active = ranks[0].n_active
    assert sum(b.stats["local_rows"] for b in ranks) == n_active
    assert sum(b.stats["local_edges"] for b in ranks) == g.edge_count()
    dev = ranks[0].device
    owner = torch.from_numpy(owner_of_rows(np.arange(n), world)).to(dev)
    mine = [owner == r for r in range(world)]
    x = [[torch.zeros(n, dtype=torch.float32, device=dev) for _ in range(2)] for _ in range(world)]
    scores = [torch.empty(n, dtype=torch.float32, device=dev) for _ in range(world)]
    err = [torch.zeros(1, dtype=torch.float64, device=dev) for _ in range(world)]
    for r, b in enumerate(ranks):
        b.init(damping, x[r][0], x[r][1], scores[r])
    total = 0.0
    for sweep in range(1, sweeps + 1):
        cur, nxt = (sweep - 1) & 1, sweep & 1
        for r, b in enumerate(ranks):
            b.step(damping, sweep, x[r][cur], x[r][nxt], None, scores[r], err[r])
        torch.cuda.synchronize()
        for r in range(world):  # the all-gather: every rank's rows go to every other rank
            for q in range(world):
                if q != r:
                    x[q][nxt][mine[r]] = x[r][nxt][mine[r]]
        total = sum(float(e.item()) for e in err)
    full = torch.stack(scores).sum(dim=0)   # own rows + zeros elsewhere (rows without in-edges: rank 0)
    got = ranks[0].finish(full).cpu().numpy()
    # every (row, block) partial is the same set of addends on every shard count; only the tree that
    # adds a pair's 4-id groups depends on where the pair sits in its 32-group step: <= 1 ulp per partial
    assert np.max(np.abs(got - want.scores()) / want.scores()) <= 5e-7
    assert abs(total - want.error) <= 1e-7 + 1e-6 * want.error


@pytest.mark.parametrize("world", [2, 5])
def test_wcc_shard_phases_virtual_ranks_bit_exact(gb, world):
    """Multi-GPU WCC on one GPU: every virtual rank runs the phases on its vertex range over its own
    full parent array; the all-gather is a list of tensors.  Labels must equal the single-GPU run."""
    from graph_b200 import _capi
    from graph_b200.multigpu import CudaWccBackend, vertex_ranges
    g = gb.DiGraph.rmat(16, seed=3, layout=gb.Layout.Sorted)
    want = g.wcc().components()
    b = CudaWccBackend(g)
    ranges = vertex_ranges(g.node_count(), world)
    parents = [b.new_parent() for _ in range(world)]

    def merge_all():
        snap = [p.clone() for p in parents]
        for r, p in enumerate(parents):
            for q in range(world):
                if q != r:
                    b.phase(_capi.WCC_MERGE, p, other=snap[q])
            b.phase(_capi.WCC_COMPRESS, p)

    for r, p in enumerate(parents):
        b.phase(_capi.WCC_INIT, p)
        b.phase(_capi.WCC_SAMPLE, p, *ranges[r])
        b.phase(_capi.WCC_COMPRESS, p)
    merge_all()
    labels = [b.sample_label(p) for p in parents]
    assert len(set(labels)) == 1                      # same forest, same seed -> same giant component
    for r, p in enumerate(parents):
        b.phase(_capi.WCC_LINK_REMAINING, p, *ranges[r], labels[r][0], labels[r][1])
        b.phase(_capi.WCC_COMPRESS, p)
    merge_all()
    for p in parents:
        assert (p.cpu().numpy().view(np.uint32) == want).all()


def test_single_device_communicator(gb, rmat16):
    """gb_comm_* with one device: the same entry point a multi-GPU host uses, no peers."""
    src, dst, n, out, inc = rmat16
    g = gb.DiGraph.from_csr(out[0], out[1], inc[0], inc[1])
    comm = gb.Comm([0])
    assert comm.multicast is False
    want, it, err = oracle.page_rank_jacobi(inc[0], inc[1], out[0], 20, 0.0, 0.85)
    pr = comm.page_rank([g], max_iterations=20, tolerance=0.0)
    assert pr.ran_iterations == 20 and np.max(np.abs(pr.scores() - want) / want) <= PR_RTOL
    assert abs(pr.error - err) <= ERR_ATOL
    with pytest.raises(ValueError):
        comm.page_rank([g, g])


# ---- column-block layout under stress: tiny blocks / chunks so that segments are cut by chunk and
# step boundaries, several hot blocks, the fixup path -------------------------------------------------
@pytest.mark.parametrize("block,chunk,tau", [(1024, 32, 1.0), (4096, 64, 2.0), (2048, 32, 0.5), (32768, 0, 1e9)])
def test_page_rank_column_block_knobs(gb, monkeypatch, block, chunk, tau):
    monkeypatch.setenv("GB_PR_BLOCK", str(block))
    monkeypatch.setenv("GB_PR_CHUNK", str(chunk))
    monkeypatch.setenv("GB_PR_TAU", str(tau))
    monkeypatch.setenv("GB_PR_MEGA", "200")       # rows above 200 in-edges take the sort path of the layout build
    src, dst = oracle.rmat_edges(16, seed=5)
    n = 1 << 16
    out, inc = oracle_digraph(src, dst, n, oracle.SORTED)
    g = gb.DiGraph.from_csr(out[0], out[1], inc[0], inc[1])
    info = g.page_rank_plan_info()
    if tau < 100:
        assert info["hot_blocks"] > 1 and info["block_edges"] > 0.5 * info["local_edges"]
        if chunk == 32:
            assert info["cut_segments"] > 0          # the hub rows' segments span several chunks
    else:
        assert info["hot_blocks"] == 0 and info["block_edges"] == 0   # everything through SELL
    want, it, err = oracle.page_rank_jacobi(inc[0], inc[1], out[0], 20, 0.0, 0.85)
    pr = g.page_rank(max_iterations=20, tolerance=0.0, mode="jacobi")
    rel = np.abs(pr.scores() - want) / want
    assert rel.max() <= PR_RTOL, rel.max()
    assert abs(pr.error - err) <= ERR_ATOL
    assert g.page_rank(max_iterations=20, tolerance=0.0, mode="jacobi").scores().tobytes() == pr.scores().tobytes()
