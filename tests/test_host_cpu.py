"""CPU-side checks of the product package: the C-ABI library loads and exports every symbol the
header declares, the host-side readers follow the reference formats, and — with no GPU in this
container — every constructor fails loudly instead of falling back to a CPU path."""
import ctypes
import re
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent


def header_functions():
    text = (ROOT / "include" / "graph_b200.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(gb_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    import graph_b200._capi as capi
    names = header_functions()
    assert len(names) >= 30
    lib = ctypes.CDLL(str(capi.LIB_PATH))
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, f"declared in include/graph_b200.h but not exported: {missing}"
    # and the ctypes table binds exactly the declared set
    assert sorted(capi.SIGNATURES) == names
    assert lib.gb_abi_version() == 1


def test_struct_layouts_match_header():
    import graph_b200._capi as capi
    assert ctypes.sizeof(capi.PageRankConfig) == 24
    assert ctypes.sizeof(capi.WccConfig) == 24
    assert ctypes.sizeof(capi.SsspConfig) == 16
    assert ctypes.sizeof(capi.GraphInfo) == 40
    assert ctypes.sizeof(capi.Timing) == 32


def test_no_cpu_fallback_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("this box has a GPU")
    import graph_b200 as gb
    assert gb.device_count() == 0
    with pytest.raises(gb.GraphB200Error, match="no CUDA device"):
        gb.DiGraph.from_numpy(np.array([[0, 1], [1, 2]], dtype=np.uint32))
    with pytest.raises(gb.GraphB200Error, match="no CUDA device"):
        gb.Graph.rmat(4)


def test_product_never_imports_the_oracle():
    for path in (ROOT / "graph_b200").rglob("*.py"):
        src = path.read_text()
        assert "import oracle" not in src and "from oracle" not in src, path


def test_graph500_reader_matches_reference_format(golden_dir, goldens, tmp_path):
    import graph_b200 as gb
    import oracle
    src, dst, n = gb._read_graph500(golden_dir / "scale_8.graph500")
    osrc, odst, on = oracle.graph500_decode((golden_dir / "scale_8.graph500").read_bytes())
    assert n == on == 256 and (src == osrc).all() and (dst == odst).all()
    # ids above 32 bits are rejected like Idx::new (index.rs:51-54)
    bad = np.array([1, 2, 0x00010000], dtype="<u4")
    p = tmp_path / "bad.graph500"
    bad.tofile(p)
    with pytest.raises(ValueError):
        gb._read_graph500(p)


def test_edge_list_reader(golden_dir):
    import graph_b200 as gb
    import oracle
    for name in ("test.el", "example.el", "windows.el"):
        src, dst = gb._read_edge_list(golden_dir / name)
        osrc, odst = oracle.edgelist_parse((golden_dir / name).read_bytes())
        assert (src == osrc).all() and (dst == odst).all(), name
    src, dst, w = gb._read_edge_list(golden_dir / "test.wel", with_values=True)
    o = oracle.edgelist_parse((golden_dir / "test.wel").read_bytes(), with_values=True)
    assert (src == o[0]).all() and (dst == o[1]).all() and (w == o[2]).all()


def test_edge_list_reader_is_bounded_by_the_buffer(tmp_path):
    """The parser works on (pointer, length): no trailing newline, a trailing space and a missing value
    must neither read past the buffer nor pull the next line's numbers into this line's value."""
    import ctypes as C
    import graph_b200 as gb
    from graph_b200._capi import lib, check

    def parse(text: bytes):
        # the buffer handed over is exactly len(text) bytes, followed by bytes that must not be read
        buf = C.create_string_buffer(text + b"9999", len(text) + 4)
        m = C.c_uint64(0)
        check(lib.gb_edge_list_parse(buf, len(text), None, None, None, C.byref(m)))
        src, dst, w = np.empty(m.value, np.uint32), np.empty(m.value, np.uint32), np.empty(m.value, np.float32)
        P = lambda a: a.ctypes.data_as(C.c_void_p)
        check(lib.gb_edge_list_parse(buf, len(text), P(src), P(dst), P(w), C.byref(m)))
        return list(zip(src.tolist(), dst.tolist(), w.tolist()))

    assert parse(b"0 1 2.5\n3 4 1.5") == [(0, 1, 2.5), (3, 4, 1.5)]          # no trailing newline
    assert parse(b"0 1 \n3 4") == [(0, 1, 0.0), (3, 4, 0.0)]                  # trailing space, value missing
    assert parse(b"0 1 7") == [(0, 1, 7.0)]                                    # value ends at the buffer end
    assert parse(b"5 6 1e-3\r\n7 8 +2\r\n") == [(5, 6, float(np.float32(0.001))), (7, 8, 2.0)]  # CRLF, exponent, +
    assert parse(b"1 2 0.25xyz\n3 4 5\n") == [(1, 2, 0.25), (3, 4, 5.0)]     # longest valid prefix (parse_partial)


def test_from_csr_rejects_short_arrays():
    import graph_b200 as gb
    off = np.array([0, 1, 2], np.uint32)
    tgt = np.array([1, 0], np.uint32)
    with pytest.raises(ValueError):
        gb.DiGraph.from_csr(np.array([], np.uint32), tgt, off, tgt)            # empty offsets
    with pytest.raises(ValueError):
        gb.DiGraph.from_csr(off, tgt, off[:2], tgt)                            # in offsets shorter than out
    with pytest.raises(ValueError):
        gb.DiGraph.from_csr(off, tgt[:1], off, tgt)                            # targets shorter than offsets[n]
    with pytest.raises(ValueError):
        gb.DiGraph.from_csr(off, tgt, off, tgt, out_weights=np.ones(1, np.float32))
    with pytest.raises(ValueError):
        gb.Graph.from_csr(off, tgt[:1])


def test_from_numpy_argument_checks():
    import graph_b200 as gb
    with pytest.raises(TypeError, match="2-dimensional array with at least 2 columns"):
        gb._edges_from_numpy(np.array([1, 2, 3], dtype=np.uint32))
    with pytest.raises(TypeError):
        gb._edges_from_numpy(np.array([[1], [2]], dtype=np.uint32))
    with pytest.raises(TypeError):
        gb._edges_from_numpy(np.array([[0.5, 1.0]]))
    s, d = gb._edges_from_numpy(np.array([[0, 1, 9], [2, 3, 9]], dtype=np.int64))
    assert s.dtype == np.uint32 and s.tolist() == [0, 2] and d.tolist() == [1, 3]
    assert gb._layout_value(None) == 0 and gb._layout_value(gb.Layout.Deduplicated) == 2
    with pytest.raises(TypeError):
        gb._layout_value("Sorted")


def test_defaults_match_reference_configs():
    import graph_b200 as gb
    assert (gb.PageRankConfig().max_iterations, gb.PageRankConfig().tolerance,
            gb.PageRankConfig().damping_factor) == (20, 1e-4, 0.85)  # page_rank.rs:46-48
    w = gb.WccConfig()
    assert (w.chunk_size, w.neighbor_rounds, w.sampling_size) == (16384, 2, 1024)  # wcc.rs:67-69


def test_graph_mate_shim_exposes_the_reference_module_surface():
    """crates/mate/graph_mate.pyi: the names the reference's tests and notebooks import."""
    import graph_mate
    import graph_b200
    for name in ("DiGraph", "Graph", "Layout", "FileFormat", "PageRankResult", "WccResult", "TriangleCountResult"):
        assert getattr(graph_mate, name) is getattr(graph_b200, name)
    for meth in ("load", "from_numpy", "from_pandas", "node_count", "edge_count", "out_degree", "in_degree",
                 "out_neighbors", "in_neighbors", "copy_out_neighbors", "copy_in_neighbors", "to_undirected",
                 "page_rank", "wcc"):
        assert callable(getattr(graph_mate.DiGraph, meth)), meth
    for meth in ("load", "from_numpy", "from_pandas", "node_count", "edge_count", "degree", "neighbors",
                 "copy_neighbors", "make_degree_ordered", "global_triangle_count"):
        assert callable(getattr(graph_mate.Graph, meth)), meth
    assert {graph_mate.Layout.Sorted.name, graph_mate.Layout.Unsorted.name, graph_mate.Layout.Deduplicated.name} == \
        {"Sorted", "Unsorted", "Deduplicated"}


def test_native_readers_match_oracle_on_large_inputs(tmp_path):
    """csrc/io.cu (multi-threaded, chunked at line boundaries) against the oracle's single-threaded
    restatement of input/graph500.rs and input/edgelist.rs, on inputs large enough for many chunks."""
    import graph_b200 as gb
    import oracle
    rng = np.random.default_rng(5)
    m = 600_000
    src = rng.integers(0, 1 << 20, m).astype(np.uint32)
    dst = rng.integers(0, 1 << 20, m).astype(np.uint32)
    # Graph500 packed records
    rec = np.zeros((m, 3), dtype="<u4")
    rec[:, 0], rec[:, 1] = src, dst
    p = tmp_path / "g.graph500"
    rec.tofile(p)
    s, d, n = gb._read_graph500(p)
    os_, od, on = oracle.graph500_decode(p.read_bytes())
    assert n == on == m // 16 and (s == os_).all() and (d == od).all() and (s == src).all()
    # text edge lists: plain, CRLF, weighted, and a last line without newline
    w = (rng.integers(0, 1 << 16, m) / 256.0).astype(np.float32)
    plain = "".join(f"{a} {b}\n" for a, b in zip(src.tolist(), dst.tolist()))
    crlf = plain.replace("\n", "\r\n")
    weighted = "".join(f"{a} {b} {c}\n" for a, b, c in zip(src.tolist(), dst.tolist(), w.tolist()))
    for name, text, vals in (("plain", plain, False), ("crlf", crlf, False), ("weighted", weighted, True),
                             ("no_trailing_newline", plain[:-1], False)):
        f = tmp_path / f"{name}.el"
        f.write_text(text)
        got = gb._read_edge_list(f, with_values=vals)
        want = oracle.edgelist_parse(text.encode(), with_values=vals)
        assert (got[0] == want[0]).all() and (got[1] == want[1]).all() and (got[0] == src).all(), name
        if vals:
            assert (got[2] == want[2]).all() and (got[2] == w).all()
    # ids above 32 bits are rejected like Idx::new (index.rs:51-54)
    f = tmp_path / "big.el"
    f.write_text("1 2\n4294967296 3\n")
    with pytest.raises(ValueError, match="32 bits"):
        gb._read_edge_list(f)
    (tmp_path / "empty.el").write_text("")
    e = gb._read_edge_list(tmp_path / "empty.el")
    assert len(e[0]) == 0


def test_graph500_writer_round_trips_through_both_readers(tmp_path):
    import graph_b200 as gb
    import oracle
    src, dst = oracle.rmat_edges(12, seed=3)           # 65536 edges, 4096 nodes = edges / 16
    p = tmp_path / "rmat12.graph500"
    gb.write_graph500(p, src, dst)
    assert p.stat().st_size == 12 * len(src)
    s, d, n = gb._read_graph500(p)
    os_, od, on = oracle.graph500_decode(p.read_bytes())
    assert n == on == 4096 and (s == src).all() and (d == dst).all() and (os_ == src).all() and (od == dst).all()
    with pytest.raises(ValueError):
        gb.write_graph500(p, src, dst[:-1])
