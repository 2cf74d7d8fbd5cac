#!/usr/bin/env python3
"""Regenerates tests/golden/ from a checkout of neo4j-labs/graph:

  python tests/golden/make_golden.py <path of the reference checkout>

The Rust reference cannot be executed here (no cargo/rustc), so the golden OUTPUTS below are
transcribed from the assertions of the reference's own tests — each entry carries the file:line
it was read from — and the golden INPUT files are the reference's test resources, copied as data
(they are binary/text fixtures, not source code).  It rewrites `reference_goldens.json` and refreshes
the resource copies; nothing under tests/ reads the reference checkout at test time.
"""
import json
import shutil
import sys
from pathlib import Path

HERE = Path(__file__).resolve().parent

RESOURCES = ["scale_8.graph500", "test.el", "example.el", "test.wel", "example.wel", "windows.el"]

GOLDENS = {
    "page_rank_13_nodes": {
        "cite": "crates/algos/src/lib.rs:96-140 (doc-test; also crates/mate/README)",
        "edges": [[1, 2], [2, 1], [4, 0], [4, 1], [5, 4], [5, 1], [5, 6], [6, 1], [6, 5], [7, 1],
                  [7, 5], [8, 1], [8, 5], [9, 1], [9, 5], [10, 1], [10, 5], [11, 5], [12, 5]],
        "layout": "Unsorted",
        "config": {"max_iterations": 10, "tolerance": 1e-4, "damping_factor": 0.85},
        "iterations": 10,
        "scores": ["0.024064068", "0.3145448", "0.27890152", "0.01153846", "0.029471997",
                   "0.06329483", "0.029471997", "0.01153846", "0.01153846", "0.01153846",
                   "0.01153846", "0.01153846", "0.01153846"],
    },
    "page_rank_two_components": {
        "cite": "crates/algos/src/page_rank.rs:176-197 (gdl (a)-->()-->()<--(a),(b)-->()-->()<--(b))",
        "edges": [[0, 1], [1, 2], [0, 2], [3, 4], [4, 5], [3, 5]],
        "layout": "Sorted",
        "config": {"max_iterations": 20, "tolerance": 1e-4, "damping_factor": 0.85},
        "scores": ["0.024999997", "0.035624996", "0.06590624", "0.024999997", "0.035624996",
                   "0.06590624"],
    },
    "page_rank_scale8_properties": {
        "cite": "crates/mate/tests/page_rank_test.py:6-33",
        "file": "scale_8.graph500",
        "layout": "Sorted",
        "damping_zero_score": 1.0 / 256.0,
    },
    "sssp": {
        "cite": "crates/algos/src/sssp.rs:283-313",
        "edges": [[0, 1, 4.0], [0, 2, 2.0], [1, 2, 5.0], [1, 3, 10.0], [2, 4, 3.0], [3, 5, 11.0],
                  [4, 3, 4.0]],
        "layout": "Deduplicated",
        "start_node": 0,
        "delta": 3.0,
        "distances": [0.0, 4.0, 2.0, 9.0, 5.0, 20.0],
    },
    "triangle_count": [
        {"cite": "crates/algos/src/triangle_count.rs:94-104; crates/mate/tests/triangle_count_test.py:12-32",
         "edges": [[0, 1], [1, 2], [2, 0], [3, 4], [4, 5], [5, 3]], "layout": "Deduplicated", "triangles": 2},
        {"cite": "crates/algos/src/triangle_count.rs:94-104 (gdl ids)",
         "edges": [[0, 1], [1, 2], [0, 2], [3, 4], [4, 5], [3, 5]], "layout": "Deduplicated", "triangles": 2},
        {"cite": "crates/algos/src/triangle_count.rs:107-117; triangle_count_test.py:35-55",
         "edges": [[0, 1], [1, 2], [2, 0], [0, 3], [3, 4], [4, 0]], "layout": "Deduplicated", "triangles": 2},
        {"cite": "crates/algos/src/triangle_count.rs:120-130; triangle_count_test.py:58-77",
         "edges": [[0, 1], [1, 2], [2, 0], [1, 3], [3, 2]], "layout": "Deduplicated", "triangles": 2},
    ],
    "triangle_count_scale8_degree_ordered": {
        "cite": "crates/mate/tests/triangle_count_test.py:5-9 after graph_test.py:56-64 (test_reorder mutates the package-scoped `ug`)",
        "file": "scale_8.graph500", "layout": "Sorted", "triangles": 227874,
    },
    "scale8_lists": {
        "cite": "crates/builder/tests/builder.rs:449-491",
        "file": "scale_8.graph500", "layout": "Sorted",
        "node_count": 256, "edge_count": 4096,
        "out_neighbors_0": [37, 157],
        "in_neighbors_0": [12, 26, 50, 50, 52, 82, 82, 82, 106, 109, 172, 186, 250, 250],
        "neighbors_0": [12, 26, 37, 50, 50, 52, 82, 82, 82, 106, 109, 157, 172, 186, 250, 250],
    },
    "sort_and_deduplicate": {
        "cite": "crates/builder/src/graph/csr.rs:1011-1021",
        "offsets": [0, 3, 7, 7, 10], "targets": [1, 1, 0, 4, 2, 3, 2, 5, 6, 7],
        "new_offsets": [0, 1, 4, 4, 7], "new_targets": [1, 2, 3, 4, 5, 6, 7],
    },
    "to_undirected": {
        "cite": "crates/builder/src/graph/csr.rs:1195-1219 (single-thread order)",
        "edges": [[0, 1], [3, 0], [0, 3], [7, 0], [0, 42], [21, 0]],
        "neighbors_0": {"Unsorted": [1, 3, 42, 3, 7, 21], "Sorted": [1, 3, 3, 7, 21, 42],
                        "Deduplicated": [1, 3, 7, 21, 42]},
    },
    "to_undirected_layouts": {
        "cite": "crates/mate/tests/graph_test.py:21-53",
        "edges": [[0, 1], [0, 1], [0, 2], [1, 2], [2, 1], [0, 3]],
        "Sorted": [[1, 1, 2, 3], [0, 0, 2, 2], [0, 1, 1], [0]],
        "Deduplicated": [[1, 2, 3], [0, 2], [0, 1], [0]],
    },
    "relabel_by_degree": {
        "cite": "crates/builder/src/graph_ops.rs:718-774",
        "edges": [[0, 1], [1, 2], [1, 3], [2, 0], [2, 1], [2, 3], [3, 0], [3, 2]],
        "sorted_pairs": [[5, 2], [4, 3], [4, 1], [3, 0]],
        "new_id": [3, 2, 0, 1],
        "degrees": [5, 4, 4, 3],
        "neighbors": [[1, 1, 2, 2, 3], [0, 0, 2, 3], [0, 0, 1, 3], [0, 1, 2]],
    },
    "greedy_partition": {
        "cite": "crates/builder/src/graph_ops.rs:700-707 (node_map = identity, n = 10, batch 6, max 3)",
        "weights": [0, 1, 2, 3, 4, 5, 6, 7, 8, 9], "batch_size": 6, "max_batches": 3,
        "ranges": [0, 4, 6, 10],
    },
    "in_degree_partition_doc": {
        "cite": "crates/builder/src/graph_ops.rs:415-430 (doc-test)",
    },
    "afforest_union": {
        "cite": "crates/algos/src/afforest.rs:121-133",
        "unions": [[9, 7], [7, 4], [4, 2], [2, 0]], "size": 10, "find_9": 0,
    },
    "wcc_two_components": {
        "cite": "crates/algos/src/wcc.rs:307-329",
        "edges": [[0, 1], [2, 3]], "same": [[0, 1], [2, 3]], "different": [[1, 2]],
    },
    "edge_list_test_el": {
        "cite": "crates/mate/tests/graph_edgelist_test.py:5-24; crates/builder/tests/builder.rs:493-564",
        "file": "test.el", "node_count": 5, "edge_count": 6,
        "out_neighbors": [[1, 2], [2, 3], [4], [4], []],
        "neighbors": [[1, 2], [0, 2, 3], [0, 1, 4], [1, 4], [2, 3]],
    },
    "numpy_graph": {
        "cite": "crates/mate/tests/ds_test.py:7-62",
        "edges": [[0, 1], [2, 3], [4, 1]], "node_count": 5, "edge_count": 3,
        "neighbors": [[1], [0, 4], [3], [2], [1]],
        "out_neighbors": {"0": [1], "2": [3], "4": [1]}, "in_neighbors": {"1": [0, 4], "3": [2]},
    },
    "survey_derived": {
        "cite": "SURVEY.md header table (derived with throw-away restatements, NOT in the reference)",
        "scale8_triangles_sorted_unrelabelled": 256533,
        "scale8_triangles_deduplicated": 10508,
        "scale8_self_loops": 85, "scale8_duplicate_edges": 1925,
        "scale8_components": 16, "scale8_largest_component": 241,
    },
}


def main():
    if len(sys.argv) != 2:
        sys.exit(f"usage: {sys.argv[0]} <path of the reference checkout>")
    ref = Path(sys.argv[1])
    for name in RESOURCES:
        shutil.copyfile(ref / "resources" / name, HERE / name)
    (HERE / "reference_goldens.json").write_text(json.dumps(GOLDENS, indent=1) + "\n")
    print("wrote", HERE / "reference_goldens.json")


if __name__ == "__main__":
    main()
