"""CPU: the C-ABI library loads and exports every symbol include/rgnn.h declares (no compute calls
without a GPU); host-side mirrors of utils/utils.py keep the reference's error behaviour; the batcher
reproduces the task batcher's tensor contract."""
import ctypes
import os
import re

import numpy as np
import pytest

import tf_gnn_samples_b200 as G
from tf_gnn_samples_b200 import _build, batching, engine, utils, weights as W

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    with open(os.path.join(ROOT, "include", "rgnn.h")) as f:
        return sorted(set(re.findall(r"RGNN_API\s+[\w\s\*]+?\b(rgnn_\w+)\s*\(", f.read())))


def test_header_declares_expected_entry_points():
    syms = declared_symbols()
    for name in ("rgnn_plan_create", "rgnn_rgcn_forward", "rgnn_ggnn_forward", "rgnn_rgat_forward",
                 "rgnn_film_forward", "rgnn_edge_mlp_forward", "rgnn_rgin_forward", "rgnn_last_error"):
        assert name in syms


def test_library_exports_every_declared_symbol():
    path = _build.build()                                   # nvcc cross-compiles without a GPU
    lib = ctypes.CDLL(path)
    for name in declared_symbols():
        assert hasattr(lib, name), "librgnn.so does not export %s" % name
    lib.rgnn_version.restype = ctypes.c_int
    assert lib.rgnn_version() == 200
    # every declared symbol has a ctypes signature in the binding and vice versa
    assert set(declared_symbols()) == set(engine.SIGNATURES) - (engine.OPTIONAL_SYMBOLS - set(declared_symbols()))


def test_no_cpu_fallback():
    import torch
    h = torch.zeros(4, 8)
    w = W.to_torch(W.rgcn_weights(1, 8, 8), "cpu")
    with pytest.raises(engine.RgnnError, match="no CPU path"):
        G.sparse_rgcn_layer(h, [np.zeros((0, 2), np.int32)], np.zeros((1, 4), np.float32), 8, weights=w)


def test_utils_error_behaviour():
    assert utils.get_activation("ReLU") == utils.ACT_RELU and utils.get_activation("TANH") == utils.ACT_TANH
    assert utils.get_activation(None) == utils.ACT_LINEAR and utils.get_activation("linear") == utils.ACT_LINEAR
    with pytest.raises(ValueError, match="Unknown activation function 'swish'!"):
        utils.get_activation("swish")
    assert utils.get_aggregation_function("sqrt_n") == utils.AGG_SQRT_N
    assert utils.get_aggregation_function("unsorted_segment_max") == utils.AGG_MAX
    with pytest.raises(ValueError, match="Unknown aggregation function 'SUM'!"):   # case-sensitive like utils.py:23-33
        utils.get_aggregation_function("SUM")
    assert utils.get_gated_unit(8, "GRU", "tanh") == (utils.CELL_GRU, utils.ACT_TANH)
    with pytest.raises(Exception, match="Unknown RNN cell type 'foo'."):
        utils.get_gated_unit(8, "foo", "tanh")
    with pytest.raises(NotImplementedError):
        utils.get_gated_unit(8, "lstm", "tanh")
    assert utils.SMALL_NUMBER == 1e-7 and utils.BIG_NUMBER == 1e7


def test_ppi_like_batch_contract():
    b = batching.ppi_like_batch()
    assert b.num_nodes == 2245 and b.num_edges == 120245 and len(b.adjacency_lists) == 3
    fwd, loops, bkwd = b.adjacency_lists
    assert all(a.dtype == np.int32 and a.shape[1] == 2 for a in b.adjacency_lists)
    assert np.array_equal(fwd[:, ::-1], bkwd)                                    # ppi_task.py:144-148
    assert np.array_equal(loops[:, 0], np.arange(2245)) and np.array_equal(loops[:, 0], loops[:, 1])   # :125-127
    c = b.type_to_num_incoming_edges
    assert c.dtype == np.float32 and c.shape == (3, 2245)
    for l, a in enumerate(b.adjacency_lists):
        assert np.array_equal(c[l], np.bincount(a[:, 1], minlength=2245))
    assert np.all(c[1] == 1)


def test_pack_batch_offsets_and_budget():
    gs = [batching.make_ppi_like_graph(100 + 10 * i, 300, seed=i) for i in range(4)]
    b = batching.pack_batch(gs)
    assert b.num_graphs == 4 and b.num_nodes == sum(100 + 10 * i for i in range(4))
    off = b.graph_node_offsets
    for l in range(3):                                                           # block-diagonal: ppi_task.py:228
        a = b.adjacency_lists[l]
        g_src = np.searchsorted(off, a[:, 0], side="right")
        g_tgt = np.searchsorted(off, a[:, 1], side="right")
        assert np.array_equal(g_src, g_tgt)
    # strict '<' packing budget of ppi_task.py:220
    assert batching.pack_batch(gs, max_nodes_per_batch=210).num_graphs == 1      # 100 + 110 < 210 is false
    assert batching.pack_batch(gs, max_nodes_per_batch=211).num_graphs == 2
    assert batching.pack_batch(gs, max_nodes_per_batch=101).num_graphs == 1
    # an edge type with no edges becomes a (0, 2) array (:246-249)
    g = batching.GraphSample([np.zeros((0, 2), np.int32), np.array([[0, 1]], np.int32)],
                             np.array([[0, 0], [0, 1]]), np.zeros((2, 3), np.float32))
    assert batching.pack_batch([g]).adjacency_lists[0].shape == (0, 2)


def test_qm9_like_shape_statistics():
    b = batching.qm9_like_batch(500, seed=1)
    assert len(b.adjacency_lists) == 4
    assert 16.5 < b.num_nodes / 500 < 19.5                                        # QM9 mean 18.0 nodes/graph
    assert 30 < b.num_edges / 500 < 45                                            # ~37 messages/graph (tied fwd/bkwd)
    a = b.adjacency_lists[0]
    both = set(map(tuple, a.tolist()))
    assert all((t, s) in both for (s, t) in list(both)[:200])                     # tie_fwd_bkwd: both directions


def test_weight_shapes():
    w = W.ggnn_weights(4, 32)
    assert w["cell"]["kernel"].shape == (32, 96) and w["cell"]["bias"].shape == (96,)
    u = w["cell"]["recurrent_kernel"][:, :32]
    np.testing.assert_allclose(u.T @ u, np.eye(32), atol=1e-5)                    # orthogonal recurrent init
    e = W.edge_mlp_weights(2, 16, 24, num_edge_hidden_layers=2)
    assert [k.shape for k in e["edge_mlps"][0]] == [(32, 24), (24, 24), (24, 24)]
    r = W.rgin_weights(2, 16, 24, num_edge_MLP_hidden_layers=None, num_aggr_MLP_hidden_layers=1, use_target_state_as_input=True)
    assert "edge_mlps" not in r and [k.shape for k in r["aggr_mlp"]] == [(32, 24), (24, 24)]


def _qm9_subset():
    import os
    from tf_gnn_samples_b200 import batching
    return batching.load_qm9_jsonl(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "qm9_valid_subset.json.gz"))


def test_qm9_records_to_batch_follows_the_reference_loader():
    """tasks/qm9_task.py:85-147,200-261 on 200 real QM9 validation records (tests/golden/make_qm9_subset.py)."""
    from tf_gnn_samples_b200 import batching
    recs = _qm9_subset()
    assert len(recs) == 200 and len(recs[0]["node_features"][0]) == 15 and len(recs[0]["targets"]) == 13
    raw_bonds = sum(len(r["graph"]) for r in recs)
    V = sum(len(r["node_features"]) for r in recs)
    b, graph_nodes_list, targets = batching.qm9_batch(recs)                       # defaults: self loops, tied directions
    assert len(b.adjacency_lists) == 5 and b.num_nodes == V and b.num_graphs == 200
    assert b.num_edges == 2 * raw_bonds + V                                      # both directions in the bond's type + one loop per node
    assert b.adjacency_lists[0].shape[0] == V and np.all(b.adjacency_lists[0][:, 0] == b.adjacency_lists[0][:, 1])
    assert np.all(b.type_to_num_incoming_edges[0] == 1)
    for l, a in enumerate(b.adjacency_lists):                                    # in-degrees are the bincount of the targets
        assert np.array_equal(b.type_to_num_incoming_edges[l], np.bincount(a[:, 1], minlength=V)), l
    first = batching.qm9_graph_to_sample(recs[0], 5)
    for a in first.adjacency_lists:                                              # sorted by (src, dst) (:135)
        assert [tuple(x) for x in a] == sorted(tuple(x) for x in a)
    assert graph_nodes_list.shape == (V,) and graph_nodes_list[0] == 0 and graph_nodes_list[-1] == 199
    assert targets.shape == (1, 200) and np.isclose(targets[0, 0], recs[0]["targets"][0][0])
    b4, _, _ = batching.qm9_batch(recs, add_self_loop_edges=False)                # BASELINE's "4 edge types"
    assert len(b4.adjacency_lists) == 4 and b4.num_edges == 2 * raw_bonds
    bu, _, _ = batching.qm9_batch(recs[:20], tie_fwd_bkwd_edges=False)            # untied: reversed lists as extra types
    assert len(bu.adjacency_lists) == 10
    for t in range(5):
        assert np.array_equal(np.sort(bu.adjacency_lists[5 + t][:, ::-1], axis=0), np.sort(bu.adjacency_lists[t], axis=0))
    small, _, _ = batching.qm9_batch(recs, max_nodes_per_batch=100)               # the packing loop stops before the limit
    assert small.num_nodes < 100 and small.num_graphs < 200


def test_qm9_structure_archive_reproduces_the_full_validation_batch():
    """tests/golden/qm9_valid_structure.npz (structure of all 10,000 validation molecules) -> the BASELINE config-3 batch:
    SURVEY.md 8d: V = 180,560, M = 373,466 (4 bond types) / 554,026 (with the self-loop type); and it agrees with the
    200-record subset that carries real features."""
    import os
    from tf_gnn_samples_b200 import batching
    here = os.path.dirname(os.path.abspath(__file__))
    recs = batching.qm9_records_from_structure(os.path.join(here, "golden", "qm9_valid_structure.npz"))
    assert len(recs) == 10000 and len(recs[0]["node_features"][0]) == 15
    b4, _, _ = batching.qm9_batch(recs, add_self_loop_edges=False)
    b5, gl, tg = batching.qm9_batch(recs)
    assert (b4.num_nodes, b4.num_edges, len(b4.adjacency_lists)) == (180560, 373466, 4)
    assert (b5.num_graphs, b5.num_nodes, b5.num_edges, len(b5.adjacency_lists)) == (10000, 180560, 554026, 5)
    assert gl.shape == (180560,) and tg.shape == (1, 10000)
    real = _qm9_subset()
    for r_struct, r_real in zip(recs[:200], real):
        assert r_struct["graph"] == r_real["graph"] and len(r_struct["node_features"]) == len(r_real["node_features"])


def test_ppi_fold_loader_follows_the_reference(tmp_path):
    """tasks/ppi_task.py:68-160 on a tiny data set written in the dgl ppi.zip layout: two graphs interleaved in node-id
    ranges [0, 4) and [4, 7), links in arbitrary order."""
    import json
    from tf_gnn_samples_b200 import batching
    links = [(0, 1), (5, 4), (2, 3), (3, 0), (6, 5), (1, 1)]
    (tmp_path / "train_graph.json").write_text(json.dumps({"links": [{"source": s, "target": t} for s, t in links]}))
    rng = np.random.default_rng(0)
    np.save(tmp_path / "train_feats.npy", rng.standard_normal((7, 5)).astype(np.float32))
    np.save(tmp_path / "train_labels.npy", (rng.random((7, 3)) < 0.5).astype(np.int64))
    np.save(tmp_path / "train_graph_id.npy", np.array([11, 11, 11, 11, 12, 12, 12]))
    graphs, labels = batching.load_ppi_fold(str(tmp_path), "train")
    assert len(graphs) == 2 and [g.node_features.shape[0] for g in graphs] == [4, 3] and labels[1].shape == (3, 3)
    g0, g1 = graphs
    assert len(g0.adjacency_lists) == 3                                       # fwd, self-loop, bkwd (:99-106)
    assert g0.adjacency_lists[0].tolist() == [[0, 1], [2, 3], [3, 0], [1, 1]]     # file order, ids already local
    assert g1.adjacency_lists[0].tolist() == [[1, 0], [2, 1]]                     # shifted by the graph's first node id 4
    assert g0.adjacency_lists[1].tolist() == [[i, i] for i in range(4)]
    assert g1.adjacency_lists[2].tolist() == [[0, 1], [1, 2]]                     # (tgt, src)
    assert g0.type_to_node_to_num_incoming_edges.tolist() == [[1, 2, 0, 1], [1, 1, 1, 1], [1, 1, 1, 1]]
    b = batching.pack_batch(graphs)
    assert b.num_nodes == 7 and b.num_edges == 6 + 7 + 6
    assert b.adjacency_lists[0].tolist()[-2:] == [[5, 4], [6, 5]]                 # second graph offset by 4 in the batch
    tied, _ = batching.load_ppi_fold(str(tmp_path), "train", add_self_loop_edges=False, tie_fwd_bkwd_edges=True)
    assert len(tied[0].adjacency_lists) == 1
    import pytest
    with pytest.raises(ValueError):
        batching.load_ppi_fold(str(tmp_path), "dev")


def test_header_is_plain_c_and_the_c_host_example_links():
    """include/rgnn.h must be consumable from C (the drop-in boundary is a C ABI, no C++ / torch types): compile the C99
    example against it with warnings on, and link it against the built library when the CUDA runtime library is present."""
    import shutil
    import subprocess
    import tempfile
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    src = os.path.join(ROOT, "examples", "c_abi_demo.c")
    with tempfile.TemporaryDirectory() as tmp:
        obj = os.path.join(tmp, "demo.o")
        res = subprocess.run([gcc, "-std=c99", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), "-c", src, "-o", obj],
                             capture_output=True, text=True)
        assert res.returncode == 0, res.stderr
        cudart = "/usr/local/cuda/lib64"
        if os.path.exists(os.path.join(cudart, "libcudart.so")):
            lib_dir = os.path.dirname(_build.build())
            res = subprocess.run([gcc, obj, "-o", os.path.join(tmp, "demo"), "-L", lib_dir, "-lrgnn", "-L", cudart, "-lcudart",
                                  "-Wl,-rpath," + lib_dir], capture_output=True, text=True)
            assert res.returncode == 0, res.stderr
