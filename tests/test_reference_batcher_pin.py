"""SURVEY.md 8 rows a12/a13 (the input tensor contract and the task batchers): batching.py against the REFERENCE'S OWN
loaders and minibatch iterators.

* tasks/qm9_task.py and tasks/ppi_task.py, executed unmodified under tests/tf1_shim (tf.placeholder as a feed_dict key,
  dpu_utils RichPath for local files -- nothing numerical is restated) on the 200 real QM9 validation molecules / a seeded
  PPI fold in the dgl layout, produce the minibatch feeds stored in tests/golden/ref_batcher_feeds.npz
  (tests/golden/make_batcher_fixtures.py); every feed is compared with batching.py's: adjacency lists bit-exact INCLUDING
  edge order, graph ids, in-degrees, features, targets / labels, counts;
* SHA-256 digests of the same feeds, of the reference's full QM9 validation batch and the exceptions the reference raises
  are recorded in tests/golden/ref_records.json (tests/golden/ref_records.py batchers): the fixture and batching.py must
  reproduce them;
* the two configurations the reference itself cannot run are pinned as such."""
import importlib
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
for p in (HERE, os.path.join(HERE, "golden")):
    if p not in sys.path:
        sys.path.insert(0, p)

import batcher_cases as BC      # noqa: E402
import ref_records              # noqa: E402

batching = importlib.import_module("tf_gnn_samples_b200.batching")
FIXTURE = os.path.join(HERE, "golden", "ref_batcher_feeds.npz")
RAN = ref_records.load()["batchers"]


@pytest.fixture(scope="module")
def ppi_dir(tmp_path_factory):
    return BC.write_ppi_dir(str(tmp_path_factory.mktemp("ppi")), "test")


@pytest.fixture(scope="module")
def fixture():
    return np.load(FIXTURE)


@pytest.mark.parametrize("case", sorted(BC.QM9_CASES))
def test_qm9_feeds_equal_the_committed_reference_feeds(case, fixture):
    params, budget = BC.QM9_CASES[case]
    got, L = BC.repo_qm9_feeds(params, budget)
    assert L == int(fixture[case + "/num_edge_types"])
    BC.compare_feeds(got, BC.unpack_feeds(fixture, case), case)


@pytest.mark.parametrize("case", sorted(BC.PPI_CASES))
def test_ppi_feeds_equal_the_committed_reference_feeds(case, fixture, ppi_dir):
    params, budget = BC.PPI_CASES[case]
    got, L = BC.repo_ppi_feeds(params, budget, ppi_dir)
    assert L == int(fixture[case + "/num_edge_types"])
    BC.compare_feeds(got, BC.unpack_feeds(fixture, case), case)


def check_digests(feeds, want, what):
    assert len(feeds) == len(want), (what, len(feeds), len(want))
    for i, (f, w) in enumerate(zip(feeds, want)):
        got = ref_records.feed_digests(f)
        assert set(got) == set(w), "%s minibatch %d: %s" % (what, i, sorted(set(got) ^ set(w)))
        assert got == w, "%s minibatch %d: %s" % (what, i, sorted(k for k in w if got[k] != w[k]))


@pytest.mark.parametrize("case", sorted(BC.QM9_CASES))
def test_qm9_feeds_equal_the_reference_loader_run_here(case, fixture):
    """batching.py's feeds and the committed fixture both equal a later, recorded run of the reference's QM9 loader."""
    params, budget = BC.QM9_CASES[case]
    ran = RAN["qm9"][case]
    got, L2 = BC.repo_qm9_feeds(params, budget)
    assert ran["num_edge_types"] == L2
    assert len(ran["feeds"]) > 1 or budget >= 5000
    check_digests(got, ran["feeds"], case)
    check_digests(BC.unpack_feeds(fixture, case), ran["feeds"], case + " (fixture is current)")


@pytest.mark.parametrize("case", sorted(BC.PPI_CASES))
def test_ppi_feeds_equal_the_reference_loader_run_here(case, fixture, ppi_dir):
    """batching.py's feeds and the committed fixture both equal a later, recorded run of the reference's PPI loader."""
    params, budget = BC.PPI_CASES[case]
    ran = RAN["ppi"][case]
    got, L2 = BC.repo_ppi_feeds(params, budget, ppi_dir)
    assert ran["num_edge_types"] == L2
    check_digests(got, ran["feeds"], case)
    check_digests(BC.unpack_feeds(fixture, case), ran["feeds"], case + " (fixture is current)")


@pytest.mark.parametrize("case", sorted(BC.QM9_REFERENCE_RAISES))
def test_untied_qm9_cannot_run_in_the_reference(case):
    """qm9_task.py:139-145 appends to the list it enumerates -> IndexError on the first molecule.  batching.py builds what the
    loop evidently meant (forward types, then their reversals) instead of failing; stated here so the difference is on record."""
    params, budget = BC.QM9_REFERENCE_RAISES[case]
    assert RAN["qm9_untied"][case] == "IndexError"
    feeds, L = BC.repo_qm9_feeds(params, budget)
    half = L // 2
    for f in feeds:
        for t in range(half):
            fwd, bwd = f["adjacency_e%d" % t], f["adjacency_e%d" % (half + t)]
            assert sorted(map(tuple, fwd[:, ::-1].tolist())) == list(map(tuple, bwd.tolist()))


def test_a_linkless_ppi_graph_breaks_the_reference_batcher_only(tmp_path):
    """A graph without links becomes np.array([]) of shape (0,) in ppi_task.py:152; packed next to a graph with links,
    np.concatenate (:247) raises.  batching.py keeps (0, 2) lists and packs it."""
    d = BC.write_ppi_dir(str(tmp_path), "test", linkless_graph=2)
    assert RAN["ppi_linkless"] == "ValueError"
    feeds, L = BC.repo_ppi_feeds({}, 10 ** 6, d)
    assert len(feeds) == 1 and feeds[0]["num_graphs"] == 5


def test_minibatches_cover_every_graph_once_and_respect_the_budget():
    graphs = batching.make_qm9_like_graphs(300, seed=5)
    seen, budget = 0, 97
    for batch, first in batching.minibatches(graphs, budget):
        assert first == seen and batch.num_graphs >= 1 and batch.num_nodes < budget
        nxt = first + batch.num_graphs
        if nxt < len(graphs):            # the next graph is the one that did not fit (strict '<' of ppi_task.py:220)
            assert not (batch.num_nodes + graphs[nxt].node_features.shape[0] < budget)
        seen = nxt
    assert seen == len(graphs)


def test_minibatches_refuse_a_graph_that_can_never_fit():
    graphs = batching.make_qm9_like_graphs(3, seed=1)
    n = graphs[1].node_features.shape[0]
    with pytest.raises(ValueError, match="does not fit"):
        list(batching.minibatches(graphs, n))       # node_offset + n < n is false even for an empty batch


def test_the_full_qm9_validation_set_is_packed_like_the_reference():
    """BASELINE config 3's batch: all 10,000 validation molecules of data/qm9/valid.jsonl.gz through the reference's loader and
    batcher in ONE minibatch (V = 180,560, M = 554,026, L = 5; recorded as digests) against batching.py on the
    structure-only archive that bench.py and test_reference_pin.py use for config 3 -- every edge in the same position."""
    ran = RAN["qm9_full_valid"]
    assert ran["num_edge_types"] == 5 and ran["num_minibatches"] == 1 and ran["counts"] == [10000, 180560, 554026]
    recs = batching.qm9_records_from_structure(os.path.join(HERE, "golden", "qm9_valid_structure.npz"))
    b, graph_nodes_list, _ = batching.qm9_batch(recs)
    assert len(b.adjacency_lists) == 5 and (b.num_graphs, b.num_nodes, b.num_edges) == (10000, 180560, 554026)
    got = {"graph_nodes_list": graph_nodes_list, "type_to_num_incoming_edges": b.type_to_num_incoming_edges}
    got.update(("adjacency_e%d" % i, a) for i, a in enumerate(b.adjacency_lists))
    assert ref_records.feed_digests(got) == ran["digests"]
