"""The oracle is pinned against THE REFERENCE'S OWN CODE: tests/golden/ref_*.npz hold outputs of the unmodified
/root/reference/gnns/*.py + utils/utils.py executed through tests/tf1_shim (tests/golden/make_ref_fixtures.py).

  test_oracle_matches_reference_fixture      oracle float64 == reference-through-shim float64 to 1e-12 (small cases: every
                                             element; BASELINE configs 2-5: committed rows + projection + column sums), and
                                             the oracle's float32 mode tracks the reference's float32 arithmetic;
  test_reference_code_reproduces_fixtures    the reference re-executed through the shim (recorded in tests/golden/ref_records.json
                                             by tests/golden/ref_records.py layer_fixtures: the variables it created and a seeded
                                             summary of its float64 output) against the committed files and the oracle -- so
                                             the fixtures cannot drift from the reference;
  test_variable_names_round_trip             the variables the reference creates, sorted by checkpoint.sort_variables, feed the
                                             oracle and reproduce the same output (pins the TF-name mapping both ways);
  test_engine_matches_reference_fixture      -m gpu: the CUDA engine through the C ABI against the same fixtures at 1e-4, and
                                             within 10x of the reference path's own float32 error where that is larger
                                             (SURVEY.md 8c acceptance).
"""
import json
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
sys.path.insert(0, HERE)

import ref_cases as RC                       # noqa: E402
import ref_records                           # noqa: E402
from oracle import ref_layers as R           # noqa: E402
from helpers import assert_parity            # noqa: E402

SMALL = [n for n, c in RC.CASES.items() if not c.get("big")]
BIG = [n for n, c in RC.CASES.items() if c.get("big")]
# the heavy float64 oracle passes (QM9-10k x 4 timesteps, 1M-edge FiLM) take tens of seconds each: CPU suite runs them once
BIG_CPU = ["config2_rgcn_ppi", "config4_rgat_ppi", "config5_film_random", "config3_ggnn_qm9"]
REEXECUTED = SMALL + ["config2_rgcn_ppi", "config4_rgat_ppi"]


def load(name):
    path = RC.fixture_path(name)
    assert os.path.exists(path), "missing fixture %s (python tests/golden/make_ref_fixtures.py %s)" % (path, name)
    return np.load(path)


def oracle_run(case, h, adj, indeg, weights, dtype):
    args = (indeg,) if case["indeg"] else ()
    return R.LAYERS[case["kind"]](h, adj, *args, **case["kw"], weights=weights, dtype=dtype)


def check_inputs(z, h, adj, indeg):
    assert float(z["h_sum"]) == float(np.asarray(h, np.float64).sum()), "seeded node states drifted from the fixture's"
    np.testing.assert_array_equal(z["adj_len"], [len(a) for a in adj])
    np.testing.assert_array_equal(z["adj_sum"], [int(np.asarray(a, np.int64).sum()) for a in adj])


@pytest.mark.parametrize("name", SMALL)
def test_oracle_matches_reference_fixture(name):
    case, z = RC.CASES[name], load(name)
    h, adj, indeg = case["graph"]()
    w = case["weights"]()
    np.testing.assert_array_equal(z["h"], h)
    check_inputs(z, h, adj, indeg)
    o64 = oracle_run(case, h, adj, indeg, w, np.float64)
    assert R.max_norm_rel_err(o64, z["out"]) <= 1e-12, "oracle float64 differs from the reference's code"
    np.testing.assert_allclose(o64, z["out"], rtol=1e-11, atol=1e-12)
    o32 = oracle_run(case, h, adj, indeg, w, np.float32)
    # same op order in float32: only BLAS summation order may differ between two numpy matmul shapes
    assert R.max_norm_rel_err(o32, z["out32"]) <= 2e-6
    assert float(z["err32"]) < 5e-6            # the reference's float32 arithmetic sits this close to the float64 truth


@pytest.mark.parametrize("name", BIG_CPU)
def test_oracle_matches_reference_fixture_baseline_configs(name):
    case, z = RC.CASES[name], load(name)
    h, adj, indeg = case["graph"]()
    check_inputs(z, h, adj, indeg)
    o64 = oracle_run(case, h, adj, indeg, case["weights"](), np.float64)
    err_rows, err_proj, err_col = RC.compare_with_summary(o64, z, name)
    assert max(err_rows, err_proj, err_col) <= 1e-12, (err_rows, err_proj, err_col)


@pytest.mark.parametrize("name", REEXECUTED)
def test_reference_code_reproduces_fixtures(name):
    case, z = RC.CASES[name], load(name)
    ran = ref_records.load()["layer_fixtures"][name]
    h, adj, indeg = case["graph"]()
    w = case["weights"]()
    assert ran["created"] == [str(s) for s in z["variable_names"]]
    o64 = oracle_run(case, h, adj, indeg, w, np.float64)
    assert ref_records.summary_err(o64, ran["out"]) <= 1e-12
    if case.get("big"):                        # committed rows, projection, column sums = those of the re-executed run
        assert {k: ref_records.sha(z[k]) for k in ran["fixture_summary"]} == ran["fixture_summary"]
    else:
        assert ref_records.summary_err(z["out"], ran["out"]) <= 1e-13


@pytest.mark.parametrize("name", SMALL)
def test_variable_names_round_trip(name):
    """reference-created variables (TF names) -> checkpoint.sort_variables -> oracle reproduces the reference output."""
    from tf_gnn_samples_b200 import checkpoint
    case, z = RC.CASES[name], load(name)
    named = {k[4:]: z[k] for k in z.files if k.startswith("var:")}
    assert sorted(named) == [str(s) for s in z["variable_names"]]
    assert all(n.startswith("graph_model/gnn_layer_0/") and n.endswith(":0") for n in named)
    sorted_vars = checkpoint.sort_variables(named)
    assert not sorted_vars["unused"] and not sorted_vars["outside"], sorted_vars["unused"]
    layer = checkpoint.split_layer_norms(sorted_vars["layers"][0], case["kw"].get("num_timesteps", 1))
    if case["kind"] == "rgdcn" and case["kw"].get("tie_channel_weights"):
        pass                                                     # one kernel per type, stored at channel 0
    h, adj, indeg = case["graph"]()
    o64 = oracle_run(case, h, adj, indeg, layer, np.float64)
    assert R.max_norm_rel_err(o64, z["out"]) <= 1e-12


def test_fixture_metadata_names_the_reference():
    for name in RC.CASES:
        z = load(name)
        meta = json.loads(str(z["meta"]))
        assert meta["kind"] == RC.CASES[name]["kind"] and "reference" in meta["source"]


# ------------------------------------------------------------------------------------------------------------
# GPU: the engine against the reference-generated fixtures
# ------------------------------------------------------------------------------------------------------------
def engine_run(case, h, adj, indeg, weights, device):
    import torch
    import tf_gnn_samples_b200 as G
    from tf_gnn_samples_b200 import weights as W
    fns = {"rgcn": G.sparse_rgcn_layer, "ggnn": G.sparse_ggnn_layer, "rgat": G.sparse_rgat_layer,
           "gnn-film": G.sparse_gnn_film_layer, "gnn-edge-mlp": G.sparse_gnn_edge_mlp_layer, "rgin": G.sparse_rgin_layer,
           "rgdcn": G.sparse_rgdcn_layer}
    ht = torch.as_tensor(h).to(device)
    args = (torch.as_tensor(indeg).to(device),) if case["indeg"] else ()
    out = fns[case["kind"]](ht, adj, *args, **case["kw"], weights=W.to_torch(weights, device))
    torch.cuda.synchronize()
    return out.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("name", SMALL)
def test_engine_matches_reference_fixture(cuda_device, name):
    case, z = RC.CASES[name], load(name)
    h, adj, indeg = case["graph"]()
    got = engine_run(case, h, adj, indeg, case["weights"](), cuda_device)
    err = assert_parity(got, z["out"], "reference fixture %s" % name, tol=1e-4)
    print("%s: engine %.2e, reference float32 path %.2e (max-norm rel. error vs float64 reference code)" % (name, err, float(z["err32"])))


@pytest.mark.gpu
@pytest.mark.parametrize("name", BIG)
def test_engine_matches_reference_fixture_baseline_configs(cuda_device, name):
    """BASELINE.json configs 2-5 at full size, tolerance 1e-4 (north star) on the committed rows, projection and column sums."""
    case, z = RC.CASES[name], load(name)
    h, adj, indeg = case["graph"]()
    check_inputs(z, h, adj, indeg)
    got = engine_run(case, h, adj, indeg, case["weights"](), cuda_device)
    assert np.all(np.isfinite(got))
    err_rows, err_proj, err_col = RC.compare_with_summary(got, z, name)
    err32 = float(z["err32"])
    print("%s: engine rows %.2e proj %.2e colsum %.2e | reference float32 path %.2e" % (name, err_rows, err_proj, err_col, err32))
    assert max(err_rows, err_proj, err_col) <= 1e-4, (err_rows, err_proj, err_col)
    assert err_rows <= max(10.0 * err32, 2e-5), "engine error %.2e is more than 10x the reference float32 path's %.2e" % (err_rows, err32)
