"""utils/utils.py's name factories (get_activation, get_aggregation_function, get_gated_unit) and utils/model_utils.py's
name_to_model_class: the names accepted, the exception types and messages raised -- the REFERENCE's functions (run under
tests/tf1_shim) against the package's.  What the reference returned or raised for every name is stored in
tests/golden/ref_records.json (tests/golden/ref_records.py utils)."""
import importlib
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
for _p in (HERE, os.path.join(HERE, "golden")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import ref_records                                           # noqa: E402

mine = importlib.import_module("tf_gnn_samples_b200.utils")
scaffold = importlib.import_module("tf_gnn_samples_b200.scaffold")

ACTIVATION_NAMES = [None, "linear", "Linear", "tanh", "TANH", "relu", "ReLU", "leaky_relu", "Leaky_ReLU", "elu", "ELU", "selu", "gelu",
                    "GeLU", "sigmoid", "swish", "", "relu ", "leaky-relu"]
AGGREGATION_NAMES = ["sum", "max", "mean", "sqrt_n", "unsorted_segment_sum", "unsorted_segment_max", "unsorted_segment_mean",
                     "unsorted_segment_sqrt_n", "Sum", "MAX", "avg", "", None, "sqrt-n"]
CELL_NAMES = ["rnn", "RNN", "gru", "GRU", "Gru", "lstm", "cnn", ""]
MODEL_NAMES = ["ggnn", "GGNN", "ggnn_model", "gnn_edge_mlp", "gnn-edge-mlp", "GNN-Edge-MLP", "gnn_edge_mlp_model", "gnn_edge_mlp0",
               "gnn-edge-mlp0", "gnn_edge_mlp1", "GNN-Edge-MLP1", "gnn_film", "gnn-film", "GNN-FiLM", "gnn_film_model", "rgat",
               "rgat_model", "rgcn", "RGCN", "rgcn_model", "rgdcn", "rgdcn_model", "rgin", "RGIN", "rgin_model", "gcn", "gat", ""]


outcome = ref_records.outcome


@pytest.fixture(scope="module")
def reference():
    return ref_records.load()["utils"]


def test_activation_names_and_errors(reference):
    import math
    x = np.linspace(-3, 3, 25)
    elu = lambda v: np.where(v > 0, v, np.expm1(np.minimum(v, 0)))                          # noqa: E731
    values = {mine.ACT_LINEAR: lambda v: v, mine.ACT_TANH: np.tanh, mine.ACT_RELU: lambda v: np.maximum(v, 0),
              mine.ACT_LEAKY_RELU: lambda v: np.where(v > 0, v, 0.2 * v), mine.ACT_ELU: elu,
              mine.ACT_SELU: lambda v: 1.0507009873554804934193349852946 * np.where(v > 0, v, 1.6732632423543772848170429916717 * np.expm1(np.minimum(v, 0))),
              mine.ACT_GELU: lambda v: v * 0.5 * (1.0 + np.vectorize(math.erf)(v / np.sqrt(2.0)))}
    assert len(reference["activation"]) == len(ACTIVATION_NAMES)
    for name, ref in zip(ACTIVATION_NAMES, reference["activation"]):
        got = outcome(mine.get_activation, name)
        if ref[0] != "ok":
            assert got == ref, (name, got, ref)               # same exception type, same message
            continue
        assert got[0] == "ok", (name, got)
        want = np.array(ref[1])                              # the reference's function on x (None = no activation: x itself)
        assert np.allclose(values[got[1]](x), want, rtol=0, atol=1e-15), name


def test_aggregation_names_and_errors(reference):
    codes = {mine.AGG_SUM: "sum", mine.AGG_MAX: "max", mine.AGG_MEAN: "mean", mine.AGG_SQRT_N: "sqrt_n"}
    assert len(reference["aggregation"]) == len(AGGREGATION_NAMES)
    for name, ref in zip(AGGREGATION_NAMES, reference["aggregation"]):
        got = outcome(mine.get_aggregation_function, name)
        if ref[0] != "ok":
            assert got == ref, (name, got, ref)
        else:
            assert got[0] == "ok" and codes[got[1]] == ref[1], (name, got, ref)


def test_gated_unit_names_and_errors(reference):
    assert len(reference["gated_unit"]) == len(CELL_NAMES)
    for name, ref in zip(CELL_NAMES, reference["gated_unit"]):
        got = outcome(mine.get_gated_unit, 8, name, "tanh")
        if name.lower() == "lstm":                            # constructs in the reference, cannot be CALLED there (ggnn.py:92)
            assert ref[0] == "ok" and ref[2] == "ValueError" and got[0] == "NotImplementedError"
            continue
        if ref[0] != "ok":
            assert got == ref, (name, got, ref)
        else:
            cell = {"_SimpleRNNCell": mine.CELL_RNN, "_GRUCell": mine.CELL_GRU}[ref[1]]
            assert got == ["ok", (cell, mine.ACT_TANH)], (name, got)
    assert outcome(mine.get_gated_unit, 8, "gru", "swish") == reference["gated_unit_gru_swish"]


def test_model_names_resolve_like_name_to_model_class(reference):
    import test_reference_model_pin as P
    kinds = {v: k for k, v in P.MC.MODEL_CLASSES.items()}
    assert len(reference["model_names"]) == len(MODEL_NAMES)
    for name, ref in zip(MODEL_NAMES, reference["model_names"]):
        got = outcome(scaffold.model_default_params, name)
        if ref[0] != "ok":
            assert got == ref, (name, got, ref)
            continue
        _, cls_name, want = ref
        assert got[0] == "ok", (name, got)
        for k, v in got[1].items():
            assert want[k] == ref_records.jsonable(v), (name, k, want[k], v)
        assert scaffold.resolve_model_name(name)[0] == kinds[cls_name], name


def test_layer_function_signatures_equal_the_references(reference):
    """gnns/__init__.py exports seven sparse_<x>_layer functions; the package's take the same positional / keyword parameters in
    the same order with the same defaults, plus keyword-only extras (weights=, plan=, ...) that the reference cannot know."""
    import inspect
    pkg = importlib.import_module("tf_gnn_samples_b200.gnns")
    signatures = reference["layer_signatures"]
    assert sorted(signatures) == ["sparse_ggnn_layer", "sparse_gnn_edge_mlp_layer", "sparse_gnn_film_layer", "sparse_rgat_layer",
                                  "sparse_rgcn_layer", "sparse_rgdcn_layer", "sparse_rgin_layer"]
    for n, ref in signatures.items():
        got = inspect.signature(getattr(pkg, n)).parameters
        shared = [p for p in got.values() if p.kind != inspect.Parameter.KEYWORD_ONLY]
        assert [[p.name, repr(p.default)] for p in shared] == ref, (n, [p.name for p in shared], ref)
        extras = [p.name for p in got.values() if p.kind == inspect.Parameter.KEYWORD_ONLY]
        assert "weights" in extras, (n, extras)
