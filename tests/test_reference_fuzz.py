"""Randomised differential test: oracle/ref_layers.py against the REFERENCE's own layer functions (gnns/*.py through
tests/tf1_shim) on seeded random graphs, shapes and keyword arguments -- the corners the hand-picked fixtures may miss (edge
types without edges, isolated and duplicate-heavy nodes, d_in != state_dim, every activation x aggregation, MLP depths,
heads, channels, timesteps).  Both sides are float64 numpy in the same op order, so the bar is 1e-12.  What the reference
computed for every case (its exception, or a seeded summary of its output) is stored in tests/golden/ref_records.json
(tests/golden/ref_records.py fuzz); the GPU engine is tested against the same oracle over a far wider space than the
committed fixtures cover."""
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
for p in (HERE, os.path.join(HERE, "golden")):
    if p not in sys.path:
        sys.path.insert(0, p)

from oracle import ref_layers as R                        # noqa: E402
from tf_gnn_samples_b200 import weights as W              # noqa: E402
from helpers import node_states, tiny_graph               # noqa: E402
import ref_records                                        # noqa: E402

ACTS = [None, "linear", "tanh", "ReLU", "leaky_relu", "elu", "selu", "gelu"]
AGGS = ["sum", "max", "mean", "sqrt_n"]
CASES_PER_KIND = 40
KINDS = ["rgcn", "ggnn", "rgat", "gnn-film", "gnn-edge-mlp", "rgin", "rgdcn"]


def random_graph(rng):
    V = int(rng.integers(5, 40))
    L = int(rng.integers(1, 5))
    edges = tuple(int(rng.integers(0, 90)) if rng.random() > 0.2 else 0 for _ in range(L))
    adj, indeg = tiny_graph(V, edges, seed=int(rng.integers(1 << 30)), with_isolated=bool(rng.integers(2)),
                            duplicates=bool(rng.integers(2)))
    return V, L, adj, indeg


def pick(rng, options):
    return options[int(rng.integers(len(options)))]


def make_case(kind, rng):
    V, L, adj, indeg = random_graph(rng)
    T = int(rng.integers(1, 4))
    D = int(pick(rng, [4, 8, 12]))
    d_in = D if T > 1 or rng.random() < 0.5 else int(pick(rng, [4, 8, 12]))    # several timesteps feed the output back in
    seed = int(rng.integers(1 << 20))
    act = pick(rng, ACTS if kind == "ggnn" or rng.random() < 0.1 else ACTS[2:])   # None / 'linear' only run in the GGNN cell
    agg = pick(rng, AGGS)
    if kind == "rgcn":
        both = bool(rng.integers(2))
        kw = dict(state_dim=D, num_timesteps=T, activation_function=act, message_aggregation_function=agg,
                  normalize_by_num_incoming=bool(rng.integers(2)), use_both_source_and_target=both)
        w, needs_indeg = W.rgcn_weights(L, d_in, D, seed, use_both_source_and_target=both), True
    elif kind == "ggnn":
        d_in, cell = D, pick(rng, ["gru", "GRU", "rnn", "RNN"])
        kw = dict(state_dim=D, num_timesteps=T, gated_unit_type=cell, activation_function=act, message_aggregation_function=agg)
        w, needs_indeg = W.ggnn_weights(L, D, seed, cell=cell, random_bias=True), False
    elif kind == "rgat":
        heads = int(pick(rng, [h for h in (1, 2, 4) if D % h == 0]))
        kw = dict(state_dim=D, num_heads=heads, num_timesteps=T, activation_function=act)
        w, needs_indeg = W.rgat_weights(L, d_in, D, seed), False
    elif kind == "gnn-film":
        kw = dict(state_dim=D, num_timesteps=T, activation_function=act, message_aggregation_function=agg,
                  normalize_by_num_incoming=bool(rng.integers(2)))
        w, needs_indeg = W.film_weights(L, d_in, D, seed, num_timesteps=T, random_ln=True), True
    elif kind == "gnn-edge-mlp":
        hidden, tgt = int(rng.integers(0, 3)), bool(rng.integers(2))
        kw = dict(state_dim=D, num_timesteps=T, activation_function=act, message_aggregation_function=agg,
                  normalize_by_num_incoming=bool(rng.integers(2)), use_target_state_as_input=tgt, num_edge_hidden_layers=hidden)
        w, needs_indeg = W.edge_mlp_weights(L, d_in, D, hidden, tgt, seed, num_timesteps=T, random_ln=True), True
    elif kind == "rgin":
        eh, ah, tgt = pick(rng, [None, 0, 1, 2]), pick(rng, [None, 0, 1]), bool(rng.integers(2))
        if eh is None:
            d_in, tgt = D, False                                  # no edge MLP: the message keeps the input width
        kw = dict(state_dim=D, num_timesteps=T, activation_function=act, message_aggregation_function=agg,
                  use_target_state_as_input=tgt, num_edge_MLP_hidden_layers=eh, num_aggr_MLP_hidden_layers=ah)
        w, needs_indeg = W.rgin_weights(L, d_in, D, eh, ah, tgt, seed, num_timesteps=T, random_ln=True), False
    else:
        C, cd = int(pick(rng, [1, 2, 4])), int(pick(rng, [2, 4]))
        d_in, full, tie = C * cd, bool(rng.integers(2)), bool(rng.integers(2))
        kw = dict(num_channels=C, channel_dim=cd, num_timesteps=T, use_full_state_for_channel_weights=full, tie_channel_weights=tie,
                  activation_function=act, message_aggregation_function=agg)
        w, needs_indeg = W.rgdcn_weights(L, C, cd, full, tie, seed, stddev=0.3), True
    h = node_states(V, d_in, seed=seed + 1)
    return dict(kind=kind, kw=kw, indeg=needs_indeg), h, adj, indeg, w


@pytest.mark.parametrize("kind", KINDS)
def test_oracle_equals_reference_on_random_cases(kind):
    import builtins
    recorded = ref_records.load()["fuzz"][kind]
    assert len(recorded) == CASES_PER_KIND
    rng = np.random.default_rng(sum(map(ord, kind)))
    worst, ran, none_act = 0.0, 0, 0
    for i in range(CASES_PER_KIND):
        case, h, adj, indeg, w = make_case(kind, rng)
        what = "%s case %d: V=%d edges=%s h=%s %s" % (kind, i, h.shape[0], [len(a) for a in adj], h.shape, case["kw"])
        ref = recorded[i]
        if "raises" in ref:
            no_act = case["kw"].get("activation_function") in (None, "linear")
            if no_act and ((ref["raises"] == "TypeError" and "NoneType" in ref["message"]) or
                           (ref["raises"] == "AssertionError" and "without an activation" in ref["message"])):
                none_act += 1       # get_activation returned None and the layer calls it (e.g. rgcn.py:114, rgin.py:129), or MLP refuses two
                continue            # linear layers (utils/utils.py:105): no reference behaviour; oracle and engine apply the identity (documented)
            # any other combination the REFERENCE rejects must be rejected by the oracle too (same exception type)
            with pytest.raises(getattr(builtins, ref["raises"])):
                R.LAYERS[kind](h, adj, *((indeg,) if case["indeg"] else ()), **case["kw"], weights=w, dtype=np.float64)
            continue
        got = R.LAYERS[kind](h, adj, *((indeg,) if case["indeg"] else ()), **case["kw"], weights=w, dtype=np.float64)
        err = ref_records.summary_err(got, ref)
        assert err <= 1e-12, "%s: %.3e" % (what, err)
        worst, ran = max(worst, err), ran + 1
    assert ran >= CASES_PER_KIND // 2, "%s: only %d of %d random cases ran in the reference" % (kind, ran, CASES_PER_KIND)
    print("%s: %d random cases, worst error %.2e (%d more with activation None / 'linear' crash in the reference)" % (kind, ran, worst, none_act))
