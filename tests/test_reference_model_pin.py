"""SURVEY.md 8f (the scaffold around the hot path): oracle/ref_model.py, checkpoint.py's variable-name sorting and
SparseGraphModel's snapshot loading against the REFERENCE'S OWN model scaffold and task heads.

models/sparse_graph_model.py + models/<x>_model.py + tasks/{ppi,qm9}_task.py are executed unmodified under
tests/tf1_shim.graph_mode (placeholders hand out the feed, so the static graph runs eagerly while the constructor builds it;
only TF kernel semantics are restated).  What comes out -- the variables under the names the reference created them with, the
pickle its own save_model wrote, final node representations, loss / MAE / micro-F1, the "Model has N parameters." count --
is committed as tests/golden/ref_model_<case>.npz and compared here:

* everywhere: snapshot -> load_reference_checkpoint -> sort_variables -> oracle whole model on batching.py's feed == the
  reference's outputs (1e-12); snapshot -> SparseGraphModel.load_reference_weights -> every parameter lands where the
  oracle reads it; parameter counts equal the reference's;
* against runs of the reference recorded in tests/golden/ref_records.json (tests/golden/ref_records.py models): the
  fixtures are current, default_params of every model class, README.md:29's 699257 parameters counted by the reference's
  own loop, the export direction (the reference's scaffold fed with a package model's values, its restore() of a snapshot
  written here) and the train step."""
import importlib
import json
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
for p in (HERE, os.path.join(HERE, "golden")):
    if p not in sys.path:
        sys.path.insert(0, p)

import batcher_cases as BC      # noqa: E402
import model_cases as MC        # noqa: E402
import ref_records              # noqa: E402

checkpoint = importlib.import_module("tf_gnn_samples_b200.checkpoint")
ALL = sorted(MC.CASES)


def fixture(name):
    z = np.load(os.path.join(HERE, "golden", "ref_model_%s.npz" % name))
    snap = checkpoint.load_reference_checkpoint(z["pickle"].tobytes())
    return z, snap


@pytest.fixture(scope="module")
def ppi_dir(tmp_path_factory):
    return BC.write_ppi_dir(str(tmp_path_factory.mktemp("ppi")), "test")


def repo_feed(case, task_params, ppi_dir):
    """The case's minibatch from batching.py (bit-identical to the reference batcher's: test_reference_batcher_pin.py)."""
    if case["task"] == "qm9":
        feeds, L = BC.repo_qm9_feeds(task_params, case["budget"])
    else:
        feeds, L = BC.repo_ppi_feeds(task_params, case["budget"], ppi_dir)
    return feeds[0], L


def rel(a, b):
    return float(np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64)).max() / np.abs(np.asarray(b, np.float64)).max())


def check_metrics(got, want, what):
    assert set(got) == set(want), (what, sorted(got), sorted(want))
    for k, v in want.items():
        tol = 1e-6 if k == "f1_score" else 1e-11              # the reference casts F1 to float32 (utils/utils.py:74)
        assert abs(float(got[k]) - float(v)) <= tol * max(1.0, abs(float(v))), (what, k, float(got[k]), float(v))


@pytest.mark.parametrize("name", ALL)
def test_oracle_whole_model_on_the_reference_snapshot(name, ppi_dir):
    case = MC.CASES[name]
    z, snap = fixture(name)
    assert snap.model_class == json.loads(str(z["meta"]))["model"] and snap.task_class == json.loads(str(z["meta"]))["task"]
    assert sorted(snap.weights) == list(z["variable_names"])
    feed, L = repo_feed(case, snap.task_params, ppi_dir)
    assert L == int(z["num_edge_types"]) and int(feed["num_nodes"]) == int(z["num_nodes"])
    o = MC.run_oracle(case, feed, snap.weights, snap.model_params, snap.task_params, L)
    assert rel(o["final"], z["final"]) <= 1e-12, name
    check_metrics(o["metrics"], json.loads(str(z["metrics"])), name)
    o32 = MC.run_oracle(case, feed, snap.weights, snap.model_params, snap.task_params, L, dtype=np.float32)
    assert o32["final"].dtype == np.float32 and rel(o32["final"], z["final"]) <= 4 * float(z["err32"]) + 1e-6


@pytest.mark.parametrize("name", ALL)
def test_snapshot_loads_into_the_scaffold_by_variable_name(name, ppi_dir):
    """Every parameter of SparseGraphModel receives the value the oracle reads for it (same sorted dictionaries), none is left
    at its initial value, and the parameter count is the one the reference printed."""
    import torch
    scaffold = importlib.import_module("tf_gnn_samples_b200.scaffold")
    case = MC.CASES[name]
    z, snap = fixture(name)
    feed, L = repo_feed(case, snap.task_params, ppi_dir)
    feature_size = feed["initial_node_features"].shape[1]
    kw = dict(num_labels=feed["target_labels"].shape[1]) if case["task"] == "ppi" else dict(task_ids=tuple(snap.task_params["task_ids"]))
    model = scaffold.SparseGraphModel(case["kind"], case["task"], L, feature_size, params=snap.model_params, device="cpu", **kw)
    assert model.num_parameters() == int(z["num_parameters"])
    before = {n: p.detach().clone() for n, p in model.named_parameters()}
    left = model.load_reference_weights(snap.weights)
    assert left == [], left
    o = MC.run_oracle(case, feed, snap.weights, snap.model_params, snap.task_params, L)

    def same(dst, src, path):
        if isinstance(dst, dict):
            for k, v in dst.items():
                if k != "kind" and v is not None:
                    same(v, src[k], path + "." + k)
        elif isinstance(dst, (list, tuple)):
            assert len(dst) == len(src), path
            for i, v in enumerate(dst):
                same(v, src[i], "%s.%d" % (path, i))
        else:
            assert np.array_equal(dst.detach().numpy(), np.asarray(src, np.float32)), path

    for l, w in enumerate(model.layers):
        same(w, o["layers"][l], "gnn_layer_%d" % l)
    if model.projection is not None:
        same(model.projection, o["outside"]["projection"], "projection")
    if case["task"] == "ppi":
        same(model.head, [h for h in o["outside"]["head"] if "bias" in h][-1], "head")
    else:
        for i, t in enumerate(snap.task_params["task_ids"]):
            same(model.head[i], o["outside"]["qm9_heads"][t], "out_layer_task%d" % t)
    untouched = [n for n, p in model.named_parameters() if torch.equal(p, before[n]) and float(p.detach().abs().max()) not in (0.0, 1.0)]
    assert untouched == [], untouched


def test_default_params_of_the_snapshots_are_the_packages():
    """model_params in the reference's pickle = <X>_Model.default_params() + the case's overrides; scaffold.model_default_params
    restates those defaults (keys the loops never read -- max_epochs, patience, lr_for_num_graphs_per_batch -- aside)."""
    scaffold = importlib.import_module("tf_gnn_samples_b200.scaffold")
    for name in ALL:
        case = MC.CASES[name]
        _, snap = fixture(name)
        mine = dict(scaffold.model_default_params(case["kind"]), **case["model_params"])
        for k, v in mine.items():
            assert snap.model_params[k] == v, (name, k, snap.model_params[k], v)
        extra = set(snap.model_params) - set(mine)
        if case["kind"] == "rgdcn":                                # derived in RGDCN_Model.__init__ (rgdcn_model.py:31)
            assert snap.model_params["channel_dim"] == mine["hidden_size"] // mine["num_channels"]
            extra -= {"channel_dim"}
        assert extra <= {"max_epochs", "patience", "lr_for_num_graphs_per_batch"}, name


# ---- against a fresh run of the reference (recorded) ----
@pytest.mark.parametrize("name", ALL)
def test_fixture_equals_the_reference_scaffold_run_here(name, ppi_dir):
    """The committed fixture equals a later, recorded run of the reference's scaffold (digests of the final node states and
    every variable, parameter count, metrics); the oracle on batching.py's feed reproduces the fixture."""
    case = MC.CASES[name]
    z, snap = fixture(name)
    r = ref_records.load()["models"]["runs"][name]
    assert ref_records.sha(z["final"]) == r["final"] and r["num_parameters"] == int(z["num_parameters"])
    assert sorted(r["variables"]) == list(z["variable_names"])
    for k, v in r["variables"].items():
        assert ref_records.sha(np.asarray(snap.weights[k])) == v, k
    check_metrics(r["metrics"], json.loads(str(z["metrics"])), name)
    feed, L = repo_feed(case, snap.task_params, ppi_dir)          # bit-identical to the reference's feed (batcher pin)
    o = MC.run_oracle(case, feed, snap.weights, snap.model_params, snap.task_params, L)
    assert rel(o["final"], z["final"]) <= 1e-12


def test_readme_parameter_count_by_the_references_own_loop():
    """README.md:29 'Model has 699257 parameters' (RGCN on PPI: 50 features, 121 labels, 3 edge types, hidden 256, 3 layers),
    counted by sparse_graph_model.py:153-157 over the variables the reference's scaffold creates -- and by the package."""
    scaffold = importlib.import_module("tf_gnn_samples_b200.scaffold")
    assert ref_records.load()["models"]["readme_num_parameters"] == 699257
    assert scaffold.RGCNPPIModel(device="cpu").num_parameters() == 699257
    params = MC.README_RGCN_PPI["model_params"]
    assert scaffold.SparseGraphModel("rgcn", "ppi", 3, 50, params=params, device="cpu").num_parameters() == 699257


def test_default_params_equal_the_reference_classes():
    scaffold = importlib.import_module("tf_gnn_samples_b200.scaffold")
    recorded = ref_records.load()["models"]["default_params"]
    assert sorted(recorded) == sorted(MC.MODEL_CLASSES)
    for kind, ref in recorded.items():
        mine = scaffold.model_default_params(kind)
        for k, v in mine.items():
            assert ref[k] == ref_records.jsonable(v), (kind, k, ref[k], v)
        assert set(ref) - set(mine) <= {"max_epochs", "patience", "lr_for_num_graphs_per_batch"}, (kind, set(ref) - set(mine))


# ---- the export direction: a model of THIS package handed to the reference ----
# The reference's side of these tests -- its scaffold fed with the exported values, its restore() of a snapshot written here, its
# train step on prescribed gradients -- is recorded by tests/golden/ref_records.py (models) from the same package-side set-up.
EXPORT_CASES = ["rgcn_ppi_scaffold", "film_ppi_scaffold", "rgin_ppi_scaffold", "ggnn_ppi_hidden_is_feature_size",
                "rgcn_qm9", "ggnn_qm9", "rgat_qm9", "edge_mlp_qm9", "rgdcn_qm9"]
RESTORE_CASES = ["rgin_ppi_scaffold", "edge_mlp_qm9", "ggnn_qm9"]
OPTIMIZERS = ["SGD", "RMSProp", "Adam"]
TASK_DEFAULTS = {"qm9": {"add_self_loop_edges": True, "tie_fwd_bkwd_edges": True, "task_ids": [0]},
                 "ppi": {"add_self_loop_edges": True, "tie_fwd_bkwd_edges": False}}


def recorded(section):
    return ref_records.load()["models"][section]


def _package_model(case, feed, L, seed):
    scaffold = importlib.import_module("tf_gnn_samples_b200.scaffold")
    params = dict(scaffold.model_default_params(case["kind"]), **case["model_params"], random_seed=seed)
    task_params = dict({"task_ids": [0]} if case["task"] == "qm9" else {}, **case["task_params"])
    kw = dict(num_labels=feed["target_labels"].shape[1]) if case["task"] == "ppi" else dict(task_ids=tuple(task_params["task_ids"]))
    model = scaffold.SparseGraphModel(case["kind"], case["task"], L, feed["initial_node_features"].shape[1], params=params, device="cpu", **kw)
    import torch
    with torch.no_grad():                                        # zero / one initial values would hide a swapped bias or gamma
        for i, (n, p) in enumerate(sorted(model.named_parameters())):
            if float(p.abs().max()) in (0.0, 1.0):
                p.add_(0.01 * torch.randn(p.shape, generator=torch.Generator().manual_seed(i)))
    return model, task_params


def to_numpy(obj):
    if isinstance(obj, dict):
        return {k: to_numpy(v) for k, v in obj.items()}
    if isinstance(obj, (list, tuple)):
        return [to_numpy(v) for v in obj]
    if obj is None or isinstance(obj, str):
        return obj
    return obj.detach().cpu().numpy()


def export_setup(name, ppi_dir):
    """The seeded package model of an export case, its feed, and to_reference_weights() without the graph counter."""
    case = MC.CASES[name]
    feed, L = repo_feed(case, dict(TASK_DEFAULTS[case["task"]], **case["task_params"]), ppi_dir)
    model, task_params = _package_model(case, feed, L, seed=5)
    named = model.to_reference_weights()
    counter = named.pop("total_num_graphs:0")
    assert counter.dtype == np.int64 and counter.shape == ()
    return case, feed, L, model, task_params, named


@pytest.mark.parametrize("name", EXPORT_CASES)
def test_exported_variables_drive_the_reference_scaffold(name, ppi_dir):
    """SparseGraphModel.to_reference_weights() names every variable the reference's scaffold creates (and nothing else); fed
    with those values the reference's own forward equals the oracle run on the model's weight dictionaries directly."""
    from oracle import ref_model
    case, feed, L, model, task_params, named = export_setup(name, ppi_dir)
    ran = recorded("exported")[name]
    assert ref_records.tree_digest(named) == ran["exported"]                   # the names and values the reference was fed
    assert ref_records.tree_digest(sorted(named)) == ran["used"]               # it read every one of them ...
    assert ref_records.tree_digest(sorted(set(named) | {"total_num_graphs:0"})) == ran["variables"]   # ... and created no other
    assert ran["num_parameters"] == model.num_parameters()
    feats = np.asarray(feed["initial_node_features"], np.float32).astype(np.float64)
    adj = MC.adjacency_of(feed, L)
    indeg = np.asarray(feed["type_to_num_incoming_edges"], np.float32).astype(np.float64)
    final = ref_model.node_representations(model.kind, feats, adj, indeg, model.params, to_numpy(model.projection), to_numpy(model.layers))
    assert ref_records.summary_err(final, ran["final"]) <= 1e-12
    if case["task"] == "ppi":
        head = to_numpy(model.head)
        want = ref_model.ppi_metrics(final @ head["kernel"].astype(np.float64) + head["bias"], feed["target_labels"])
    else:
        outs = ref_model.qm9_outputs(final, feats, feed["graph_nodes_list"], int(feed["num_graphs"]), to_numpy(model.head))
        want = ref_model.qm9_metrics(outs, np.asarray(feed["target_values"]).astype(np.float32), task_params["task_ids"])
    check_metrics(want, ran["metrics"], name)


def restore_setup(name, ppi_dir, directory):
    """A seeded package model of a restore case, saved as a reference snapshot under ``directory``."""
    case = MC.CASES[name]
    task_params = dict(TASK_DEFAULTS[case["task"]], out_layer_dropout_keep_prob=1.0, **case["task_params"])
    feed, L = repo_feed(case, task_params, ppi_dir)
    model, _ = _package_model(case, feed, L, seed=9)
    F = feed["initial_node_features"].shape[1]
    metadata = {"params": task_params, "num_edge_types": L}
    metadata.update({"annotation_size": F} if case["task"] == "qm9" else
                    {"initial_node_feature_size": F, "num_labels": feed["target_labels"].shape[1]})
    path = os.path.join(directory, "snapshot.pickle")
    model.save_reference_snapshot(path, task_params, metadata)
    return case, feed, L, model, path


@pytest.mark.parametrize("name", RESTORE_CASES)
def test_the_references_restore_accepts_a_snapshot_written_here(name, ppi_dir, tmp_path):
    """utils/model_utils.py:58-77 restore(): class names resolve, the task restores from the metadata, the model builds, and
    load_weights finds a saved value for EVERY variable and uses EVERY saved value (it prints a line otherwise)."""
    import pickle
    case, feed, L, model, path = restore_setup(name, ppi_dir, str(tmp_path))
    ran = recorded("restored")[name]
    with open(path, "rb") as f:
        assert ref_records.tree_digest(pickle.load(f)) == ran["snapshot"]      # the file the reference restored
    out = ran["printed"]
    assert "Loaded model from snapshot" in out
    assert "Freshly initializing" not in out and "not used by model" not in out, out
    assert ran["model_class"] == MC.MODEL_CLASSES[case["kind"]] and ran["num_edge_types"] == L
    want = model.to_reference_weights()
    assert sorted(ran["variables"]) == sorted(want)
    for k, v in ran["variables"].items():
        assert ref_records.sha(np.asarray(want[k], np.float64)) == v, k


# ---- the train step (sparse_graph_model.py:226-260) ----
def train_step_case(optimizer):
    hp = {"optimizer": optimizer, "learning_rate": 0.003, "learning_rate_decay": 0.9, "momentum": 0.7, "clamp_gradient_norm": 0.5}
    return dict(MC.CASES["film_ppi_scaffold"], model_params=dict(MC.CASES["film_ppi_scaffold"]["model_params"], **hp))


def gradient_prescriber():
    """The gradient the train step receives for each variable, drawn in the order the variables are asked for."""
    rng = np.random.default_rng(8)
    prescribed = {}

    def gradient_hook(name, shape):
        if name.endswith("gnn_layer_1/LayerNorm/beta:0"):
            prescribed[name] = None                               # a variable the loss does not depend on
        else:                                                    # norms on both sides of the clamp
            prescribed[name] = rng.standard_normal(shape) * (0.5 / np.sqrt(max(1, int(np.prod(shape))))) * rng.choice([0.2, 3.0])
        return prescribed[name]
    return gradient_hook, prescribed


@pytest.mark.parametrize("optimizer", OPTIMIZERS)
def test_train_step_construction_and_per_tensor_clipping(optimizer, ppi_dir):
    """__make_train_step run by the reference with PRESCRIBED gradients: which optimizer it builds with which hyper-parameters,
    that the differentiated quantity is task_metrics['loss'], and that every gradient is clipped BY ITS OWN norm (tf.clip_by_norm,
    not a global norm), None gradients passing through -- against scaffold.make_optimizer / clip_gradients_ on the same numbers.
    The reference's clipped gradients are recorded as the factor it scaled each prescribed gradient by."""
    import torch
    scaffold = importlib.import_module("tf_gnn_samples_b200.scaffold")
    tfo = importlib.import_module("tf_gnn_samples_b200.tf_optimizers")
    case = train_step_case(optimizer)
    r = recorded("train_step")[optimizer]
    gradient_hook, prescribed = gradient_prescriber()
    for name, shape in r["gradient_order"]:                      # the order the reference asked for them
        gradient_hook(name, tuple(shape))
    assert r["loss_is_task_loss"]
    (cls_name, kwargs), = r["optimizers"]
    feed, L = repo_feed(case, {"add_self_loop_edges": True, "tie_fwd_bkwd_edges": True}, ppi_dir)
    model = scaffold.SparseGraphModel(case["kind"], "ppi", L, feed["initial_node_features"].shape[1], params=r["params"],
                                      num_labels=feed["target_labels"].shape[1], device="cpu")
    opt = model.make_optimizer()
    if optimizer == "SGD":
        assert cls_name == "GradientDescentOptimizer" and kwargs == {"learning_rate": 0.003}
        assert isinstance(opt, torch.optim.SGD) and opt.defaults["lr"] == 0.003 and opt.defaults["momentum"] == 0
    elif optimizer == "RMSProp":
        assert cls_name == "RMSPropOptimizer" and kwargs == {"learning_rate": 0.003, "decay": 0.9, "momentum": 0.7}
        assert isinstance(opt, tfo.TF1RMSProp)
        assert (opt.defaults["lr"], opt.defaults["decay"], opt.defaults["momentum"], opt.defaults["epsilon"]) == (0.003, 0.9, 0.7, 1e-10)
    else:
        assert cls_name == "AdamOptimizer" and kwargs == {"learning_rate": 0.003}
        assert isinstance(opt, tfo.TF1Adam) and opt.defaults["lr"] == 0.003 and opt.defaults["epsilon"] == 1e-8
    # the package's clipping on the same gradients, parameters matched to variables by the exported names
    checkpoint_mod = importlib.import_module("tf_gnn_samples_b200.checkpoint")
    named = checkpoint_mod.model_to_variables(model.projection, model.layers, "ppi", model.head)
    assert set(named) == set(prescribed)
    for name, p in named.items():
        p.grad = None if prescribed[name] is None else torch.as_tensor(prescribed[name], dtype=torch.float64).to(p.dtype)
    pre = {n: None if p.grad is None else float(p.grad.norm()) for n, p in named.items()}
    assert min(v for v in pre.values() if v is not None) < 0.5 < max(v for v in pre.values() if v is not None)
    model.clip_gradients_()
    applied = {n: None if s is None else s * prescribed[n] for n, s in r["applied_scale"].items()}
    assert set(applied) == set(named)
    for name, p in named.items():
        if prescribed[name] is None:
            assert applied[name] is None and p.grad is None
        else:
            assert np.allclose(p.grad.numpy(), applied[name], rtol=2e-6, atol=1e-9), name
            assert float(np.linalg.norm(applied[name])) <= 0.5 * (1 + 1e-12)


def lr_case():
    hp = {"optimizer": "RMSProp", "learning_rate": 0.003, "lr_for_num_graphs_per_batch": 30}
    return dict(MC.CASES["rgcn_qm9"], model_params=dict(MC.CASES["rgcn_qm9"]["model_params"], **hp))


def test_learning_rate_normalised_per_graph_count():
    """lr_for_num_graphs_per_batch = n (sparse_graph_model.py:230-238): the reference hands the optimizer
    learning_rate * num_graphs / n; set_learning_rate_ puts the same number into the torch optimizer before the step."""
    scaffold = importlib.import_module("tf_gnn_samples_b200.scaffold")
    r = recorded("lr_per_graph_count")
    (cls_name, kwargs), = r["optimizers"]
    G = r["num_graphs"]
    assert cls_name == "RMSPropOptimizer" and G not in (0, 30)
    model = scaffold.SparseGraphModel("rgcn", "qm9", r["num_edge_types"], 15, params=r["params"], task_ids=(0, 4), device="cpu")
    opt = model.make_optimizer()
    assert opt.param_groups[0]["lr"] == 0.003
    model.set_learning_rate_(opt, G)
    assert abs(opt.param_groups[0]["lr"] - float(kwargs["learning_rate"])) <= 1e-6 * float(kwargs["learning_rate"])
    assert abs(opt.param_groups[0]["lr"] - 0.003 * G / 30) <= 1e-9
    with pytest.raises(ValueError):
        model.set_learning_rate_(opt, None)
    plain = scaffold.SparseGraphModel("rgcn", "qm9", 5, 15, params={"hidden_size": 16, "graph_num_layers": 1}, device="cpu")
    o2 = plain.make_optimizer()
    plain.set_learning_rate_(o2, None)                           # not configured: untouched, num_graphs not needed
    assert o2.param_groups[0]["lr"] == plain.params["learning_rate"]
