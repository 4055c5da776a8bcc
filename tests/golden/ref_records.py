"""What the reference computed for the tests that compare the package with the reference's own code, stored so that those
tests run without a reference checkout.

    python tests/golden/ref_records.py [section ...]   (needs a checkout of microsoft/tf-gnn-samples at tf1_shim.REFERENCE_ROOT)

executes the reference through tests/tf1_shim exactly as the tests used to, and writes tests/golden/ref_records.json:
exception types and messages, names, parameter counts, default parameters, log lines, and for arrays either a (96-bit)
SHA-256 digest of their exact values (where the tests compared bit for bit) or a few seeded random projections (where they compared to a
tolerance and the arrays would be too large to store).  The tests import the helpers below to reduce their own results
the same way."""
import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
PATH = os.path.join(HERE, "ref_records.json")
for _p in (HERE, os.path.dirname(HERE), os.path.dirname(os.path.dirname(HERE))):
    if _p not in sys.path:
        sys.path.insert(0, _p)


def load():
    with open(PATH) as f:
        return json.load(f)


def sha(arr):
    """Digest of an array's values, shape and kind: int arrays as int64, float arrays as float64 (exact widening)."""
    a = np.asarray(arr)
    a = a.astype(np.float64) if a.dtype.kind == "f" else a.astype(np.int64) if a.dtype.kind in "iub" else a
    h = hashlib.sha256(repr((a.dtype.str, a.shape)).encode())
    h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()[:24]


def feed_digests(feed):
    """{placeholder name: sha} of one minibatch feed as its placeholders receive it: adjacency lists as [E, 2] int (an empty
    list may come as shape (0,)), ids and counts as int, everything else after the float32 cast of the placeholder
    (tasks/sparse_graph_task.py:139-146).  The dropout keep-probability is not part of the batch."""
    out = {}
    for k, v in feed.items():
        v = np.asarray(v)
        if k.startswith("adjacency_"):
            out[k] = sha(v.reshape(-1, 2).astype(np.int64))
        elif k in ("graph_nodes_list", "num_graphs", "num_nodes", "num_edges"):
            out[k] = sha(v.astype(np.int64))
        elif k != "out_layer_dropout_keep_prob":
            out[k] = sha(v.astype(np.float32))
    return out


def summary(out, seed=20261017, samples=8):
    """Max |x|, three seeded bilinear forms u^T X w (u, w standard normal) and ``samples`` seeded elements of a 2-D float
    array (float64)."""
    x = np.asarray(out, np.float64).reshape(np.shape(out)[0], -1)
    rng = np.random.default_rng(seed)
    u, w = rng.standard_normal((3, x.shape[0])), rng.standard_normal((3, x.shape[1]))
    idx = rng.integers(0, x.size, samples)
    return {"shape": list(np.shape(out)), "maxabs": float(np.abs(x).max()) if x.size else 0.0,
            "forms": [float(u[i] @ x @ w[i]) for i in range(3)], "sample": [float(v) for v in x.reshape(-1)[idx]]}


def summary_err(got, want):
    """Error of ``got`` against a stored summary, relative to the stored max |x|.  For an error matrix E, u^T E w with
    independent standard-normal u, w has mean 0 and variance ||E||_F^2 >= max|E|^2, so each form estimates the Frobenius norm
    of the error -- never smaller on average than the max-norm error, and a single element off by d moves it by |u_i w_j| d;
    three independent forms make a miss of a large error unlikely.  The samples are element-wise errors."""
    s = summary(got)
    assert s["shape"] == want["shape"], (s["shape"], want["shape"])
    scale = max(want["maxabs"], 1e-30)
    errs = [abs(s["maxabs"] - want["maxabs"])]
    errs += [abs(a - b) for a, b in zip(s["forms"], want["forms"])]
    errs += [abs(a - b) for a, b in zip(s["sample"], want["sample"])]
    return max(errs) / scale


def outcome(fn, *args):
    try:
        return ["ok", fn(*args)]
    except Exception as e:                                   # noqa: BLE001 -- the exception IS the behaviour recorded
        return [type(e).__name__, str(e)]


def tree_digest(obj):
    """Digest of a nested structure of dicts, lists and arrays (a pickled snapshot): arrays by sha, everything else by repr."""
    def canon(o):
        if isinstance(o, dict):
            return [[repr(k), canon(v)] for k, v in sorted(o.items(), key=lambda kv: repr(kv[0]))]
        if isinstance(o, (list, tuple)):
            return [canon(v) for v in o]
        if isinstance(o, (np.ndarray, np.generic)):
            return sha(o)
        return repr(o)
    return hashlib.sha256(json.dumps(canon(obj)).encode()).hexdigest()[:24]


def jsonable(v):
    return json.loads(json.dumps(v, default=lambda o: o.item() if hasattr(o, "item") else repr(o)))


# ------------------------------------------------------------------------------------------------------------------
# recording (runs the reference)
# ------------------------------------------------------------------------------------------------------------------
def record_utils():
    import inspect
    import tf1_shim
    import test_reference_utils_pin as U
    rec = {}
    x = np.linspace(-3, 3, 25)
    with tf1_shim.installed(dtype=np.float64) as session:
        import utils as ref_utils
        tf = session.tf
        segment_fns = {tf.unsorted_segment_sum: "sum", tf.unsorted_segment_max: "max", tf.unsorted_segment_mean: "mean",
                       tf.unsorted_segment_sqrt_n: "sqrt_n"}
        mu = tf1_shim.import_reference_model_utils()
        acts = []
        for name in U.ACTIVATION_NAMES:
            r = outcome(ref_utils.get_activation, name)
            acts.append(r if r[0] != "ok" else ["ok", [float(v) for v in (x if r[1] is None else r[1](x))]])
        rec["activation"] = acts
        rec["aggregation"] = [r if r[0] != "ok" else ["ok", segment_fns[r[1]]]
                              for r in (outcome(ref_utils.get_aggregation_function, n) for n in U.AGGREGATION_NAMES)]
        cells = []
        for name in U.CELL_NAMES:
            r = outcome(ref_utils.get_gated_unit, 8, name, "tanh")
            if r[0] == "ok":
                call = outcome(r[1], np.zeros((2, 8)), [np.zeros((2, 8))])
                r = ["ok", type(r[1]).__name__, call[0]]
            cells.append(r)
        rec["gated_unit"] = cells
        rec["gated_unit_gru_swish"] = outcome(ref_utils.get_gated_unit, 8, "gru", "swish")
        models = []
        for name in U.MODEL_NAMES:
            r = outcome(mu.name_to_model_class, name)
            if r[0] == "ok":
                cls, extra = r[1]
                want = cls.default_params()
                want.update(extra)
                r = ["ok", cls.__name__, jsonable(want)]
            models.append(r)
        rec["model_names"] = models
        import gnns as ref_gnns
        rec["layer_signatures"] = {n: [[p.name, repr(p.default)] for p in inspect.signature(getattr(ref_gnns, n)).parameters.values()]
                                   for n in dir(ref_gnns) if n.startswith("sparse_") and n.endswith("_layer")}
    return rec


def record_fuzz():
    import test_reference_fuzz as F
    import make_ref_fixtures as MRF
    rec = {}
    for kind in F.KINDS:
        rng = np.random.default_rng(sum(map(ord, kind)))
        cases = []
        for _ in range(F.CASES_PER_KIND):
            case, h, adj, indeg, w = F.make_case(kind, rng)
            try:
                ref, _ = MRF.run_reference(case, h, adj, indeg, w, np.float64)
            except Exception as exc:                          # noqa: BLE001
                cases.append({"raises": type(exc).__name__, "message": str(exc)})
                continue
            cases.append(summary(ref))
        rec[kind] = cases
    return rec


def record_layer_fixtures():
    import make_ref_fixtures as MRF
    import ref_cases as RC
    import test_reference_pin as P
    rec = {}
    for name in P.REEXECUTED:
        case = RC.CASES[name]
        h, adj, indeg = case["graph"]()
        out64, created = MRF.run_reference(case, h, adj, indeg, case["weights"](), np.float64)
        rec[name] = {"created": sorted(created), "out": summary(out64)}
        if case.get("big"):                    # what the fixture commits of a big case, in the fixture's own terms
            rec[name]["fixture_summary"] = {k: sha(v) for k, v in RC.summarize(out64).items() if k != "rows"}
    return rec


def record_batchers():
    import tempfile
    import batcher_cases as BC
    import tf1_shim
    rec = {"qm9": {}, "ppi": {}}
    for case, (params, budget) in sorted(BC.QM9_CASES.items()):
        want, L = BC.reference_qm9_feeds(params, budget)
        rec["qm9"][case] = {"num_edge_types": L, "feeds": [feed_digests(f) for f in want]}
    with tempfile.TemporaryDirectory() as tmp:
        d = BC.write_ppi_dir(tmp, "test")
        for case, (params, budget) in sorted(BC.PPI_CASES.items()):
            want, L = BC.reference_ppi_feeds(params, budget, d)
            rec["ppi"][case] = {"num_edge_types": L, "feeds": [feed_digests(f) for f in want]}
    rec["qm9_untied"] = {case: outcome(BC.reference_qm9_feeds, params, budget)[0]
                         for case, (params, budget) in sorted(BC.QM9_REFERENCE_RAISES.items())}
    with tempfile.TemporaryDirectory() as tmp:
        rec["ppi_linkless"] = outcome(BC.reference_ppi_feeds, {}, 10 ** 6, BC.write_ppi_dir(tmp, "test", linkless_graph=2))[0]
    want, L = BC.reference_qm9_feeds({}, 10 ** 9, path=os.path.join(tf1_shim.REFERENCE_ROOT, "data", "qm9", "valid.jsonl.gz"))
    rec["qm9_full_valid"] = {"num_edge_types": L, "num_minibatches": len(want),
                             "counts": [int(want[0][k]) for k in ("num_graphs", "num_nodes", "num_edges")],
                             "digests": {k: v for k, v in feed_digests(want[0]).items()
                                         if k.startswith("adjacency_") or k in ("graph_nodes_list", "type_to_num_incoming_edges")}}
    return rec


def record_models():
    import model_cases as MC
    import tf1_shim
    rec = {"runs": {}}
    for name in sorted(MC.CASES):
        r = MC.run_reference(MC.CASES[name], np.float64)
        rec["runs"][name] = {"final": sha(r["final"]), "num_parameters": r["num_parameters"],
                             "variables": {k: sha(v) for k, v in r["variables"].items()},
                             "metrics": {k: float(v) for k, v in r["metrics"].items()}}
    readme = dict(kind="rgcn", task="ppi", model_params=MC.README_RGCN_PPI["model_params"], task_params={}, budget=10 ** 6)
    rec["readme_num_parameters"] = MC.run_reference(readme, np.float32, ppi_kw=dict(feature_dim=50, num_labels=121))["num_parameters"]
    with tf1_shim.installed():
        tf1_shim.import_reference_task("sparse_graph_task")
        import models
        rec["default_params"] = {kind: jsonable(getattr(models, cls).default_params()) for kind, cls in MC.MODEL_CLASSES.items()}
    rec.update(_record_model_io())
    return rec


def _record_model_io():
    """The reference's side of the export / restore / train-step tests, from the tests' own package-side set-up."""
    import contextlib
    import io
    import pickle
    import tempfile
    import batcher_cases as BC
    import model_cases as MC
    import tf1_shim
    import test_reference_model_pin as P
    from tf1_shim import variables as TV
    rec = {"exported": {}, "restored": {}, "train_step": {}}
    with tempfile.TemporaryDirectory() as tmp:
        ppi_dir = BC.write_ppi_dir(os.path.join(tmp, "ppi"), "test")
        for name in P.EXPORT_CASES:
            case, _, _, _, _, named = P.export_setup(name, ppi_dir)
            provider = TV.provider_from(named)
            r = MC.run_reference(case, np.float64, provider=provider)
            rec["exported"][name] = {"exported": tree_digest(named), "used": tree_digest(sorted(provider.used)),
                                     "variables": tree_digest(sorted(r["variables"])), "num_parameters": r["num_parameters"],
                                     "final": summary(r["final"]), "metrics": {k: float(v) for k, v in r["metrics"].items()}}
        for name in P.RESTORE_CASES:
            d = os.path.join(tmp, "restore_" + name)
            os.makedirs(d)
            case, feed, _, _, path = P.restore_setup(name, ppi_dir, d)
            with open(path, "rb") as f:
                snapshot = tree_digest(pickle.load(f))
            printed = io.StringIO()
            with tf1_shim.installed(dtype=np.float32) as session, contextlib.redirect_stdout(printed):
                session.feeds = dict(feed, out_layer_dropout_keep_prob=1.0)
                mu = tf1_shim.import_reference_model_utils()
                restored = mu.restore(path, d, run_id="restored")
                rec["restored"][name] = {"snapshot": snapshot, "printed": printed.getvalue().replace(d, "<DIR>"),
                                         "model_class": type(restored).__name__, "num_edge_types": restored.task.num_edge_types,
                                         "variables": {k: sha(np.asarray(v, np.float64)) for k, v in session.variables.items()}}
    for optimizer in P.OPTIMIZERS:
        gradient_hook, prescribed = P.gradient_prescriber()
        order = []

        def hook(name, shape):
            order.append([name, [int(n) for n in shape]])
            return gradient_hook(name, shape)
        r = MC.run_reference(P.train_step_case(optimizer), np.float64, gradient_hook=hook)
        scale = {}
        for g, n in r["applied"]:
            if g is None:
                scale[n] = None
                continue
            p = prescribed[n]
            scale[n] = float(np.vdot(g, p) / np.vdot(p, p))
            assert np.allclose(g, scale[n] * p, rtol=1e-13, atol=0), n      # tf.clip_by_norm scales each tensor as a whole
        rec["train_step"][optimizer] = {"gradient_order": order, "loss_is_task_loss": bool(r["loss_is_task_loss"]),
                                        "optimizers": jsonable(r["optimizers"]), "params": jsonable(r["params"]),
                                        "applied_scale": scale}
    r = MC.run_reference(P.lr_case(), np.float32)
    rec["lr_per_graph_count"] = {"optimizers": jsonable(r["optimizers"]), "num_graphs": int(r["feed"]["num_graphs"]),
                                 "params": jsonable(r["params"]), "num_edge_types": r["num_edge_types"]}
    return rec


def _reference_loop(task_name, data_dir, task_params, model_params, max_nodes, test_path):
    import tf1_shim
    import types
    import batcher_cases as BC
    from test_reference_training_pin import scripted, make_counter_clock
    calls = []
    with tf1_shim.installed(dtype=np.float32) as session:
        from dpu_utils.utils import RichPath
        sgt = tf1_shim.import_reference_task("sparse_graph_task")
        mod = tf1_shim.import_reference_task(task_name + "_task")
        cls = mod.QM9_Task if task_name == "qm9" else mod.PPI_Task
        params = cls.default_params()
        params.update(task_params)
        task = cls(params)
        task.load_data(RichPath.create(data_dir))
        target = "target_values" if task_name == "qm9" else "target_labels"
        names = ["initial_node_features", "type_to_num_incoming_edges", "graph_nodes_list", target, "out_layer_dropout_keep_prob"]
        feed = BC._feeds_of(task, list(task._loaded_data[sgt.DataFold.VALIDATION]), sgt.DataFold.VALIDATION, names, max_nodes)[0]
        session.feeds = feed                                       # only to BUILD the model; the loop's results are scripted
        import models
        import models.sparse_graph_model as sgm
        mparams = models.GGNN_Model.default_params()
        mparams.update(model_params)
        model = models.GGNN_Model(mparams, task, "run", data_dir)
        ph = model._Sparse_Graph_Model__placeholders
        state = {"epoch": 1, "fold": None, "step": 0}

        def hook(fetches, feed_dict):
            if not isinstance(fetches, dict) or "task_metrics" not in fetches:       # save_model's variable fetch
                return {k: v.value() for k, v in fetches.items()}
            fold = "train" if "train_step" in fetches else "valid"
            if state["epoch"] == 99:
                fold = "test"
            if fold != state["fold"]:
                if fold == "train" and state["fold"] == "valid":
                    state["epoch"] += 1
                state["fold"], state["step"] = fold, 0
            g = int(feed_dict[ph["num_graphs"]])
            calls.append({"fold": fold, "epoch": state["epoch"], "num_graphs": g,
                          "num_nodes": int(np.asarray(feed_dict[ph["initial_node_features"]]).shape[0]),
                          "keep_prob_fed": ph["graph_layer_input_dropout_keep_prob"] in feed_dict,
                          "first_feature_row": np.asarray(feed_dict[ph["initial_node_features"]])[0].astype(np.float32)})
            out = {"task_metrics": scripted(task_name, fold, state["epoch"], state["step"], g, params.get("task_ids", [0]))}
            state["step"] += 1
            return out

        session.run_hook = hook
        sgm.time = types.SimpleNamespace(time=make_counter_clock())   # the module's clock; the source file is untouched
        try:
            model.train(quiet=True)
            if test_path is not None:                            # Sparse_Graph_Model.test (:373-385) on a held-out file / fold
                state.update(epoch=99, fold=None, step=0)
                model.test(RichPath.create(test_path), quiet=True)
        finally:
            import time as real_time
            sgm.time = real_time
        with open(model.log_file) as f:
            lines = f.read().splitlines()
        return lines, calls, model.best_model_file, os.path.exists(model.best_model_file)


def record_training():
    import tempfile
    import test_reference_training_pin as T
    rec = {}
    model_params = {"hidden_size": 16, "graph_num_layers": 1, "patience": T.PATIENCE, "random_seed": T.SEED}
    for task in ("qm9", "ppi"):
        with tempfile.TemporaryDirectory() as d:
            if task == "qm9":
                _, _, test_path = T.write_qm9_data(d)
                lines, calls, best, saved = _reference_loop("qm9", d, {"task_ids": [0, 4]}, dict(model_params, max_nodes_in_batch=T.MAX_NODES),
                                                            T.MAX_NODES, test_path)
            else:
                T.write_ppi_data(d)
                lines, calls, best, saved = _reference_loop("ppi", d, {}, dict(model_params, max_nodes_in_batch=120), 120, d)
            for c in calls:
                c["first_feature_row"] = sha(c["first_feature_row"])
            rec[task] = {"lines": [line.replace(d, "<DIR>") for line in lines], "calls": calls,
                         "best_model_file": os.path.relpath(best, d), "saved": saved}
    return rec


SECTIONS = {"utils": record_utils, "fuzz": record_fuzz, "layer_fixtures": record_layer_fixtures, "batchers": record_batchers,
            "models": record_models, "training": record_training}


if __name__ == "__main__":
    import warnings
    warnings.simplefilter("ignore", SyntaxWarning)
    rec = load() if os.path.exists(PATH) else {}
    for name in sys.argv[1:] or SECTIONS:
        rec[name] = SECTIONS[name]()
        print("recorded", name, file=sys.stderr)
        with open(PATH, "w") as f:
            json.dump(rec, f, indent=0, sort_keys=True, separators=(",", ":"))
            f.write("\n")
