"""training.py's epoch loop against the REFERENCE's own Sparse_Graph_Model.train / __run_epoch (models/sparse_graph_model.py:
263-371) and the tasks' summaries (tasks/ppi_task.py:258-264, tasks/qm9_task.py:263-282).

The reference's loop runs unmodified under tests/tf1_shim.graph_mode: its task loads real data (QM9 molecules / a dgl-layout
PPI fold, train + valid), its batcher makes the minibatches, ``sess.run`` is SCRIPTED (session.run_hook returns a prescribed
metric dictionary per batch and records the feed_dict the loop assembled), the clock is a counter.  training.train gets the
same data through batching.py, a stub model producing the same scripted metrics and the same clock -- and must write the
same log, line for line: epoch headers, Train / Valid lines with loss, MAE / error ratios or micro-F1, graphs / nodes /
edges per second, save-best lines, early stopping after ``patience`` epochs, the final summary.  The reference's log and the
minibatches its loop fed are recorded in tests/golden/ref_records.json (tests/golden/ref_records.py training), with the
data directory written as <DIR>."""
import gzip
import importlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
for p in (HERE, os.path.join(HERE, "golden")):
    if p not in sys.path:
        sys.path.insert(0, p)

import batcher_cases as BC      # noqa: E402
import ref_records              # noqa: E402

batching = importlib.import_module("tf_gnn_samples_b200.batching")
training = importlib.import_module("tf_gnn_samples_b200.training")

PATIENCE, MAX_NODES, SEED = 2, 700, 4


def scripted(task, fold, epoch, step, num_graphs, task_ids):
    """Metrics of batch ``step`` of ``fold`` in ``epoch``: validation improves for three epochs, then gets worse."""
    if fold == "test":
        quality = 0.52
    else:
        quality = [1.0, 0.7, 0.55, 0.6, 0.65, 0.5, 0.4][min(epoch - 1, 6)] if fold == "valid" else 1.0 / epoch
    loss = quality * (1.0 + 0.01 * step)
    m = {"loss": loss, "total_loss": loss * num_graphs}
    if task == "qm9":
        for t in task_ids:
            m["abs_err_task%d" % t] = quality * num_graphs * (0.1 + 0.01 * t)
    else:
        m["f1_score"] = np.float32(1.0 - 0.5 * quality + 0.001 * step)
    return m


def make_counter_clock():
    state = {"t": 0.0}

    def clock():
        state["t"] += 1.0
        return state["t"]
    return clock


def write_qm9_folds(d):
    recs = batching.load_qm9_jsonl(BC.QM9_SUBSET)
    for name, part in (("train", recs[:150]), ("valid", recs[150:])):
        with gzip.open(os.path.join(d, name + ".jsonl.gz"), "wt") as f:
            for r in part:
                f.write(json.dumps(r) + "\n")
    return recs[:150], recs[150:]


class ScriptedModel:
    """The scaffold interface training.run_epoch drives, answering with the scripted metrics."""

    def __init__(self, task, task_ids):
        self.task, self.task_ids, self.epoch, self.fold, self.step, self.calls, self.testing = task, task_ids, 1, None, 0, [], False

    def _next(self, fold, num_graphs):
        if fold != self.fold:
            if fold == "train" and self.fold == "valid":
                self.epoch += 1
            self.fold, self.step = fold, 0
        m = scripted(self.task, fold, self.epoch, self.step, num_graphs, self.task_ids)
        self.step += 1
        return m

    def train_step_async(self, optimizer, tb, *rest):
        self.calls.append({"fold": "train", "epoch": self.epoch if self.fold != "valid" else self.epoch + 1,
                           "num_graphs": tb.batch.num_graphs, "num_nodes": tb.batch.num_nodes,
                           "first_feature_row": tb.batch.node_features[0]})
        return self._next("train", tb.batch.num_graphs)

    def eval(self):
        return self

    def __call__(self, tb, *rest):
        return tb

    def task_metrics(self, tb, targets):
        fold = "test" if self.testing else "valid"
        self.calls.append({"fold": fold, "epoch": 99 if self.testing else self.epoch, "num_graphs": tb.batch.num_graphs,
                           "num_nodes": tb.batch.num_nodes, "first_feature_row": tb.batch.node_features[0]})
        return self._next(fold, tb.batch.num_graphs)


def run_package_loop(task, train_samples, valid_samples, task_ids, best_model_file, max_nodes=MAX_NODES, test_samples=None,
                     test_description=""):
    def batches(samples, shuffle):
        def make():
            if shuffle:
                np.random.shuffle(samples)                       # DataFold.TRAIN: np.random.shuffle(data) (qm9_task.py:207, ppi_task.py:204)
            return [training.TaskBatch(b, np.zeros(0)) for b, _ in batching.minibatches(samples, max_nodes)]
        return make

    np.random.seed(SEED)                                         # Sparse_Graph_Model.__init__ seeds numpy with random_seed (:68)
    model, lines, saves = ScriptedModel(task, task_ids), [], []
    res = training.train(model, None, task, batches(train_samples, True), batches(valid_samples, False),
                         to_device=lambda tb: (tb, None, None, None), max_epochs=10000, patience=PATIENCE, log=lines.append,
                         save_best=lambda: saves.append(model.epoch), best_model_file=best_model_file, task_ids=task_ids,
                         clock=make_counter_clock())
    if test_samples is not None:
        model.testing = True
        training.test(model, task, batches(test_samples, False)(), to_device=lambda tb: (tb, None, None, None),
                      data_description=test_description, log=lines.append, task_ids=task_ids, clock=make_counter_clock())
    return lines, model.calls, saves, res


def write_qm9_data(d):
    """150 training and 50 validation molecules, and a held-out file of 80 of them."""
    train_recs, valid_recs = write_qm9_folds(d)
    test_file = os.path.join(d, "heldout.jsonl.gz")
    with gzip.open(test_file, "wt") as f:
        for r in (train_recs + valid_recs)[40:120]:
            f.write(json.dumps(r) + "\n")
    return train_recs, valid_recs, test_file


def write_ppi_data(d):
    BC.write_ppi_dir(d, "train", seed=1, num_graphs=9)
    BC.write_ppi_dir(d, "valid", seed=2, num_graphs=4)
    BC.write_ppi_dir(d, "test", seed=3, num_graphs=3)


def recorded_reference_loop(task, data_dir):
    """The reference's log lines, the minibatches its loop fed and its best-model file, for data written to ``data_dir``."""
    r = ref_records.load()["training"][task]
    assert r["saved"]
    return ([line.replace("<DIR>", data_dir) for line in r["lines"]], r["calls"],
            os.path.join(data_dir, r["best_model_file"]))


def compare(ref_lines, ref_calls, pkg_lines, pkg_calls):
    assert ref_lines[0].startswith("Model has ") and ref_lines[1:] == pkg_lines, "\n".join(
        "%s\n%s" % (a, b) for a, b in zip(ref_lines[1:], pkg_lines) if a != b)
    assert len(ref_calls) == len(pkg_calls)
    for a, b in zip(ref_calls, pkg_calls):                        # the same minibatches in the same (shuffled) order
        assert (a["fold"], a["epoch"], a["num_graphs"], a["num_nodes"]) == (b["fold"], b["epoch"], b["num_graphs"], b["num_nodes"])
        assert a["first_feature_row"] == ref_records.sha(np.asarray(b["first_feature_row"], np.float32))
        assert a["keep_prob_fed"] == (a["fold"] == "train")       # dropout keep-prob only fed while training (:277-279)
    assert {c["fold"] for c in ref_calls} == {"train", "valid", "test"}


def test_qm9_epoch_loop_writes_the_references_log(tmp_path):
    train_recs, valid_recs, test_file = write_qm9_data(str(tmp_path))
    task_ids = [0, 4]
    ref_lines, ref_calls, best_file = recorded_reference_loop("qm9", str(tmp_path))
    L = batching.qm9_num_edge_types(train_recs + valid_recs)
    samples = lambda recs: [batching.qm9_graph_to_sample(r, L) for r in recs]
    held_out = samples(batching.load_qm9_jsonl(test_file))
    pkg_lines, pkg_calls, saves, res = run_package_loop("qm9", samples(train_recs), samples(valid_recs), task_ids, best_file,
                                                        test_samples=held_out, test_description=test_file)
    compare(ref_lines, ref_calls, pkg_lines, pkg_calls)
    assert saves == [1, 2, 3] and res["best_epoch"] == 3
    assert pkg_lines[-5] == "Stopping training after %d epochs without improvement on validation loss." % PATIENCE
    assert pkg_lines[-4].startswith("Training took ") and "MAEs: 0:" in pkg_lines[-4] and "Error Ratios: 0:" in pkg_lines[-4]
    assert pkg_lines[-3] == "== Running Test on %s ==" % test_file and pkg_lines[-2].startswith("Loss 0.5") and pkg_lines[-2].endswith(" on 80 graphs")
    assert pkg_lines[-1].startswith("Metrics: MAEs: 0:")


def test_ppi_epoch_loop_writes_the_references_log(tmp_path):
    d = str(tmp_path)
    write_ppi_data(d)
    ref_lines, ref_calls, best_file = recorded_reference_loop("ppi", d)
    tr, _ = batching.load_ppi_fold(d, "train")
    va, _ = batching.load_ppi_fold(d, "valid")
    te, _ = batching.load_ppi_fold(d, "test")
    pkg_lines, pkg_calls, saves, res = run_package_loop("ppi", list(tr), list(va), (0,), best_file, max_nodes=120,
                                                        test_samples=list(te), test_description=d)
    compare(ref_lines, ref_calls, pkg_lines, pkg_calls)
    assert saves == [1, 2, 3] and pkg_lines[-1].startswith("Metrics: Avg MicroF1: ") and pkg_lines[-3] == "== Running Test on %s ==" % d
