"""BASELINE config 1: the container's own entry point `algorithm_mode.train.sagemaker_train` on top of this package bound as
`xgboost`, REPLAYED on the CPU test engine.  tests/golden/make_container_goldens.py ran sagemaker_train unchanged (oracle-backed
engine) and recorded every `xgb.train` call it made -- parameters, rounds, evaluation sets, callbacks, the rows a k-fold split
sliced -- with the evaluation lines it printed, the error it raised and the model each call trained
(tests/golden/container/entrypoint.json, entrypoint_models.npz).  Here the same calls run through this package's loaders and
callbacks and must reproduce those records: tree structure identical, leaves within 1e-5, every evaluation line to the
printed precision.  Plus what test/integration/local/test_abalone.py asserts (model file present, no failure) and a model
file the oracle can read back."""
import json
import os
import re
import shutil

import numpy as np
import pytest

from util import assert_same_structure, max_leaf_diff

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
G = os.path.join(GOLDEN, "abalone")
RECORDS = json.load(open(os.path.join(GOLDEN, "container", "entrypoint.json")))
LEAF_TOL = 1e-5


@pytest.fixture()
def xgb_cpu(monkeypatch):
    import sagemaker_xgboost_container_b200 as xgb
    from sagemaker_xgboost_container_b200 import backend
    from oracle.engine import OracleBackend
    monkeypatch.setattr(backend, "_BACKEND", OracleBackend(error_cls=xgb.XGBoostError))
    return xgb


def _libsvm_to_csv(src, dst):
    with open(dst, "w") as out:
        for line in open(src):
            p = line.split()
            vals = {int(k): v for k, v in (kv.split(":") for kv in p[1:])}
            out.write(",".join([p[0]] + [vals.get(i, "") for i in range(1, 9)]) + "\n")


def _channel(path, files, fmt):
    """A channel directory as the container reads it, and the URI its loader hands to xgb.DMatrix (data_utils.py:309-313,361)."""
    path.mkdir()
    for f in files:
        if fmt == "csv":
            _libsvm_to_csv(os.path.join(G, f), path / (f + ".csv"))
        else:
            shutil.copy(os.path.join(G, f), path / f)
    return str(path) + ("?format=csv&label_column=0&delimiter=," if fmt == "csv" else "?format=libsvm")


def _golden_model(case, i):
    g = np.load(os.path.join(GOLDEN, "container", "entrypoint_models.npz"))
    prefix = "%s/%d/" % (case, i)
    return {k[len(prefix):]: g[k] for k in g.files if k.startswith(prefix)}


def _replay(xgb, call, dtrain, evals, tmp_path, hyperparameters):
    """The recorded xgb.train call on this package; the container's own metric function (configure_feval, built from the
    eval_metric hyperparameter, which it then removes from the parameters) is replaced by that eval_metric, so the numbers
    it printed can be compared."""
    params = dict(call["params"])
    if call["has_custom_metric"]:
        params["eval_metric"] = hyperparameters["eval_metric"]
    callbacks = []
    for cb in call["callbacks"]:
        if cb["class"] == "EarlyStopping":
            callbacks.append(xgb.callback.EarlyStopping(rounds=cb["rounds"], metric_name=cb["metric_name"], data_name=cb["data_name"],
                                                        maximize=cb["maximize"], save_best=cb["save_best"]))
        elif cb["class"] == "TrainingCheckPoint":
            (tmp_path / "ck").mkdir(exist_ok=True)
            callbacks.append(xgb.callback.TrainingCheckPoint(directory=str(tmp_path / "ck"), name=cb["name"], as_pickle=cb["as_pickle"], interval=cb["interval"]))
        else:
            assert cb["class"] in ("EvaluationMonitor", "container.SaveIntermediateModelCallBack"), cb
    res = {}
    bst = xgb.train(params, dtrain, num_boost_round=call["num_boost_round"], evals=evals, evals_result=res, callbacks=callbacks, verbose_eval=False)
    return bst, res


def _assert_same_model(xgb, bst, call, ref):
    from oracle import ubjson
    got = ubjson.model_from_xgb_json(ubjson.loads(bytes(bst.save_raw("ubj"))))
    assert abs(got["base_score"] - call["base_score"]) <= 1e-6 * max(1.0, abs(call["base_score"]))
    assert_same_structure(got, ref)
    assert max_leaf_diff(got, ref) <= LEAF_TOL
    assert bst.num_boosted_rounds() == call["num_boosted_rounds"]


def _assert_eval_lines(lines, results):
    """Printed lines "[i]\\t<set>-<metric>:%.5f...": each value within the printed precision of the replayed one."""
    for line in lines:
        i = int(re.match(r"^\[(\d+)\]", line).group(1))
        for name, metric, value in re.findall(r"\t([A-Za-z0-9_]+)-([A-Za-z0-9@:_-]+?):([-0-9.eE+naif]+)", line):
            assert abs(float(value) - results[name][metric][i]) <= 6e-6, (line, results[name][metric][i])


def test_sagemaker_train_abalone_csv_50_rounds(xgb_cpu, tmp_path):
    xgb, rec = xgb_cpu, RECORDS["abalone_csv_50_rounds"]
    (call,) = rec["train_calls"]
    assert rec["error"] is None and rec["model_files"] == ["xgboost-model"] and call["evals"] == ["train", "validation"]
    dtrain = xgb.DMatrix(_channel(tmp_path / "train", ["abalone.train_0", "abalone.train_1"], "csv"))
    dval = xgb.DMatrix(_channel(tmp_path / "validation", ["abalone.validation"], "csv"))
    bst, res = _replay(xgb, call, dtrain, [(dtrain, "train"), (dval, "validation")], tmp_path, rec["hyperparameters"])
    lines = rec["eval_lines"]
    assert len(lines) == 50 and "validation-rmse:" in lines[-1] and float(lines[-1].split("validation-rmse:")[1]) < 2.6
    _assert_eval_lines(lines, res)
    _assert_same_model(xgb, bst, call, _golden_model("abalone_csv_50_rounds", 0))
    # the saved model is UBJSON in the container's schema: the independent reader + the oracle reproduce the eval line
    model_file = tmp_path / "xgboost-model"
    bst.save_model(str(model_file))                                  # train.py:479-480: extension-less => UBJSON
    from oracle import gbt_oracle as O, ubjson
    m = ubjson.model_from_xgb_json(ubjson.load(str(model_file)))
    assert len(m["tree_info"]) == 50 and m["num_feature"] == 8
    Xv = np.genfromtxt(tmp_path / "validation" / "abalone.validation.csv", delimiter=",", dtype=np.float32)
    rm = float(np.sqrt(np.mean((O.predict_margin(m, Xv[:, 1:])[:, 0] - Xv[:, 0]) ** 2)))
    assert abs(rm - res["validation"]["rmse"][-1]) < 1e-4
    # and serving loads it the way serve_utils.get_loaded_booster does
    b = xgb.Booster()
    b.load_model(str(model_file))
    assert json.loads(b.save_config())["learner"]["objective"]["name"] == "reg:squarederror"


def test_sagemaker_train_libsvm_with_checkpoints_and_early_stopping(xgb_cpu, tmp_path):
    xgb, rec = xgb_cpu, RECORDS["libsvm_checkpoints_early_stopping"]
    (call,) = rec["train_calls"]
    assert rec["error"] is None and rec["model_files"] == ["xgboost-model"]
    assert {cb["class"] for cb in call["callbacks"]} >= {"EarlyStopping", "TrainingCheckPoint"}
    dtrain = xgb.DMatrix(_channel(tmp_path / "train", ["abalone.train_0"], "libsvm"))
    dval = xgb.DMatrix(_channel(tmp_path / "validation", ["abalone.validation"], "libsvm"))
    bst, res = _replay(xgb, call, dtrain, [(dtrain, "train"), (dval, "validation")], tmp_path, rec["hyperparameters"])
    _assert_eval_lines(rec["eval_lines"], res)
    _assert_same_model(xgb, bst, call, _golden_model("libsvm_checkpoints_early_stopping", 0))
    assert bst.best_iteration == call["best_iteration"]
    assert len(os.listdir(tmp_path / "ck")) >= 1
    assert 1 <= bst.num_boosted_rounds() <= 12 and bst.num_features() == 9          # libsvm indices kept: 9 columns


def test_bad_labels_become_user_error(xgb_cpu, tmp_path):
    """The container maps the XGBoostError of its xgb.train call to UserError by its message (train.py: 'label must be in')."""
    xgb, rec = xgb_cpu, RECORDS["bad_labels"]
    (call,) = rec["train_calls"]
    assert rec["error"]["type"] == "UserError" and "label must be in" in rec["error"]["message"]
    tr = tmp_path / "train"
    tr.mkdir()
    (tr / "d.csv").write_text("5,1,2\n7,3,4\n")
    d = xgb.DMatrix(str(tr) + "?format=csv&label_column=0&delimiter=,")
    with pytest.raises(xgb.XGBoostError) as e:
        _replay(xgb, call, d, [(d, "train")], tmp_path, rec["hyperparameters"])
    assert str(e.value) == call["raises"]["message"]


def test_sagemaker_train_kfold_branch(xgb_cpu, tmp_path):
    """train.py:378-459: RepeatedKFold -> DMatrix.slice(idx) -> xgb.train per fold -> booster.predict(fold) -> N model files
    (what test/integration/local/test_kfold.py asserts), one out-of-fold prediction per row of train + validation."""
    xgb, rec = xgb_cpu, RECORDS["kfold"]
    assert rec["model_files"] == ["xgboost-model-0", "xgboost-model-1", "xgboost-model-2"] and rec["predictions_csv_rows"] == 1461 + 626
    dtrain = xgb.DMatrix(_channel(tmp_path / "train", ["abalone.train_0"], "libsvm"))
    dval = xgb.DMatrix(_channel(tmp_path / "validation", ["abalone.validation"], "libsvm"))
    # the container reads both channels into one matrix (the files of both, in name order) and slices the folds out of it
    both = xgb.DMatrix(_channel(tmp_path / "both", ["abalone.train_0", "abalone.validation"], "libsvm"))
    assert both.num_row() == 1461 + 626
    predicted = []
    for i, call in enumerate(rec["train_calls"]):
        rows = np.array(call["dtrain"]["rows"])
        held_out = np.setdiff1d(np.arange(both.num_row()), rows)
        bst, res = _replay(xgb, call, both.slice(rows), [(dtrain, "train"), (dval, "validation")], tmp_path, rec["hyperparameters"])
        _assert_same_model(xgb, bst, call, _golden_model("kfold", i))
        n = call["num_boost_round"]
        _assert_eval_lines(rec["eval_lines"][i * n:(i + 1) * n], res)          # each fold prints its rounds, in fold order
        predicted.append(held_out[np.isfinite(bst.predict(both.slice(held_out)))])
    assert len(rec["train_calls"]) == 3
    np.testing.assert_array_equal(np.sort(np.concatenate(predicted)), np.arange(1461 + 626))
