"""The REFERENCE's own unit tests (test/unit of aws/sagemaker-xgboost-container) against this package bound as `xgboost`:
boundary conformance (SURVEY.md section 4: "the reference's unit tests for loaders / checkpointing / feval are reusable as
boundary conformance tests").  tests/golden/make_unit_goldens.py ran each file unchanged on the CPU test engine, one
interpreter per file, and recorded how its tests ended and everything they asked of the package
(tests/golden/container/unit_calls.npz).  Here, without the container, each file's record is REPLAYED:
  * every public name its code looked up on `xgboost` and its submodules must exist here with the same kind of object;
  * every DMatrix it built -- loaders (CSV, libsvm, parquet files behind a URI), request encoders, labels for custom
    metrics, checkpoint data -- must hold the same matrix, labels and weights, or raise the same error;
  * every model it trained or resumed from a checkpoint must come out with the same trees (leaves within 1e-5), and every
    prediction must return the same array.
recordio-protobuf cases were deselected: `sagemaker_containers.record_pb2` is not part of this package's scope (SURVEY.md
section 2 row 10)."""
import importlib
import inspect
import json
import os

import numpy as np
import pytest

from util import assert_same_structure, max_leaf_diff

GOLDEN = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "container", "unit_calls.npz"))
INDEX = json.loads(str(GOLDEN["index"]))
LEAF_TOL = 1e-5

CASES = [
    ("test_checkpointing.py", None, 8),                       # xgb.train + checkpoint callbacks + resume (test_checkpointing.py:164-244)
    ("test_data_utils.py", "not protobuf", 17),               # CSV / libsvm / parquet -> DMatrix shapes, pipe-mode errors
    ("test_encoder.py", "not protobuf", 18),                  # serving payload -> DMatrix
    ("test_distributed.py", None, 6),                         # multi-process Rabit / tracker / collective.broadcast
    ("algorithm_mode/test_custom_metrics.py", None, 25),      # feval on raw margins with DMatrix.get_label
    ("algorithm_mode/test_train_utils.py", None, 3),
    ("algorithm_mode/test_serve_utils.py", "not protobuf", 50),   # get_loaded_booster, predict, selectable inference
    ("test_prediction_utils.py", None, 9),
    ("algorithm_mode/test_algorithm_mode.py", None, 15),      # the train entry point's error mapping (XGBoostError messages -> UserError / AlgorithmError)
    ("distributed_gpu/test_distributed_gpu_training.py", None, 9),    # validate_gpu_train_configuration, with this package's xgboost.dask bound
    ("distributed_gpu/test_dask_data_utils.py", None, 5),
]
# Not runnable for lack of third-party packages, all platform glue outside the hot path: algorithm_mode/test_serve.py (flask),
# test_serving.py / test_handler_service.py / test_training.py / test_serving_mms.py (sagemaker_containers.beta).


@pytest.fixture()
def xgb_cpu(monkeypatch):
    import sagemaker_xgboost_container_b200 as xgb
    from sagemaker_xgboost_container_b200 import backend
    from oracle.engine import OracleBackend
    monkeypatch.setattr(backend, "_BACKEND", OracleBackend(error_cls=xgb.XGBoostError))
    return xgb


def _dec(v, arr):
    import pandas as pd
    import scipy.sparse as sp
    if isinstance(v, list):
        return [_dec(x, arr) for x in v]
    if not isinstance(v, dict):
        return v
    if "array" in v and len(v) == 1:
        return arr(v["array"])
    if "csr" in v:
        return sp.csr_matrix(tuple(arr(k) for k in v["csr"]), shape=tuple(v["shape"]))
    if "frame" in v:
        return pd.DataFrame(arr(v["frame"]), columns=v["columns"])
    return {k: _dec(x, arr) for k, x in v.items()}


def _same(a, b):
    return a.shape == b.shape and np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(np.nan_to_num(a), np.nan_to_num(b))


def _model(xgb, raw):
    b = xgb.Booster()
    b.load_model(bytearray(raw.tobytes()))
    return b


def _trees(bst):
    from oracle import ubjson
    return ubjson.model_from_xgb_json(ubjson.loads(bytes(bst.save_raw("ubj"))))


def _kind(v):
    return "class" if inspect.isclass(v) else "module" if inspect.ismodule(v) else "callable" if callable(v) else type(v).__name__


@pytest.mark.parametrize("path,deselect,min_passed", CASES)
def test_reference_unit_file_passes_on_this_package(xgb_cpu, path, deselect, min_passed, tmp_path):
    xgb = xgb_cpu
    rec = INDEX[path]
    # the recording run: the file's tests passed on this package
    assert rec["pytest_exit"] == 0 and rec["outcome"]["failed"] == 0 and rec["outcome"]["passed"] >= min_passed, rec["outcome"]
    if path.endswith("test_serve_utils.py"):
        # test_get_loaded_booster[pickled_model|saved_booster] is xfail in the reference ("serialized with XGBoost <3.0 ...
        # incompatible", test_serve_utils.py:80): this package reads both legacy forms (csrc/legacy_io.cc), so they pass
        assert rec["outcome"]["xpassed"] == 2
    for name, kind in rec["surface"].items():
        module, attr = name.rsplit(".", 1)
        assert _kind(getattr(importlib.import_module(module), attr)) == kind, name
    arr = lambda k: GOLDEN[path + "/" + k]          # noqa: E731
    events = json.loads(str(GOLDEN[path + "/events"]))
    made, done = {}, {"DMatrix": 0, "predict": 0, "train": 0}
    for i, ev in enumerate(events):
        if ev["op"] == "DMatrix":
            data = ev["data"]
            if isinstance(data, dict) and "files" in data:           # a URI: the same files in a fresh directory
                d = tmp_path / ("uri%d" % i)
                d.mkdir()
                for name, key in data["files"].items():
                    (d / name).write_bytes(arr(key).tobytes())
                data = (str(d) if data["is_dir"] else str(d / next(iter(data["files"])))) + data["uri_query"]
            else:
                data = _dec(data, arr)
            if "raises" in ev:
                with pytest.raises(Exception) as e:
                    xgb.DMatrix(data, *_dec(ev["args"], arr), **_dec(ev["kwargs"], arr))
                assert type(e.value).__name__ == ev["raises"], (path, i)
            else:
                dm = xgb.DMatrix(data, *_dec(ev["args"], arr), **_dec(ev["kwargs"], arr))
                r = ev["result"]
                assert (dm.num_row(), dm.num_col()) == (r["num_row"], r["num_col"]), (path, i)
                assert _same(np.asarray(dm.handle.X, np.float32), arr(r["X"])), (path, i)
                np.testing.assert_array_equal(dm.get_label(), arr(r["label"]), err_msg="%s #%d" % (path, i))
                np.testing.assert_array_equal(dm.get_weight(), arr(r["weight"]), err_msg="%s #%d" % (path, i))
                made[i] = dm
        elif ev["op"] == "predict":
            out = _model(xgb, arr(ev["model"])).predict(made[ev["data"]], *_dec(ev["args"], arr), **_dec(ev["kwargs"], arr))
            np.testing.assert_allclose(out, arr(ev["result"]), rtol=0, atol=1e-6, err_msg="%s #%d" % (path, i))
        else:
            # the container's own callbacks only print and write checkpoint files; the package's EarlyStopping decides rounds
            callbacks = [xgb.callback.EarlyStopping(rounds=cb["rounds"], metric_name=cb["metric_name"], data_name=cb["data_name"],
                                                    maximize=cb["maximize"], save_best=cb["save_best"])
                         for cb in ev["callbacks"] if cb["class"] == "EarlyStopping"]
            assert not ev["has_custom_metric"] or not callbacks, "early stopping on a container metric cannot be replayed"
            start = None if ev["xgb_model"] is None else _model(xgb, arr(ev["xgb_model"]))
            bst = xgb.train(_dec(ev["params"], arr), made[ev["dtrain"]], num_boost_round=ev["num_boost_round"],
                            evals=[(made[j], n) for j, n in ev["evals"]], xgb_model=start, callbacks=callbacks, verbose_eval=False)
            got, ref = _trees(bst), _trees(_model(xgb, arr(ev["result"])))
            assert_same_structure(got, ref)
            if len(ref["tree_info"]):
                assert max_leaf_diff(got, ref) <= LEAF_TOL
        done[ev["op"]] += 1
    assert done == rec["counts"]
