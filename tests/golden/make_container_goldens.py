#!/usr/bin/env python
"""Golden vectors of the container's OWN entry points, generated from a checkout of aws/sagemaker-xgboost-container:

    python tests/golden/make_container_goldens.py <path to the sagemaker-xgboost-container checkout>

Runs the container's `algorithm_mode.train.sagemaker_train`, `algorithm_mode.serve_utils.{parse_content_data, predict}`,
`encoder.{csv,libsvm}_to_dmatrix` and `distributed_gpu_training.validate_gpu_train_configuration` UNCHANGED on top of this
package bound as `xgboost`, with the oracle-backed engine (CPU), and records
  * the exact keyword arguments the container hands to `xgb.train` (so the tests can replay the call without the container),
  * the model each call trains, the evaluation lines it prints, the error it raises,
  * the predictions serve_utils returns for a CSV payload, the matrices the container's request parsers build,
  * the arguments `sagemaker_train` hands to the multi-GPU launcher, and the launcher's configuration checks.
The container's code is not needed to run the tests: tests/test_gpu_container_conformance.py replays `index.json` on the
CUDA backend, tests/test_reference_entrypoint.py, tests/test_serving_restatements.py and tests/test_multi_gpu_launcher.py
replay the rest on the CPU test engine."""
import contextlib
import hashlib
import io
import itertools
import json
import os
import re
import shutil
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
OUT = os.path.join(HERE, "container")
G = os.path.join(HERE, "abalone")
MODEL_KEYS = ("tree_offset", "tree_info", "left", "right", "parent", "split_index", "default_left", "split_cond")


def libsvm_to_csv(src, dst, fill=""):
    with open(dst, "w") as out:
        for line in open(src):
            p = line.split()
            vals = {int(k): v for k, v in (kv.split(":") for kv in p[1:])}
            out.write(",".join([p[0]] + [vals.get(i, fill) for i in range(1, 9)]) + "\n")


def channels(tmp, fmt, train_files=("abalone.train_0", "abalone.train_1"), fill=""):
    tr, va = os.path.join(tmp, "train"), os.path.join(tmp, "validation")
    os.makedirs(tr); os.makedirs(va)
    if fmt == "csv":
        for f in train_files:
            libsvm_to_csv(os.path.join(G, f), os.path.join(tr, f + ".csv"), fill)
        libsvm_to_csv(os.path.join(G, "abalone.validation"), os.path.join(va, "abalone.validation.csv"), fill)
        ct = "text/csv"
    else:
        for f in train_files:
            shutil.copy(os.path.join(G, f), tr)
        shutil.copy(os.path.join(G, "abalone.validation"), va)
        ct = "libsvm"
    dc = {"train": {"ContentType": ct, "TrainingInputMode": "File", "S3DistributionType": "FullyReplicated"},
          "validation": {"ContentType": ct, "TrainingInputMode": "File", "S3DistributionType": "FullyReplicated"}}
    return tr, va, dc


def model_arrays(ubjson, raw):
    m = ubjson.model_from_xgb_json(ubjson.loads(bytes(raw)))
    return {k: np.asarray(m[k]) for k in MODEL_KEYS}, float(m["base_score"])


def main(reference):
    import reference_stubs
    import sagemaker_xgboost_container_b200 as xgb
    from sagemaker_xgboost_container_b200 import backend, core, multi_gpu, training
    from oracle.engine import OracleBackend
    from oracle import ubjson
    backend._BACKEND = OracleBackend(error_cls=xgb.XGBoostError)
    reference_stubs.install(xgb, reference)
    from sagemaker_xgboost_container import encoder
    from sagemaker_xgboost_container.algorithm_mode import train as ref_train
    from sagemaker_xgboost_container.algorithm_mode import serve_utils
    from sagemaker_xgboost_container.distributed_gpu import distributed_gpu_training as dgt
    os.makedirs(OUT, exist_ok=True)

    # where each DMatrix came from: the URI the container's loader built, or the rows it sliced out of another DMatrix
    real_init, real_slice = core.DMatrix.__init__, core.DMatrix.slice

    def init_spy(self, data, *a, **k):
        real_init(self, data, *a, **k)
        self._golden_src = {"uri": data} if isinstance(data, str) else None

    def slice_spy(self, rindex, *a, **k):
        d = real_slice(self, rindex, *a, **k)
        d._golden_src = {"slice_of": self._golden_src, "rows": [int(i) for i in rindex]}
        return d
    core.DMatrix.__init__, core.DMatrix.slice = init_spy, slice_spy

    calls = []
    real_train = training.train

    def spy(params, dtrain, **kw):
        rec = {"params": {k: (list(v) if isinstance(v, (list, tuple)) else v) for k, v in dict(params).items()},
               "num_boost_round": kw.get("num_boost_round"), "evals": [n for _, n in kw.get("evals") or []],
               "has_custom_metric": kw.get("custom_metric") is not None,
               "dtrain": getattr(dtrain, "_golden_src", None), "eval_sources": [getattr(d, "_golden_src", None) for d, _ in kw.get("evals") or []],
               "callbacks": []}
        for cb in kw.get("callbacks") or []:
            name = type(cb).__name__
            if type(cb).__module__.startswith("sagemaker_xgboost_container_b200"):
                if name == "EarlyStopping":
                    rec["callbacks"].append({"class": name, "rounds": cb.rounds, "data_name": cb.data, "metric_name": cb.metric_name,
                                             "save_best": cb.save_best, "maximize": cb.maximize})
                elif name == "TrainingCheckPoint":
                    rec["callbacks"].append({"class": name, "name": cb._name, "as_pickle": cb._as_pickle, "interval": cb._iterations})
                else:
                    rec["callbacks"].append({"class": name})
            else:
                rec["callbacks"].append({"class": "container." + name})
        calls.append(rec)
        try:
            bst = real_train(params, dtrain, **kw)
        except Exception as e:
            rec["raises"] = {"type": type(e).__name__, "message": str(e)}
            raise
        rec["model"], rec["base_score"] = model_arrays(ubjson, bst.save_raw("ubj"))
        rec["num_boosted_rounds"] = bst.num_boosted_rounds()
        rec["best_iteration"] = getattr(bst, "best_iteration", None)
        return bst
    xgb.train = spy
    sys.modules["xgboost"].train = spy

    def run(tmp, hp, dc, tr, va, checkpoint_config=None, env=None):
        calls.clear()
        buf = io.StringIO()
        old = {k: os.environ.get(k) for k in env or {}}
        os.environ.update(env or {})
        err = None
        try:
            with contextlib.redirect_stdout(buf):
                ref_train.sagemaker_train(train_config=dict(hp), data_config=dc, train_path=tr, val_path=va, model_dir=os.path.join(tmp, "model"),
                                          sm_hosts=["algo-1"], sm_current_host="algo-1", checkpoint_config=checkpoint_config or {})
        except Exception as e:
            err = {"type": type(e).__name__, "message": str(e)}
        finally:
            for k, v in old.items():
                if v is None:
                    os.environ.pop(k)
                else:
                    os.environ[k] = v
        return [l for l in buf.getvalue().splitlines() if l.startswith("[")], err

    # ---- index.json: replayed on the CUDA backend
    cases = {
        "cfg1_csv": dict(hp={"objective": "reg:squarederror", "tree_method": "hist", "num_round": "50"}, fmt="csv"),           # BASELINE config 1
        "fixture_hp_libsvm": dict(hp={"objective": "reg:linear", "max_depth": "5", "eta": "0.2", "gamma": "4", "min_child_weight": "6",
                                      "subsample": "0.7", "num_round": "50"}, fmt="libsvm"),                                  # test_abalone.py:36-47
    }
    index = {}
    for name, case in cases.items():
        tmp = tempfile.mkdtemp()
        tr, va, dc = channels(tmp, case["fmt"], ("abalone.train_0", "abalone.train_1") if case["fmt"] == "csv" else ("abalone.train_0",))
        lines, err = run(tmp, case["hp"], dc, tr, va)
        assert err is None, err
        md = os.path.join(tmp, "model")
        shutil.copy(os.path.join(md, "xgboost-model"), os.path.join(OUT, name + "_model.ubj"))
        call = {k: calls[0][k] for k in ("params", "num_boost_round", "evals", "has_custom_metric")}
        index[name] = {"format": case["fmt"], "hyperparameters": case["hp"], "train_call": call, "last_eval_line": lines[-1], "eval_lines": len(lines)}
        # serving: the container's own parse + predict on a CSV payload (first 40 validation rows, label column dropped)
        if name == "cfg1_csv":
            rows = open(os.path.join(va, "abalone.validation.csv")).read().splitlines()[:40]
            payload = "\n".join(",".join(r.split(",")[1:]) for r in rows).encode("utf-8")
            dtest, ctype = serve_utils.parse_content_data(payload, "text/csv")
            boosters, formats = serve_utils.get_loaded_booster(md)
            preds = serve_utils.predict(boosters, formats, dtest, ctype, objective="reg:squarederror")
            index[name]["serve"] = {"payload": payload.decode("utf-8"), "content_type": "text/csv", "model_format": formats[0],
                                    "predictions": [float(p) for p in preds]}
        shutil.rmtree(tmp)
    json.dump(index, open(os.path.join(OUT, "index.json"), "w"), indent=1)

    # ---- entrypoint.json + entrypoint_models.npz: sagemaker_train runs replayed on the CPU test engine
    entry, arrays = {}, {}
    runs = {
        "abalone_csv_50_rounds": dict(hp={"objective": "reg:squarederror", "tree_method": "hist", "num_round": "50", "max_depth": "5", "eta": "0.2",
                                          "gamma": "4", "min_child_weight": "6"}, fmt="csv", files=("abalone.train_0", "abalone.train_1")),
        "libsvm_checkpoints_early_stopping": dict(hp={"objective": "reg:linear", "num_round": "12", "max_depth": "4", "eta": "0.3", "early_stopping_rounds": "3",
                                                      "eval_metric": "rmse", "save_model_on_termination": "true"}, fmt="libsvm", checkpoints=True),
        "bad_labels": dict(hp={"objective": "binary:logistic", "num_round": "2"}, fmt="bad_csv"),
        "kfold": dict(hp={"objective": "reg:squarederror", "num_round": "5", "max_depth": "3", "_kfold": "3", "eval_metric": "rmse"}, fmt="libsvm"),
        "dask_route_single_process": dict(hp={"objective": "reg:squarederror", "tree_method": "hist", "num_round": "8", "max_depth": "4", "eta": "0.3",
                                              "eval_metric": "rmse"}, fmt="csv", fill="0", files=("abalone.train_0", "abalone.train_1")),
    }
    for name, case in runs.items():
        tmp = tempfile.mkdtemp()
        if case["fmt"] == "bad_csv":
            tr, va = os.path.join(tmp, "train"), None
            os.makedirs(tr)
            open(os.path.join(tr, "d.csv"), "w").write("5,1,2\n7,3,4\n")
            dc = {"train": {"ContentType": "text/csv", "TrainingInputMode": "File", "S3DistributionType": "FullyReplicated"}}
        else:
            tr, va, dc = channels(tmp, case["fmt"], case.get("files", ("abalone.train_0",)), case.get("fill", ""))
        ck = None
        if case.get("checkpoints"):
            ck = os.path.join(tmp, "ck")
            os.makedirs(ck)
        out = os.path.join(tmp, "output")
        os.makedirs(out)
        lines, err = run(tmp, case["hp"], dc, tr, va, {"LocalPath": ck} if ck else {}, {"SM_OUTPUT_DATA_DIR": out})
        md = os.path.join(tmp, "model")
        rec = {"hyperparameters": case["hp"], "format": case["fmt"], "eval_lines": lines, "error": err,
               "model_files": sorted(os.listdir(md)) if os.path.isdir(md) else [], "train_calls": []}
        if os.path.exists(os.path.join(out, "predictions.csv")):
            rec["predictions_csv_rows"] = len(open(os.path.join(out, "predictions.csv")).read().strip().splitlines())
        for i, c in enumerate(calls):
            c = dict(c)
            model = c.pop("model", None)
            if model is not None:
                for k, v in model.items():
                    arrays["%s/%d/%s" % (name, i, k)] = v
            for s in [c["dtrain"]] + c["eval_sources"]:
                while s is not None:
                    if "uri" in s:
                        s["uri"] = s["uri"].replace(tmp, "{tmp}")
                    s = s.get("slice_of")
            rec["train_calls"].append(c)
        entry[name] = rec
        shutil.rmtree(tmp)

    # the container's own Dask route, left unbound (distributed_gpu_training.run_training_with_dask): the calls it makes into
    # this package's xgboost.dask, and what they give back.  The Dask cluster itself is stubbed: a Client that is a context
    # manager, dask.array.from_array returning the array.
    import types
    import warnings
    from sagemaker_xgboost_container.distributed_gpu import dask_data_utils as ddu
    dask_calls = {"matrices": [], "train": None}
    real_ddm, real_dtrain = xgb.dask.DaskDMatrix, xgb.dask.train

    def ddm_spy(client, data, label=None, **kw):
        d32, l32 = np.ascontiguousarray(data, np.float32), np.ascontiguousarray(label, np.float32)
        dask_calls["matrices"].append({"shape": list(d32.shape), "kwargs": sorted(kw),
                                       "sha256": hashlib.sha256(d32.tobytes() + l32.tobytes()).hexdigest()})
        m = real_ddm(client, data, label, **kw)
        m._golden_index = len(dask_calls["matrices"]) - 1
        return m

    def dtrain_spy(client, params, dtrain, **kw):
        out = real_dtrain(client, params, dtrain, **kw)
        dask_calls["train"] = {"params": {k: (list(v) if isinstance(v, (list, tuple)) else v) for k, v in dict(params).items()},
                               "num_boost_round": kw.get("num_boost_round"), "dtrain": dtrain._golden_index,
                               "evals": [[d._golden_index, n] for d, n in kw.get("evals") or []],
                               "has_custom_metric": kw.get("custom_metric") is not None, "verbose_eval": kw.get("verbose_eval", "default"),
                               "callbacks": [type(cb).__module__.split(".")[0] + "." + type(cb).__name__ for cb in kw.get("callbacks") or []]}
        model, _ = model_arrays(ubjson, out["booster"].save_raw("ubj"))
        for k, v in model.items():
            arrays["dask_route_unbound/0/%s" % k] = v
        return out

    class Client:
        def __init__(self, address): self.address = address
        def __enter__(self): return self
        def __exit__(self, *a): return False
        def wait_for_workers(self, n, timeout): pass
        def scheduler_info(self): return {"workers": {"w0": {}, "w1": {}}}
    dask_stub = types.SimpleNamespace(DaskDMatrix=ddm_spy, train=dtrain_spy)
    dgt.Client, dgt.dxgb, ddu.dxgb = Client, dask_stub, dask_stub
    ddu.da = types.SimpleNamespace(from_array=lambda a, chunks=None: a)
    dgt.start_daemons_in_current_instance = lambda *a, **k: None
    dgt.get_host_ip = lambda h: "127.0.0.1"
    tmp = tempfile.mkdtemp()
    tr, va, _ = channels(tmp, "csv", ("abalone.train_0", "abalone.train_1"), "0")
    os.makedirs(os.path.join(tmp, "m"))
    hp = {"objective": "reg:squarederror", "tree_method": "hist", "num_round": 5, "max_depth": 3, "eval_metric": ["rmse"]}
    buf = io.StringIO()
    with warnings.catch_warnings(record=True) as caught, contextlib.redirect_stdout(buf):
        warnings.simplefilter("always")
        dgt.run_training_with_dask(hyperparameters=dict(hp), train_path=tr, validation_path=va, model_dir=os.path.join(tmp, "m"), content_type="csv",
                                   sm_hosts=["algo-1"], current_host="algo-1", checkpoint_dir=None, num_gpus=2)
    dask_calls.update(hyperparameters=hp, warnings=[str(w.message) for w in caught if issubclass(w.category, UserWarning)],
                      eval_lines=[l for l in buf.getvalue().splitlines() if l.startswith("[")], model_files=sorted(os.listdir(os.path.join(tmp, "m"))))
    entry["dask_route_unbound"] = dask_calls
    shutil.rmtree(tmp)

    # what sagemaker_train hands to the multi-GPU launcher (train.py: use_dask_gpu_training), recorded instead of run
    launcher = {}

    def launcher_spy(**kw):
        launcher.update(kw)
    dgt.run_training_with_dask = launcher_spy
    tmp = tempfile.mkdtemp()
    tr, va, dc = channels(tmp, "csv", ("abalone.train_0", "abalone.train_1"), "0")
    os.makedirs(os.path.join(tmp, "ck"))
    hp = dict(runs["dask_route_single_process"]["hp"], use_dask_gpu_training="true")
    old_gpus = os.environ.get("SM_NUM_GPUS")
    os.environ["SM_NUM_GPUS"] = "2"
    _, err = run(tmp, hp, dc, tr, va, {"LocalPath": os.path.join(tmp, "ck")})
    if old_gpus is None:
        os.environ.pop("SM_NUM_GPUS")
    assert err is None, err
    entry["dask_route_launcher_call"] = {"hyperparameters": hp, "kwargs": json.loads(json.dumps(launcher).replace(tmp, "{tmp}"))}
    shutil.rmtree(tmp)
    json.dump(entry, open(os.path.join(OUT, "entrypoint.json"), "w"), indent=1, sort_keys=True)
    np.savez_compressed(os.path.join(OUT, "entrypoint_models.npz"), **arrays)

    # ---- serving.npz: the matrices the container's request parsers build (or the error they raise) on the bodies of
    # tests/test_gpu_serving.py / tests/test_serving_restatements.py
    import test_serving_restatements as S
    mats, errors = {}, {}

    def keep(key, fn):
        try:
            mats[key] = np.asarray(fn().handle.X, np.float32)
        except Exception as e:
            errors[key] = type(e).__name__
    for i, body in enumerate(S.libsvm_bodies()):
        keep("libsvm_sparse/%d" % i, lambda: xgb.DMatrix(serve_utils._get_sparse_matrix_from_libsvm(body)))
        keep("libsvm_dense/%d" % i, lambda: encoder.libsvm_to_dmatrix(body))
    keep("libsvm_sparse/tab_inside_token", lambda: xgb.DMatrix(serve_utils._get_sparse_matrix_from_libsvm(S.TAB_INSIDE_TOKEN)))
    keep("libsvm_dense/no_entries", lambda: encoder.libsvm_to_dmatrix(S.NO_ENTRIES))
    for i, (body, delim) in enumerate(S.csv_bodies()):
        with np.errstate(over="ignore"):
            keep("csv/%d" % i, lambda: encoder.csv_to_dmatrix(body, dtype=float))
    # a dense-route matrix that is exactly the sparse-route one with its missing entries as 0.0 is stored as that fact
    derived = [k for k in mats if k.startswith("libsvm_dense/") and k.replace("dense", "sparse") in mats
               and np.array_equal(mats[k], np.nan_to_num(mats[k.replace("dense", "sparse")], nan=0.0, posinf=np.inf, neginf=-np.inf))]
    for k in derived:
        del mats[k]
    np.savez_compressed(os.path.join(OUT, "serving.npz"), errors=np.array(json.dumps(errors, sort_keys=True)),
                        dense_is_sparse_with_zeros=np.array(sorted(derived)), **mats)

    # ---- launcher_validation.json: validate_gpu_train_configuration over every combination of its inputs
    grid = []
    dcs = {"replicated": {"train": {"S3DistributionType": "FullyReplicated"}, "validation": {"S3DistributionType": "FullyReplicated"}},
           "sharded": {"train": {"S3DistributionType": "ShardedByS3Key"}},
           "mixed": {"train": {"S3DistributionType": "FullyReplicated"}, "validation": {"S3DistributionType": "ShardedByS3Key"}},
           "unset": {"train": {}}}
    for tm, hosts, gpus, mode, fmt, dck in itertools.product(("hist", "gpu_hist", "approx"), (1, 2), (0, 8), ("File", "Pipe"),
                                                             ("csv", "parquet", "libsvm", "text/csv"), sorted(dcs)):
        grid.append([tm, hosts, gpus, mode, fmt, dck, dgt.validate_gpu_train_configuration(tm, hosts, gpus, mode, fmt, dcs[dck])])
    # by the name of the module constant each message is (this package words them for its own launcher)
    messages = ["NON_GPU_ERROR_MSG", "PIPE_MODE_ERROR_MSG", "INPUT_FORMAT_ERROR_MSG", "NOT_REPLICATED_ERROR_MSG"]
    for case in grid:
        case[-1] = [[getattr(dgt, n) for n in messages].index(m) for m in case[-1]]
    json.dump({"messages": messages, "data_configs": dcs,
               "cases (tree_method, num_hosts, num_gpus, input_mode, input_format, data_config, messages)": grid},
              open(os.path.join(OUT, "launcher_validation.json"), "w"))
    print("wrote", sorted(os.listdir(OUT)))


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(os.path.abspath(sys.argv[1]))
