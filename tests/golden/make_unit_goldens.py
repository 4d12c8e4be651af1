#!/usr/bin/env python
"""Golden vectors of what the container's own unit tests ask of this package, from a checkout of
aws/sagemaker-xgboost-container:

    python tests/golden/make_unit_goldens.py <path to the sagemaker-xgboost-container checkout>

Runs the container's unit-test files (test/unit/...) UNCHANGED on top of this package bound as `xgboost`, with the
oracle-backed engine (CPU), and records every call they make into the package's data and model surface:
  * each `xgb.DMatrix` built -- its inputs (arrays, sparse matrices, frames, or the bytes of the files behind a URI) and
    what it holds afterwards (shape, float32 matrix, labels, weights), or the error it raised;
  * each `Booster.predict` on such a DMatrix -- the model (UBJSON), the arguments and the returned array;
  * each `xgb.train` -- parameters, rounds, evaluation sets, the package callbacks, the model it resumed from and the
    model trained;
  * every public name they (and the container modules they exercise) look up on `xgboost` and its submodules, with the
    kind of object found, the names the container's modules take at import included (each file runs in a fresh
    interpreter);
  * how many of the file's tests passed and unexpectedly passed.
tests/test_reference_unit_suite.py replays them on the package without the container (tests/golden/container/unit_calls.npz)."""
import hashlib
import json
import os
import sys
import tempfile
import types
import unittest.mock

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
OUT = os.path.join(HERE, "container", "unit_calls.npz")

# (file under test/unit, -k expression): the recordio-protobuf cases need sagemaker_containers.record_pb2, a format
# outside this package's scope
FILES = [
    ("test_checkpointing.py", None),
    ("test_data_utils.py", "not protobuf"),
    ("test_encoder.py", "not protobuf"),
    ("test_distributed.py", None),
    ("algorithm_mode/test_custom_metrics.py", None),
    ("algorithm_mode/test_train_utils.py", None),
    ("algorithm_mode/test_serve_utils.py", "not protobuf"),
    ("test_prediction_utils.py", None),
    ("algorithm_mode/test_algorithm_mode.py", None),
    ("distributed_gpu/test_distributed_gpu_training.py", None),
    ("distributed_gpu/test_dask_data_utils.py", None),
]
MAX_FILE_BYTES = 64 * 1024           # inputs behind a URI are stored when their files are this small
MAX_ARRAY = 64 * 1024                # elements of one stored array


class Recorder:
    def __init__(self):
        self.arrays, self.events, self.models, self.skipped = {}, [], {}, {}

    def put(self, a):
        a = np.ascontiguousarray(a)
        if a.size > MAX_ARRAY:
            raise ValueError("too large")
        key = "a%d" % len(self.arrays)
        self.arrays[key] = a
        return key

    def enc(self, v):
        import scipy.sparse as sp
        import pandas as pd
        if v is None or isinstance(v, (bool, int, float, str)):
            return v
        if isinstance(v, np.generic):
            return v.item()
        if isinstance(v, np.ndarray):
            return {"array": self.put(v)}
        if sp.issparse(v):
            c = sp.csr_matrix(v)
            return {"csr": [self.put(c.data), self.put(c.indices), self.put(c.indptr)], "shape": list(c.shape)}
        if isinstance(v, pd.DataFrame):
            return {"frame": self.put(v.to_numpy()), "columns": [str(c) for c in v.columns]}
        if isinstance(v, pd.Series):
            return {"array": self.put(v.to_numpy())}
        if isinstance(v, (list, tuple)):
            return [self.enc(x) for x in v]
        if isinstance(v, dict):
            return {str(k): self.enc(x) for k, x in v.items()}
        raise ValueError("unstorable %s" % type(v).__name__)

    def enc_uri(self, uri):
        path = uri.split("?", 1)[0]
        names = sorted(os.listdir(path)) if os.path.isdir(path) else [os.path.basename(path)]
        base = path if os.path.isdir(path) else os.path.dirname(path)
        files = {}
        for n in names:
            f = os.path.join(base, n)
            if os.path.isfile(f):
                if os.path.getsize(f) > MAX_FILE_BYTES:
                    raise ValueError("file too large")
                files[n] = self.put(np.frombuffer(open(f, "rb").read(), np.uint8))
        return {"uri_query": uri[len(path):], "is_dir": os.path.isdir(path), "files": files}

    def model(self, bst):
        raw = bytes(bst.save_raw("ubj"))
        h = hashlib.sha256(raw).hexdigest()[:16]
        if h not in self.models:
            self.models[h] = self.put(np.frombuffer(raw, np.uint8)) if len(raw) <= MAX_ARRAY else None
        if self.models[h] is None:
            raise ValueError("model too large")
        return self.models[h]

    def skip(self, op, why):
        k = "%s: %s" % (op, why)
        self.skipped[k] = self.skipped.get(k, 0) + 1


def install_spies(xgb, rec):
    from sagemaker_xgboost_container_b200 import core, training
    real_init, real_predict, real_train = core.DMatrix.__init__, core.Booster.predict, training.train

    def dmatrix_init(self, data, *a, **kw):
        self._rec_id = None
        try:
            ev = {"op": "DMatrix", "data": rec.enc_uri(data) if isinstance(data, str) else rec.enc(data), "args": rec.enc(list(a)),
                  "kwargs": rec.enc(kw)}
        except Exception as e:          # noqa: BLE001
            rec.skip("DMatrix", str(e))
            return real_init(self, data, *a, **kw)
        try:
            real_init(self, data, *a, **kw)
        except Exception as e:
            ev["raises"] = type(e).__name__
            rec.events.append(ev)
            raise
        try:
            ev["result"] = {"num_row": int(self.num_row()), "num_col": int(self.num_col()), "X": rec.put(self.handle.X),
                            "label": rec.put(self.get_label()), "weight": rec.put(self.get_weight())}
        except Exception as e:          # noqa: BLE001
            rec.skip("DMatrix", str(e))
            return
        self._rec_id = len(rec.events)
        rec.events.append(ev)

    def predict(self, data, *a, **kw):
        out = real_predict(self, data, *a, **kw)
        if getattr(data, "_rec_id", None) is None:
            rec.skip("predict", "DMatrix not recorded")
            return out
        try:
            rec.events.append({"op": "predict", "model": rec.model(self), "data": data._rec_id, "args": rec.enc(list(a)), "kwargs": rec.enc(kw),
                               "result": rec.put(np.asarray(out))})
        except Exception as e:          # noqa: BLE001
            rec.skip("predict", str(e))
        return out

    def train(params, dtrain, *a, **kw):
        start = kw.get("xgb_model")                       # taken before training, which may continue it in place
        try:
            if isinstance(start, (str, os.PathLike)):
                start = xgb.Booster(model_file=os.fspath(start))
            start = None if start is None else rec.model(start)
        except Exception as e:          # noqa: BLE001
            start = e
        bst = real_train(params, dtrain, *a, **kw)
        evals = kw.get("evals") or []
        cbs = []
        for cb in kw.get("callbacks") or []:
            name = type(cb).__name__
            if not type(cb).__module__.startswith("sagemaker_xgboost_container_b200"):
                cbs.append({"class": "container." + name})
            elif name == "EarlyStopping":
                cbs.append({"class": name, "rounds": cb.rounds, "data_name": cb.data, "metric_name": cb.metric_name,
                            "save_best": cb.save_best, "maximize": cb.maximize})
            else:
                cbs.append({"class": name})
        ids = [getattr(dtrain, "_rec_id", None)] + [getattr(d, "_rec_id", None) for d, _ in evals]
        if a or kw.get("obj") is not None or None in ids or isinstance(start, Exception):
            rec.skip("train", "positional arguments, a custom objective, an unreadable starting model or an unrecorded DMatrix")
            return bst
        try:
            rec.events.append({"op": "train", "params": rec.enc(dict(params) if not isinstance(params, list) else dict(params)),
                               "num_boost_round": kw.get("num_boost_round", 10), "dtrain": ids[0],
                               "evals": [[i, n] for i, (_, n) in zip(ids[1:], evals)], "callbacks": cbs,
                               "has_custom_metric": kw.get("custom_metric") is not None or kw.get("feval") is not None,
                               "xgb_model": start, "result": rec.model(bst)})
        except Exception as e:          # noqa: BLE001
            rec.skip("train", str(e))
        return bst
    core.DMatrix.__init__, core.Booster.predict = dmatrix_init, predict
    xgb.train = train
    sys.modules["xgboost"].train = train


def _kind(v):
    import inspect
    return "class" if inspect.isclass(v) else "module" if inspect.ismodule(v) else "callable" if callable(v) else type(v).__name__


class SurfaceProxy(types.ModuleType):
    """Stands in sys.modules for `xgboost` / `xgboost.<sub>`: forwards to the package module and notes every public name
    the container's code looks up on it, with the kind of object it got."""

    def __init__(self, real, seen):
        super().__init__(real.__name__)
        object.__setattr__(self, "_real", real)
        object.__setattr__(self, "_seen", seen)

    def __getattr__(self, name):
        v = getattr(object.__getattribute__(self, "_real"), name)
        if not name.startswith("_"):
            object.__getattribute__(self, "_seen")["%s.%s" % (self.__name__, name)] = _kind(v)
        return v

    def __setattr__(self, name, v):                 # writes (mock.patch included) reach the package module
        setattr(object.__getattribute__(self, "_real"), name, v)

    def __delattr__(self, name):
        delattr(object.__getattribute__(self, "_real"), name)


class Outcome:
    """pytest plugin: how the run's tests ended (an xfail-marked test that passed counts as xpassed)."""

    def __init__(self):
        self.counts = {"passed": 0, "xpassed": 0, "failed": 0}

    def pytest_runtest_logreport(self, report):
        if report.failed:
            self.counts["failed"] += 1
        elif report.when == "call" and report.passed:
            self.counts["xpassed" if hasattr(report, "wasxfail") else "passed"] += 1


def record_file(reference, path, deselect, part):
    """One file of the container's unit tests, in a fresh interpreter (as each runs on its own): its records, into `part`."""
    import pytest
    import reference_stubs
    import sagemaker_xgboost_container_b200 as xgb
    from sagemaker_xgboost_container_b200 import backend
    from oracle.engine import OracleBackend
    backend._BACKEND = OracleBackend(error_cls=xgb.XGBoostError)
    sys.modules.setdefault("mock", unittest.mock)
    reference_stubs.install(xgb, reference)          # binds the package as `xgboost`; the container is not imported yet
    seen = {}
    for name in [n for n in sys.modules if n == "xgboost" or n.startswith("xgboost.")]:
        sys.modules[name] = SurfaceProxy(sys.modules[name], seen)
    sys.path.insert(0, reference)
    rec = Recorder()
    install_spies(xgb, rec)
    outcome = Outcome()
    tmp = tempfile.mkdtemp()
    os.chdir(tmp)                        # some of the container's tests write scratch files into the cwd
    args = ["-q", "-p", "no:cacheprovider", "--noconftest", "-c", os.devnull, "--rootdir", tmp, os.path.join(reference, "test", "unit", path)]
    code = pytest.main(args + (["-k", deselect] if deselect else []), plugins=[outcome])
    counts = {op: sum(e["op"] == op for e in rec.events) for op in ("DMatrix", "predict", "train")}
    index = {"pytest_exit": int(code), "outcome": outcome.counts, "counts": counts, "skipped": rec.skipped, "surface": dict(sorted(seen.items()))}
    print(path, "exit", int(code), outcome.counts, counts, rec.skipped, len(seen), file=sys.stderr)
    np.savez(part, index=np.array(json.dumps(index)), events=np.array(json.dumps(rec.events)), **rec.arrays)


def main(reference):
    import subprocess
    out, index = {}, {}
    for path, deselect in FILES:
        part = os.path.join(tempfile.mkdtemp(), "part.npz")
        subprocess.run([sys.executable, os.path.abspath(__file__), reference, path, deselect or "", part], check=True)
        g = np.load(part)
        index[path] = json.loads(str(g["index"]))
        for k in g.files:
            if k != "index":
                out[path + "/" + k] = g[k]
    out["index"] = np.array(json.dumps(index, indent=1, sort_keys=True))
    np.savez_compressed(OUT, **out)
    print("wrote", OUT, os.path.getsize(OUT), "bytes", file=sys.stderr)


if __name__ == "__main__":
    if len(sys.argv) == 5:
        record_file(sys.argv[1], sys.argv[2], sys.argv[3] or None, sys.argv[4])
    elif len(sys.argv) == 2:
        main(os.path.abspath(sys.argv[1]))
    else:
        sys.exit(__doc__)
