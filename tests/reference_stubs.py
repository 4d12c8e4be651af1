"""Import stubs so the container's own modules (from a checkout of aws/sagemaker-xgboost-container, used by
tests/golden/make_container_goldens.py to record golden vectors) import without the third-party packages below, which are
not on the hot path.  Nothing of the container is copied; its modules run unchanged on top of our `xgboost` replacement."""
import os
import sys
import types


def _mod(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


def install(xgb_pkg, checkout):
    """Alias our package as `xgboost`, stub the absent third-party modules, put the container sources of `checkout` on sys.path."""
    src = os.path.join(checkout, "src")
    xgb_pkg.install_as_xgboost()
    if "xgboost.dask" not in sys.modules:
        d = _mod("xgboost.dask", DaskDMatrix=type("DaskDMatrix", (), {}), train=None)
        sys.modules["xgboost"].dask = d
    if "retrying" not in sys.modules:
        def retry(*a, **k):
            def deco(f):
                return f
            return deco if not (len(a) == 1 and callable(a[0])) else a[0]
        _mod("retrying", retry=retry)
    if "sagemaker_containers" not in sys.modules:
        ct = _mod("sagemaker_containers._content_types", CSV="text/csv", JSON="application/json", NPY="application/x-npy", OCTET_STREAM="application/octet-stream",
                  ANY="*/*", UTF8_TYPES=["application/json", "text/csv"])

        class UnsupportedFormatError(Exception):
            pass
        er = _mod("sagemaker_containers._errors", UnsupportedFormatError=UnsupportedFormatError, ClientError=Exception)
        rio = _mod("sagemaker_containers._recordio", _write_recordio=lambda *a, **k: None, _read_recordio=lambda *a, **k: iter(()))
        pb = _mod("sagemaker_containers.record_pb2", Record=type("Record", (), {}))
        _mod("sagemaker_containers", _content_types=ct, _errors=er, _recordio=rio, record_pb2=pb)
    for name in ("dask", "dask.distributed", "dask.array", "dask.dataframe"):
        if name not in sys.modules:
            _mod(name, Client=object, Array=type("Array", (), {}), DataFrame=type("DataFrame", (), {}))
    # only needed by the reference's test helpers (test/utils/local_mode.py), never by the hot path
    if "boto3" not in sys.modules:
        _mod("boto3", client=lambda *a, **k: None, Session=object)
        be = _mod("botocore.exceptions", ClientError=Exception)
        _mod("botocore", exceptions=be)
        sm = _mod("sagemaker", fw_utils=_mod("sagemaker.fw_utils"), utils=_mod("sagemaker.utils"))
        del sm
    if src not in sys.path:
        sys.path.insert(0, src)
    # algorithm_mode/__init__.py only pre-loads the serving model (and drags in flask/gunicorn): register the package
    # without executing that __init__, so that algorithm_mode.train / serve_utils themselves are imported unchanged.
    name = "sagemaker_xgboost_container.algorithm_mode"
    if name not in sys.modules:
        import sagemaker_xgboost_container  # noqa: F401
        pkg = types.ModuleType(name)
        pkg.__path__ = [os.path.join(src, "sagemaker_xgboost_container", "algorithm_mode")]
        pkg.__package__ = name
        sys.modules[name] = pkg
        sys.modules["sagemaker_xgboost_container"].algorithm_mode = pkg
