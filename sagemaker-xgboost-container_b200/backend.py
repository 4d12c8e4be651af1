"""ctypes binding of libb200xgb.so (include/b200xgb.h) -- the only compute backend of this package.

The functions bound here carry the names and conventions of libxgboost's C API, i.e. what the reference
container reaches through `import xgboost` (SURVEY.md section 8b).  There is deliberately NO CPU fallback: if the
CUDA library is missing, or no GPU is visible, every call fails loudly with XGBoostError.
"""
import ctypes as C
import json
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libb200xgb.so")

c_bst_ulong = C.c_uint64


class XGBoostError(ValueError):
    """Error raised by the native library (same name and base class as xgboost.core.XGBoostError)."""


def _cstr(s):
    return C.c_char_p(s.encode("utf-8"))


def _from_cstr_array(ptr, n):
    return [ptr[i].decode("utf-8") for i in range(n)]


_utf8_and_size = C.pythonapi.PyUnicode_AsUTF8AndSize
_utf8_and_size.restype = C.c_void_p
_utf8_and_size.argtypes = [C.py_object, C.POINTER(C.c_ssize_t)]


class CudaBackend:
    """Thin, stateless wrapper: one method per C-ABI entry point."""

    name = "cuda"

    def __init__(self, path=LIB_PATH):
        if not os.path.exists(path):
            raise XGBoostError(
                "libb200xgb.so not found at %s -- build it with `python sagemaker-xgboost-container_b200/build.py` "
                "(nvcc, sm_100a). This package has no CPU fallback." % path)
        self.lib = C.CDLL(path)
        self.lib.XGBGetLastError.restype = C.c_char_p
        self.path = path

    # ------------------------------------------------------------------ helpers
    def _check(self, ret):
        if ret != 0:
            raise XGBoostError(self.lib.XGBGetLastError().decode("utf-8", "replace"))

    def build_info(self):
        out = C.c_char_p()
        self._check(self.lib.XGBuildInfo(C.byref(out)))
        return json.loads(out.value.decode())

    # ------------------------------------------------------------------ DMatrix
    def dmatrix_from_dense(self, arr, missing):
        arr = np.ascontiguousarray(arr, dtype=np.float32)
        if arr.ndim != 2:
            raise ValueError("Expecting 2 dimensional numpy.ndarray, got: %s" % (arr.shape,))
        h = C.c_void_p()
        self._check(self.lib.XGDMatrixCreateFromMat(arr.ctypes.data_as(C.POINTER(C.c_float)), c_bst_ulong(arr.shape[0]),
                                                    c_bst_ulong(arr.shape[1]), C.c_float(missing), C.byref(h)))
        return h

    def dmatrix_from_csr(self, indptr, indices, data, ncol):
        indptr = np.ascontiguousarray(indptr, dtype=np.uint64)
        indices = np.ascontiguousarray(indices, dtype=np.uint32)
        data = np.ascontiguousarray(data, dtype=np.float32)
        h = C.c_void_p()
        self._check(self.lib.XGDMatrixCreateFromCSREx(indptr.ctypes.data_as(C.POINTER(C.c_size_t)),
                                                      indices.ctypes.data_as(C.POINTER(C.c_uint)),
                                                      data.ctypes.data_as(C.POINTER(C.c_float)), C.c_size_t(len(indptr)),
                                                      C.c_size_t(len(data)), C.c_size_t(ncol), C.byref(h)))
        return h

    def dmatrix_from_cuda_array(self, obj, missing):
        """obj exposes __cuda_array_interface__ (torch.Tensor on cuda, cupy.ndarray): float32, 2-D, C-contiguous."""
        iface = dict(obj.__cuda_array_interface__)
        iface["shape"] = list(iface["shape"])
        iface["data"] = [int(iface["data"][0]), bool(iface["data"][1])]
        iface.pop("stream", None)
        iface["strides"] = None if iface.get("strides") is None else list(iface["strides"])
        if iface["strides"] is not None:
            n, F = iface["shape"]
            if list(iface["strides"]) != [4 * F, 4]:
                raise ValueError("device array must be C-contiguous")
            iface["strides"] = None
        h = C.c_void_p()
        cfg = {} if missing is None or missing != missing else {"missing": float(missing)}
        self._check(self.lib.XGDMatrixCreateFromCudaArrayInterface(_cstr(json.dumps(iface)), _cstr(json.dumps(cfg)), C.byref(h)))
        return h

    def dmatrix_get_raw(self, h):
        n, F = self.dmatrix_num_row(h), self.dmatrix_num_col(h)
        out = np.empty(n * F, np.float32)
        self._check(self.lib.XGB200DMatrixGetRaw(h, out.ctypes.data_as(C.POINTER(C.c_float))))
        return out

    def dmatrix_from_csv_labeled(self, payload, delimiter=",", label_column=-1, weight_column=-1):
        """Device-side parse of a training CSV channel; (handle, status) like dmatrix_from_csv."""
        h = C.c_void_p()
        st = C.c_int(0)
        self._check(self.lib.XGB200DMatrixCreateFromCSVEx(C.c_char_p(payload), C.c_ulong(len(payload)), C.c_char(delimiter.encode("ascii")),
                                                          C.c_int(label_column), C.c_int(weight_column), C.byref(st), C.byref(h)))
        return (h if st.value == 0 else None), int(st.value)

    _COL_TYPES = {"<f4": 0, "<f8": 1, "<i4": 2, "<i8": 3, "|u1": 4, "|i1": 5, "<i2": 6, "<u2": 7, "<u4": 8, "<u8": 9, "|b1": 10}

    def dmatrix_from_columns(self, columns, label_column=-1, weight_column=-1):
        """Columnar input (ingest.cu): one contiguous 1-D numpy array per column, in its own dtype where the device converts it
        (float32/64, (u)int8..64, bool), anything else converted to float32 one column at a time -- never a dense host matrix."""
        cols = []
        for c in columns:
            a = np.asarray(c)
            if a.ndim != 1:
                raise ValueError("columns must be 1-dimensional")
            if a.dtype.str not in self._COL_TYPES:
                a = a.astype(np.float32)
            cols.append(np.ascontiguousarray(a))
        n = len(cols[0]) if cols else 0
        if any(len(a) != n for a in cols):
            raise ValueError("columns have different lengths")
        ptrs = (C.c_void_p * len(cols))(*[a.ctypes.data for a in cols])
        types = (C.c_int * len(cols))(*[self._COL_TYPES[a.dtype.str] for a in cols])
        h = C.c_void_p()
        self._check(self.lib.XGB200DMatrixCreateFromColumns(ptrs, types, C.c_int(len(cols)), C.c_ulong(n), C.c_int(label_column), C.c_int(weight_column), C.byref(h)))
        return h

    def dmatrix_from_libsvm_text(self, payload, whitespace_mode, absent):
        """Device-side parse of a libsvm request body (csv.cu).  Returns (handle, status); handle is None unless status == 0."""
        h = C.c_void_p()
        st = C.c_int(0)
        if isinstance(payload, str):
            size = C.c_ssize_t(0)
            ptr = _utf8_and_size(payload, C.byref(size))
            if not ptr:
                raise ValueError("libsvm payload is not valid UTF-8")
            text, length = C.c_char_p(ptr), size.value
        else:
            text, length = C.c_char_p(bytes(payload) if not isinstance(payload, bytes) else payload), len(payload)
        self._check(self.lib.XGB200DMatrixCreateFromLibsvmText(text, C.c_ulong(length), C.c_int(whitespace_mode), C.c_float(absent), C.byref(st), C.byref(h)))
        return (h if st.value == 0 else None), int(st.value)

    def dmatrix_from_csv(self, payload, delimiter=","):
        """Device-side CSV parse (csv.cu).  Returns (handle, status); handle is None unless status == 0."""
        h = C.c_void_p()
        st = C.c_int(0)
        if isinstance(payload, str):
            # CPython caches the UTF-8 form of a str (for ASCII text it IS the object's own buffer): no 200 MB .encode() copy
            size = C.c_ssize_t(0)
            ptr = _utf8_and_size(payload, C.byref(size))
            if not ptr:
                raise ValueError("CSV payload is not valid UTF-8")
            text, length = C.c_char_p(ptr), size.value
        else:
            text, length = C.c_char_p(bytes(payload) if not isinstance(payload, bytes) else payload), len(payload)
        self._check(self.lib.XGB200DMatrixCreateFromCSV(text, C.c_ulong(length), C.c_char(delimiter.encode("ascii")), C.byref(st), C.byref(h)))
        return (h if st.value == 0 else None), int(st.value)

    def dmatrix_free(self, h):
        self._check(self.lib.XGDMatrixFree(h))

    def dmatrix_num_row(self, h):
        out = c_bst_ulong()
        self._check(self.lib.XGDMatrixNumRow(h, C.byref(out)))
        return int(out.value)

    def dmatrix_num_col(self, h):
        out = c_bst_ulong()
        self._check(self.lib.XGDMatrixNumCol(h, C.byref(out)))
        return int(out.value)

    def dmatrix_set_float_info(self, h, field, arr):
        arr = np.ascontiguousarray(arr, dtype=np.float32).reshape(-1)
        self._check(self.lib.XGDMatrixSetFloatInfo(h, _cstr(field), arr.ctypes.data_as(C.POINTER(C.c_float)), c_bst_ulong(arr.size)))

    def dmatrix_get_float_info(self, h, field):
        n = c_bst_ulong()
        ptr = C.POINTER(C.c_float)()
        self._check(self.lib.XGDMatrixGetFloatInfo(h, _cstr(field), C.byref(n), C.byref(ptr)))
        if n.value == 0:
            return np.zeros(0, np.float32)
        return np.ctypeslib.as_array(ptr, shape=(n.value,)).copy()

    def dmatrix_slice(self, h, idx):
        idx = np.ascontiguousarray(idx, dtype=np.int32)
        out = C.c_void_p()
        self._check(self.lib.XGDMatrixSliceDMatrix(h, idx.ctypes.data_as(C.POINTER(C.c_int)), c_bst_ulong(len(idx)), C.byref(out)))
        return out

    def dmatrix_set_str_info(self, h, field, values):
        values = list(values or [])
        arr = (C.c_char_p * len(values))(*[v.encode("utf-8") for v in values])
        self._check(self.lib.XGDMatrixSetStrFeatureInfo(h, _cstr(field), arr, c_bst_ulong(len(values))))

    def dmatrix_get_str_info(self, h, field):
        n = c_bst_ulong()
        ptr = C.POINTER(C.c_char_p)()
        self._check(self.lib.XGDMatrixGetStrFeatureInfo(h, _cstr(field), C.byref(n), C.byref(ptr)))
        return _from_cstr_array(ptr, n.value)

    # ------------------------------------------------------------------ Booster
    def booster_create(self, dmat_handles=()):
        arr = (C.c_void_p * len(dmat_handles))(*[d.value if isinstance(d, C.c_void_p) else d for d in dmat_handles])
        h = C.c_void_p()
        self._check(self.lib.XGBoosterCreate(arr, c_bst_ulong(len(dmat_handles)), C.byref(h)))
        return h

    def booster_free(self, h):
        self._check(self.lib.XGBoosterFree(h))

    def booster_set_param(self, h, k, v):
        self._check(self.lib.XGBoosterSetParam(h, _cstr(str(k)), _cstr(str(v))))

    def booster_update(self, h, it, dh):
        self._check(self.lib.XGBoosterUpdateOneIter(h, C.c_int(it), dh))

    def booster_eval(self, h, it, dhs, names):
        dm = (C.c_void_p * len(dhs))(*[d.value for d in dhs])
        nm = (C.c_char_p * len(names))(*[n.encode("utf-8") for n in names])
        out = C.c_char_p()
        self._check(self.lib.XGBoosterEvalOneIter(h, C.c_int(it), dm, nm, c_bst_ulong(len(dhs)), C.byref(out)))
        return out.value.decode("utf-8")

    def booster_predict(self, h, dh, cfg):
        shape = C.POINTER(c_bst_ulong)()
        dim = c_bst_ulong()
        res = C.POINTER(C.c_float)()
        self._check(self.lib.XGBoosterPredictFromDMatrix(h, dh, _cstr(json.dumps(cfg)), C.byref(shape), C.byref(dim), C.byref(res)))
        shp = tuple(int(shape[i]) for i in range(dim.value))
        n = int(np.prod(shp)) if shp else 0
        if n == 0:
            return np.zeros(shp, np.float32)
        return np.ctypeslib.as_array(res, shape=(n,)).copy().reshape(shp)

    def booster_save_raw(self, h, fmt):
        n = c_bst_ulong()
        ptr = C.POINTER(C.c_char)()
        self._check(self.lib.XGBoosterSaveModelToBuffer(h, _cstr(json.dumps({"format": fmt})), C.byref(n), C.byref(ptr)))
        return C.string_at(ptr, n.value)

    def booster_load_raw(self, h, buf):
        buf = bytes(buf)
        self._check(self.lib.XGBoosterLoadModelFromBuffer(h, buf, c_bst_ulong(len(buf))))

    def booster_serialize(self, h):
        n = c_bst_ulong()
        ptr = C.POINTER(C.c_char)()
        self._check(self.lib.XGBoosterSerializeToBuffer(h, C.byref(n), C.byref(ptr)))
        return C.string_at(ptr, n.value)

    def booster_unserialize(self, h, buf):
        buf = bytes(buf)
        self._check(self.lib.XGBoosterUnserializeFromBuffer(h, buf, c_bst_ulong(len(buf))))

    def booster_save_config(self, h):
        n = c_bst_ulong()
        out = C.c_char_p()
        self._check(self.lib.XGBoosterSaveJsonConfig(h, C.byref(n), C.byref(out)))
        return out.value.decode("utf-8")

    def booster_load_config(self, h, s):
        self._check(self.lib.XGBoosterLoadJsonConfig(h, _cstr(s)))

    def booster_num_features(self, h):
        out = c_bst_ulong()
        self._check(self.lib.XGBoosterGetNumFeature(h, C.byref(out)))
        return int(out.value)

    def booster_boosted_rounds(self, h):
        out = C.c_int()
        self._check(self.lib.XGBoosterBoostedRounds(h, C.byref(out)))
        return int(out.value)

    def booster_slice(self, h, begin, end, step):
        out = C.c_void_p()
        self._check(self.lib.XGBoosterSlice(h, C.c_int(begin), C.c_int(end), C.c_int(step), C.byref(out)))
        return out

    def booster_get_attr(self, h, key):
        out = C.c_char_p()
        ok = C.c_int()
        self._check(self.lib.XGBoosterGetAttr(h, _cstr(key), C.byref(out), C.byref(ok)))
        return out.value.decode("utf-8") if ok.value else None

    def booster_set_attr(self, h, key, value):
        self._check(self.lib.XGBoosterSetAttr(h, _cstr(key), None if value is None else _cstr(str(value))))

    def booster_attr_names(self, h):
        n = c_bst_ulong()
        ptr = C.POINTER(C.c_char_p)()
        self._check(self.lib.XGBoosterGetAttrNames(h, C.byref(n), C.byref(ptr)))
        return _from_cstr_array(ptr, n.value)

    def booster_set_str_info(self, h, field, values):
        values = list(values or [])
        arr = (C.c_char_p * len(values))(*[v.encode("utf-8") for v in values])
        self._check(self.lib.XGBoosterSetStrFeatureInfo(h, _cstr(field), arr, c_bst_ulong(len(values))))

    def booster_get_str_info(self, h, field):
        n = c_bst_ulong()
        ptr = C.POINTER(C.c_char_p)()
        self._check(self.lib.XGBoosterGetStrFeatureInfo(h, _cstr(field), C.byref(n), C.byref(ptr)))
        return _from_cstr_array(ptr, n.value)

    # ------------------------------------------------------------------ collective
    def comm_unique_id(self):
        out = C.c_char_p()
        self._check(self.lib.XGCommunicatorGetUniqueId(C.byref(out)))
        return out.value.decode()

    def comm_init(self, cfg):
        self._check(self.lib.XGCommunicatorInit(_cstr(json.dumps(cfg))))

    def comm_finalize(self):
        self._check(self.lib.XGCommunicatorFinalize())

    def comm_peer_reduce_active(self):
        return bool(self.lib.XGB200CommPeerReduceActive())

    def comm_rank(self):
        return int(self.lib.XGCommunicatorGetRank())

    def comm_world(self):
        return int(self.lib.XGCommunicatorGetWorldSize())

    # ------------------------------------------------------------------ introspection (tests / bench)
    def dmatrix_get_cuts(self, h, max_bin):
        n_ptrs, n_vals = c_bst_ulong(), c_bst_ulong()
        ptrs, vals, mins = C.POINTER(C.c_int)(), C.POINTER(C.c_float)(), C.POINTER(C.c_float)()
        hm = C.c_int()
        self._check(self.lib.XGB200DMatrixGetCuts(h, C.c_int(max_bin), C.byref(n_ptrs), C.byref(ptrs), C.byref(n_vals), C.byref(vals),
                                                  C.byref(mins), C.byref(hm)))
        F = n_ptrs.value - 1
        return (np.ctypeslib.as_array(ptrs, shape=(n_ptrs.value,)).copy(), np.ctypeslib.as_array(vals, shape=(n_vals.value,)).copy(),
                np.ctypeslib.as_array(mins, shape=(F,)).copy() if F else np.zeros(0, np.float32), bool(hm.value))

    def dmatrix_set_cuts(self, h, ptrs, vals, mins):
        ptrs = np.ascontiguousarray(ptrs, np.int32)
        vals = np.ascontiguousarray(vals, np.float32)
        mins = np.ascontiguousarray(mins, np.float32)
        self._check(self.lib.XGB200DMatrixSetCuts(h, ptrs.ctypes.data_as(C.POINTER(C.c_int)), c_bst_ulong(len(ptrs)),
                                                  vals.ctypes.data_as(C.POINTER(C.c_float)), mins.ctypes.data_as(C.POINTER(C.c_float))))

    def dmatrix_get_bins(self, h, max_bin):
        n, F = self.dmatrix_num_row(h), self.dmatrix_num_col(h)
        out = np.zeros((n, F), np.uint8)
        self._check(self.lib.XGB200DMatrixGetBins(h, C.c_int(max_bin), out.ctypes.data_as(C.POINTER(C.c_uint8))))
        return out

    def booster_export_model(self, h):
        nt, nn = c_bst_ulong(), c_bst_ulong()
        bs = C.c_float()
        nc = C.c_int()
        self._check(self.lib.XGB200BoosterModelShape(h, C.byref(nt), C.byref(nn), C.byref(bs), C.byref(nc)))
        nt, nn = nt.value, nn.value
        m = {"tree_offset": np.zeros(nt + 1, np.int64), "tree_info": np.zeros(nt, np.int32)}
        for k in ("left", "right", "parent", "split_index", "split_bin"):
            m[k] = np.zeros(nn, np.int32)
        m["default_left"] = np.zeros(nn, np.uint8)
        for k in ("split_cond", "base_weight", "loss_chg", "sum_hess"):
            m[k] = np.zeros(nn, np.float32)
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        self._check(self.lib.XGB200BoosterExportModel(h, p(m["tree_offset"]), p(m["tree_info"]), p(m["left"]), p(m["right"]), p(m["parent"]),
                                                      p(m["split_index"]), p(m["split_bin"]), p(m["default_left"]), p(m["split_cond"]),
                                                      p(m["base_weight"]), p(m["loss_chg"]), p(m["sum_hess"])))
        m["base_score"] = float(bs.value)
        m["num_class"] = int(nc.value)
        return m

    def build_root_histogram(self, bh, dh, gpair, repeats=1):
        gpair = np.ascontiguousarray(gpair, np.float32)
        F = self.dmatrix_num_col(dh)
        hist = np.zeros((F, 256, 2), np.int64)
        scales = np.zeros(4, np.float32)
        ms = C.c_float()
        self._check(self.lib.XGB200BuildRootHistogram(bh, dh, gpair.ctypes.data_as(C.POINTER(C.c_float)), C.c_int(repeats),
                                                      hist.ctypes.data_as(C.POINTER(C.c_int64)), scales.ctypes.data_as(C.POINTER(C.c_float)),
                                                      C.byref(ms)))
        return hist, scales, float(ms.value)

    def build_histogram_ex(self, bh, dh, gpair, mode=0, row_ids=None, repeats=1):
        """Kernel-level entry point: (hist [F][256][2] int64, scales, ms, kernel name); see include/b200xgb.h."""
        gpair = np.ascontiguousarray(gpair, np.float32)
        F = self.dmatrix_num_col(dh)
        hist = np.zeros((F, 256, 2), np.int64)
        scales = np.zeros(4, np.float32)
        ms = C.c_float()
        name = C.c_char_p()
        ids, n_ids = None, 0
        if row_ids is not None:
            row_ids = np.ascontiguousarray(row_ids, np.uint32)
            ids, n_ids = row_ids.ctypes.data_as(C.POINTER(C.c_uint)), len(row_ids)
        self._check(self.lib.XGB200BuildHistogramEx(bh, dh, gpair.ctypes.data_as(C.POINTER(C.c_float)), C.c_int(repeats), C.c_int(mode), ids,
                                                    C.c_ulong(n_ids), hist.ctypes.data_as(C.POINTER(C.c_int64)),
                                                    scales.ctypes.data_as(C.POINTER(C.c_float)), C.byref(ms), C.byref(name)))
        return hist, scales, float(ms.value), (name.value or b"").decode()

    def booster_predict_kernel_ms(self, bh, dh, repeats=5):
        ms = C.c_float()
        self._check(self.lib.XGB200BoosterPredictKernelMs(bh, dh, C.c_int(repeats), C.byref(ms)))
        return float(ms.value)

    def predict_plan(self, data_features, model_features, node_counts, tree_begin=0, children_adjacent=True):
        """The predictor's launch plan for trees [tree_begin, tree_begin + len(node_counts)) (host code, no device)."""
        counts = np.ascontiguousarray(node_counts, np.int64)
        out = C.c_char_p()
        self._check(self.lib.XGB200PredictPlan(C.c_int(data_features), C.c_int(model_features), counts.ctypes.data_as(C.POINTER(C.c_int64)),
                                               C.c_int(tree_begin), C.c_int(tree_begin + len(counts)), C.c_int(1 if children_adjacent else 0),
                                               C.byref(out)))
        return json.loads(out.value.decode())

    def booster_predict_plan(self, bh, dh, iteration_range=(0, 0)):
        """The plan XGBoosterPredictFromDMatrix runs for `dh` over `iteration_range`."""
        out = C.c_char_p()
        self._check(self.lib.XGB200BoosterPredictPlan(bh, dh, C.c_int(int(iteration_range[0])), C.c_int(int(iteration_range[1])), C.byref(out)))
        return json.loads(out.value.decode())

    def booster_cached_margin(self, bh, dh, K):
        n = self.dmatrix_num_row(dh)
        out = np.zeros((n, K), np.float32)
        self._check(self.lib.XGB200BoosterGetCachedMargin(bh, dh, out.ctypes.data_as(C.POINTER(C.c_float))))
        return out

    def timer_start(self):
        self._check(self.lib.XGB200TimerStart())

    def timer_stop(self):
        ms = C.c_float()
        self._check(self.lib.XGB200TimerStop(C.byref(ms)))
        return float(ms.value)

    def booster_set_profile(self, bh, enable):
        self._check(self.lib.XGB200BoosterSetProfile(bh, C.c_int(1 if enable else 0)))

    def booster_get_profile(self, bh):
        out = C.c_char_p()
        self._check(self.lib.XGB200BoosterGetProfile(bh, C.byref(out)))
        return json.loads(out.value.decode())

    def launch_count(self):
        out = C.c_longlong()
        self._check(self.lib.XGB200LaunchCount(C.byref(out)))
        return int(out.value)

    def synchronize(self):
        self._check(self.lib.XGB200Synchronize())


_BACKEND = None


def get_backend():
    """The process-wide backend. Tests may replace `_BACKEND` (e.g. with the oracle-backed engine in tests/)."""
    global _BACKEND
    if _BACKEND is None:
        _BACKEND = CudaBackend()
    return _BACKEND
