"""Picked up by the GPU worker processes of multi_gpu.run_training_with_dask in the CPU tests: selects the oracle-backed test
engine (the product itself only ever creates the CUDA backend) and binds the package as `xgboost`."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def use_oracle_engine():
    for p in (ROOT, os.path.join(ROOT, "tests")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import sagemaker_xgboost_container_b200 as xgb
    from sagemaker_xgboost_container_b200 import backend
    from oracle.engine import OracleBackend
    backend._BACKEND = OracleBackend(error_cls=xgb.XGBoostError)
    xgb.install_as_xgboost()


def bind_package():
    """GPU runs: only the `xgboost` alias"""
    for p in (ROOT, os.path.join(ROOT, "tests")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import sagemaker_xgboost_container_b200 as xgb
    xgb.install_as_xgboost()


def use_oracle_engine_with_container_callbacks():
    """As use_oracle_engine, plus stand-ins for the two container helpers the launcher uses when the container is installed
    (algorithm_mode.train_utils.get_eval_metrics_and_feval, callback.get_callbacks).  Like the container's, get_callbacks
    checkpoints on the master only; every call leaves a note `get_callbacks-<pid>-<is_master>` in the checkpoint directory."""
    import types
    use_oracle_engine()
    import sagemaker_xgboost_container_b200 as xgb

    def get_eval_metrics_and_feval(tuning_metric, eval_metric):
        return eval_metric, None, None

    def get_callbacks(model_dir, checkpoint_dir, early_stopping_data_name, early_stopping_metric, early_stopping_rounds,
                      save_model_on_termination, is_master, fold=None):
        open(os.path.join(checkpoint_dir, "get_callbacks-%d-%s" % (os.getpid(), is_master)), "w").close()
        callbacks = [xgb.callback.EvaluationMonitor()]
        if is_master:
            callbacks.append(xgb.callback.TrainingCheckPoint(directory=checkpoint_dir, name="xgboost-checkpoint", interval=1))
        return None, 0, callbacks
    pkg = types.ModuleType("sagemaker_xgboost_container")
    pkg.__path__ = []
    am = types.ModuleType("sagemaker_xgboost_container.algorithm_mode")
    am.__path__ = []
    am.train_utils = types.ModuleType("sagemaker_xgboost_container.algorithm_mode.train_utils")
    am.train_utils.get_eval_metrics_and_feval = get_eval_metrics_and_feval
    pkg.callback = types.ModuleType("sagemaker_xgboost_container.callback")
    pkg.callback.get_callbacks = get_callbacks
    pkg.algorithm_mode = am
    for m in (pkg, am, am.train_utils, pkg.callback):
        sys.modules[m.__name__] = m
