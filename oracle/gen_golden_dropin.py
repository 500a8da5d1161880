#!/usr/bin/env python
"""Drop-in case: what the REFERENCE framework does with the plugin classes, recorded once, and the same case run on the
stand-alone mirror.

`reference_facts()` needs the reference tree (oracle/ref_stubs.py puts it on sys.path and stubs tensorflow/hyperopt,
nothing of the reference itself).  It records, from the reference's own code:
  * the abstract methods of elliot's BaseRecommenderModel (what a plugin class must implement);
  * what elliot's own DataSet gives for the kernel-side data views (`train_csr_of`, `eval_csr_of`) and the id order;
  * the errors `ModelCoordinator.single()` and `elliot.run.run_experiment` end in for `external.BPRMF` without a GPU;
  * the attributes the reference's `autoset_params()` fills and the reference BPRMF's `name` for the same parameters.
`plugin_facts()` computes the same facts on the stand-alone mirror (elliot_b200.recommender._bases, elliot_b200.run);
tests/test_dropin_reference.py compares the two.  Both expect CUDA to be hidden (CUDA_VISIBLE_DEVICES="").

    CUDA_VISIBLE_DEVICES= python oracle/gen_golden_dropin.py     # rewrites tests/golden/dropin_reference.json
"""
import json
import logging
import os
import sys
import tempfile
from types import SimpleNamespace

import numpy as np
import pandas as pd

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden", "dropin_reference.json")
PLUGIN = os.path.join(ROOT, "elliot_b200", "external", "__init__.py")
CLASSES = ("BPRMF", "BPRMF_batch", "MF2020", "MultiVAE", "NeuMF", "MultiDAE", "GMF")
PARAMS = dict(epochs=2, factors=8, lr=0.05, seed=42, batch_size=512, user_regularization=0.0025)
PARAMS_LIST = [("_factors", "factors", "f", 10, int, None), ("_learning_rate", "lr", "lr", 0.05, None, None),
               ("_bias_regularization", "bias_regularization", "bias_reg", 0, None, None),
               ("_user_regularization", "user_regularization", "u_reg", 0.0025, None, None),
               ("_positive_item_regularization", "positive_item_regularization", "pos_i_reg", 0.0025, None, None),
               ("_negative_item_regularization", "negative_item_regularization", "neg_i_reg", 0.00025, None, None),
               ("_update_negative_item_factors", "update_negative_item_factors", "up_neg_i_f", True, None, None),
               ("_update_users", "update_users", "up_u", True, None, None), ("_update_items", "update_items", "up_i", True, None, None),
               ("_update_bias", "update_bias", "up_b", True, None, None)]


def frames():
    g = np.random.default_rng(3)
    rows = sorted({(int(10 + 3 * g.integers(60)), int(100 + 7 * g.integers(40))) for _ in range(900)})
    g.shuffle(rows)
    tr = pd.DataFrame({"userId": [r[0] for r in rows[:700]], "itemId": [r[1] for r in rows[:700]], "rating": 1.0})
    keep = set(tr.userId)
    te_rows = [r for r in rows[700:] if r[0] in keep]
    te = pd.DataFrame({"userId": [r[0] for r in te_rows], "itemId": [r[1] for r in te_rows], "rating": 1.0})
    return rows, tr, te


def config(tmp):
    return SimpleNamespace(config_test=True, align_side_with_train=False, top_k=10, path_output_rec_weight=tmp,
                           path_output_rec_result=tmp, path_output_rec_performance=tmp,
                           evaluation=SimpleNamespace(simple_metrics=["nDCG", "HR"], relevance_threshold=0, paired_ttest=False,
                                                      wilcoxon_test=False, cutoffs=[10]))


def params():
    return SimpleNamespace(meta=SimpleNamespace(save_recs=False, verbose=False), **PARAMS)


def write_experiment(tmp, rows, logger_config=None):
    """The YAML an Elliot user writes to train the plugin's BPRMF (external_models_path + `external.BPRMF`)."""
    with open(os.path.join(tmp, "dataset.tsv"), "w") as fh:
        for u, i in rows:
            fh.write(f"{u}\t{i}\t1.0\t0\n")
    yml = (f"experiment:\n  dataset: dropin\n  data_config:\n    strategy: dataset\n    dataset_path: {tmp}/dataset.tsv\n"
           "  splitting:\n    test_splitting:\n      strategy: random_subsampling\n      test_ratio: 0.2\n"
           "  top_k: 10\n  evaluation:\n    simple_metrics: [nDCG]\n"
           f"  path_output_rec_result: {tmp}/recs\n  path_output_rec_weight: {tmp}/weights\n"
           f"  path_output_rec_performance: {tmp}/perf\n  path_log_folder: {tmp}/log\n"
           + (f"  path_logger_config: {logger_config}\n" if logger_config else "")
           + f"  external_models_path: {PLUGIN}\n"
           "  models:\n    external.BPRMF:\n      meta:\n        save_recs: False\n      epochs: 2\n      factors: 8\n      lr: 0.05\n")
    path = os.path.join(tmp, "cfg.yml")
    with open(path, "w") as fh:
        fh.write(yml)
    return path


def _external():
    import importlib.util
    spec = importlib.util.spec_from_file_location("external", PLUGIN)       # the reference's discovery (run.py:67-73)
    mod = importlib.util.module_from_spec(spec)
    sys.modules[spec.name] = mod
    spec.loader.exec_module(mod)
    return mod


def _csr_views(data):
    from elliot_b200.dataset import eval_csr_of, train_csr_of
    return {"train_csr": [a.tolist() for a in train_csr_of(data, "cpu")],
            "eval_csr": [a.tolist() for a in eval_csr_of(data, "test")],
            "users": [int(u) for u in data.users], "items": [int(i) for i in data.items]}


def _error(fn):
    try:
        fn()
        return "ran"
    except Exception as e:                                                   # noqa: BLE001
        return f"{type(e).__name__}: {e}"[:200]


def _probe(external, base, data, cfg):
    class Probe(external.BPRMF):
        def __init__(self):
            pass
    p = Probe()
    base.__init__(p, data, cfg, params())
    p.logger = logging.getLogger("probe")
    p._params_list = list(PARAMS_LIST)
    p.autoset_params()
    return p


def _ctor_after_check(external, data, cfg):
    """Past the device check the constructor must run the host-side init and fail only inside device code."""
    import torch
    avail = torch.cuda.is_available
    torch.cuda.is_available = lambda: True
    try:
        return _error(lambda: external.BPRMF(data=data, config=cfg, params=params()))
    finally:
        torch.cuda.is_available = avail


def _classes(external, base, mixin):
    out = {}
    for name in CLASSES:
        cls = getattr(external, name, None)
        if cls is not None:
            out[name] = {"subclass": issubclass(cls, base), "mixin": issubclass(cls, mixin),
                         "abstract_left": sorted(cls.__abstractmethods__)}
    return out


def reference_facts():
    from oracle import ref_stubs
    ref_stubs.install()
    logging.disable(logging.CRITICAL)
    from elliot.recommender.base_recommender_model import BaseRecommenderModel as RefBase
    from elliot.recommender.recommender_utils_mixin import RecMixin as RefMixin
    from elliot.recommender.latent_factor_models.BPRMF.BPRMF import BPRMF as RefBPRMF
    from elliot.hyperoptimization.model_coordinator import ModelCoordinator
    import elliot.dataset.dataset as ref_ds
    import elliot.utils.logging as elog
    from elliot.run import run_experiment
    from elliot_b200.recommender import _bases
    assert _bases.HOST == "elliot" and _bases.BaseRecommenderModel is RefBase and _bases.RecMixin is RefMixin

    rows, tr, te = frames()
    tmp = tempfile.mkdtemp()
    cfg = config(tmp)
    external = _external()
    data = ref_ds.DataSet(cfg, (tr, te), SimpleNamespace())
    out = {"abstract_methods": sorted(RefBase.__abstractmethods__), "classes": _classes(external, RefBase, RefMixin),
           "dataset_has_helper_methods": hasattr(data, "train_csr"), **_csr_views(data)}
    logcfg = ref_stubs.write_logger_config(os.path.join(tmp, "logger_config.yml"))
    elog.init(logcfg, os.path.join(tmp, "log"))
    elog.prepare_logger("external.BPRMF", os.path.join(tmp, "log"))
    out["model_coordinator"] = _error(lambda: ModelCoordinator([data], cfg, params(), external.BPRMF, 0).single())
    out["run_experiment"] = _error(lambda: run_experiment(write_experiment(tmp, rows, logcfg)))
    out["ctor_after_check"] = _ctor_after_check(external, data, cfg)
    p = _probe(external, RefBase, data, cfg)
    out["autoset"] = {"factors": p._factors, "lr": p._learning_rate, "u_reg": p._user_regularization}
    out["name"] = RefBPRMF.name.fget(p)
    return out


def plugin_facts():
    logging.disable(logging.CRITICAL)
    from elliot_b200.dataset import DataSet as Mirror
    from elliot_b200.recommender import _bases
    from elliot_b200.run import run_experiment
    rows, tr, te = frames()
    tmp = tempfile.mkdtemp()
    cfg = config(tmp)
    external = _external()
    data = Mirror(cfg, (tr, te))
    # what elliot's DataSet offers and nothing more: the views must come out the same without the mirror's helpers
    plain = SimpleNamespace(config=cfg, **{k: getattr(data, k) for k in
                                           ("users", "items", "public_items", "sp_i_train", "i_train_dict", "test_dict")})
    out = {"host": _bases.HOST, "abstract_methods": sorted(_bases.BaseRecommenderModel.__abstractmethods__),
           "classes": _classes(external, _bases.BaseRecommenderModel, _bases.RecMixin),
           "plain": _csr_views(plain), **_csr_views(data)}
    out["construct"] = _error(lambda: external.BPRMF(data=data, config=cfg, params=params()))
    out["run_experiment"] = _error(lambda: run_experiment(write_experiment(tmp, rows)))
    out["ctor_after_check"] = _ctor_after_check(external, data, cfg)
    p = _probe(external, _bases.BaseRecommenderModel, data, cfg)
    out["autoset"] = {"factors": p._factors, "lr": p._learning_rate, "u_reg": p._user_regularization}
    out["name"] = external.BPRMF.name.fget(p)
    return out


if __name__ == "__main__":
    facts = reference_facts()
    with open(GOLDEN, "w") as fh:
        json.dump(facts, fh, separators=(",", ":"))
        fh.write("\n")
    print("wrote", GOLDEN, os.path.getsize(GOLDEN), "bytes")
