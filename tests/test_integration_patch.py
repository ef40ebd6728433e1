"""patch_allrank() against allRank's module layout.  The reference's public names, their parameter lists and the padding
constants are stored in tests/golden/reference_api.json (oracle/make_golden.py: gen_reference_api); the test checks the
call surface against them, then runs the rebinding mechanics INTEGRATION.md describes on stand-in modules that carry
those names.  The kernels themselves are covered by the GPU tests."""
import json
import os
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def reference_api():
    with open(os.path.join(ROOT, "tests", "golden", "reference_api.json")) as fh:
        return json.load(fh)


def standin_modules(signatures):
    """allrank.* modules holding one distinct placeholder per stored name, linked into their parent packages."""
    mods = {}
    for full, names in signatures.items():
        mod = types.ModuleType(full)
        for name in names:
            setattr(mod, name, type(name, (), {}))
        mods[full] = mod
        parts = full.split(".")
        for i in range(1, len(parts)):
            mods.setdefault(".".join(parts[:i]), types.ModuleType(".".join(parts[:i])))
    for full, mod in mods.items():
        if "." in full:
            parent, child = full.rsplit(".", 1)
            setattr(mods[parent], child, mod)
    return mods


def test_patch_and_unpatch_rebinds_the_reference_names(monkeypatch):
    import inspect
    from allrank_b200 import data, inference, integration, losses, metrics, model, training
    api = reference_api()
    sig = api["signatures"]
    # same call surface: every patched callable accepts the reference's parameter names in the same order
    for name in integration.LOSS_NAMES:
        ref_params = sig["allrank.models.losses"][name]
        mine = list(inspect.signature(getattr(losses, name)).parameters)
        assert mine[:len(ref_params)] == ref_params, (name, ref_params, mine)
    for name in integration.METRIC_NAMES:
        assert list(inspect.signature(getattr(metrics, name)).parameters) == sig["allrank.models.metrics"][name], name
    ref_params = sig["allrank.models.model"]["make_model"]
    mine = list(inspect.signature(model.make_model).parameters)
    assert mine[:len(ref_params)] == ref_params and mine[len(ref_params):] == ["compute_dtype"]   # one extension
    # the callers either side of the path: same parameter names as the reference functions they replace
    for ref_mod, mine_mod, names in (("allrank.training.train_utils", training,
                                      ("metric_on_batch", "metric_on_epoch", "compute_metrics")),
                                     ("allrank.inference.inference_utils", inference, ("rank_slates",)),
                                     ("allrank.data.dataset_loading", data,
                                      ("load_libsvm_dataset", "load_libsvm_dataset_role", "load_libsvm_role",
                                       "create_data_loaders"))):
        for name in names:
            ref_params = sig[ref_mod][name]
            mine = list(inspect.signature(getattr(mine_mod, name)).parameters)
            assert mine[:len(ref_params)] == ref_params, (name, ref_params, mine)
    consts = api["dataset_loading_constants"]
    assert data.PADDED_Y_VALUE == consts["PADDED_Y_VALUE"] and data.PADDED_INDEX_VALUE == consts["PADDED_INDEX_VALUE"]

    mods = standin_modules(sig)
    for full, mod in mods.items():
        monkeypatch.setitem(sys.modules, full, mod)
    ref_losses, ref_metrics = mods["allrank.models.losses"], mods["allrank.models.metrics"]
    ref_model, ref_main = mods["allrank.models.model"], mods["allrank.main"]
    ref_tu, ref_iu = mods["allrank.training.train_utils"], mods["allrank.inference.inference_utils"]
    ref_dl = mods["allrank.data.dataset_loading"]
    originals = {n: getattr(ref_losses, n) for n in integration.LOSS_NAMES}
    orig_cm, orig_loader = ref_tu.compute_metrics, ref_dl.create_data_loaders
    saved = integration.patch_allrank(patch_data=True)
    try:
        assert ref_losses.lambdaLoss is losses.lambdaLoss
        assert ref_losses.ordinal is losses.ordinal
        assert ref_metrics.ndcg is metrics.ndcg
        assert ref_model.make_model is model.make_model
        assert ref_main.make_model is model.make_model
        assert ref_main.CustomDataParallel is integration.single_process_model
        assert ref_tu.compute_metrics is training.compute_metrics
        assert ref_iu.rank_slates is inference.rank_slates
        assert ref_dl.create_data_loaders is data.create_data_loaders
        assert ref_main.load_libsvm_dataset is data.load_libsvm_dataset
    finally:
        integration.unpatch_allrank(saved)
    for n, fn in originals.items():
        assert getattr(ref_losses, n) is fn
    assert ref_tu.compute_metrics is orig_cm and ref_dl.create_data_loaders is orig_loader
