"""L3 parity (SURVEY.md 8c): the reference's training driver -- `allrank.main.run()` -> `train_utils.fit` -- on the
reference's own dummy data, with allrank_b200's model, losses and epoch metrics on cuda:0, against what the unmodified
reference computes on the host CPU.

The driver is oracle/train_ref.py, a restatement of run() / fit() that reproduces the reference's result bit for bit
when given the reference's components.  The reference's result is stored in tests/golden/l3_reference.json
(oracle/make_golden.py: gen_l3).  Anchor: BASELINE config 1 reaches val ndcg_5 = 0.5709 on the reference
(BASELINE.md section 2).
"""
import json
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def reference_result(config):
    with open(os.path.join(ROOT, "tests", "golden", "l3_reference.json")) as fh:
        return json.load(fh)[config]


def run_on_b200(workdir, config):
    """run() on cuda:0 with allrank_b200 standing in for the reference's make_model, losses and compute_metrics.
    Returns the result with experiment_result.json's flattened keys, and whether liballrank_b200.so is loaded."""
    from allrank_b200 import losses, training
    from allrank_b200.model import make_model
    from oracle import train_ref
    with open(os.path.join(ROOT, "tests", "configs", config + ".json")) as fh:
        cfg = json.load(fh)
    data = os.path.join(str(workdir), "dummy_data")
    np_state = np.random.get_state()
    try:
        with torch.random.fork_rng(devices=[0]):
            train_ref.write_dummy_data(data)
            res = train_ref.run(cfg, data, torch.device("cuda", 0), make_model, losses, training.compute_metrics)
    finally:
        np.random.set_state(np_state)
    out = {"epochs": res["epochs"], "num_params": res["num_params"]}
    for role in ("train", "val"):
        out.update({f"{role}_metrics/{k}": v for k, v in res[role + "_metrics"].items()})
    with open("/proc/self/maps") as fh:
        out["native_so_loaded"] = "liballrank_b200.so" in fh.read()
    return out


def test_unmodified_main_run_config1_matches_the_reference_anchor(tmp_path):
    """FC[64] + listNet, batch 32, slate_length 120, Adam 1e-3, StepLR(3, 0.5), 4 epochs, seeds 42: the same seeded
    initialisation and the same data order => the GPU run follows the CPU reference's trajectory."""
    cpu = reference_result("baseline_cfg1")
    gpu = run_on_b200(tmp_path, "baseline_cfg1")
    assert gpu["native_so_loaded"]
    assert abs(cpu["val_metrics/ndcg_5"] - 0.5709) < 2e-3          # BASELINE.md anchor
    assert abs(gpu["val_metrics/ndcg_5"] - cpu["val_metrics/ndcg_5"]) < 1e-2, (gpu, cpu)
    assert abs(gpu["train_metrics/ndcg_5"] - cpu["train_metrics/ndcg_5"]) < 1e-2, (gpu, cpu)
    assert gpu["num_params"] == cpu["num_params"] == 1409
    assert gpu["epochs"] == cpu["epochs"]
    print("L3 cfg1: reference", cpu["val_metrics/ndcg_5"], "B200", gpu["val_metrics/ndcg_5"])


def test_unmodified_main_run_transformer_config_trains_like_the_reference(tmp_path):
    """Transformer(N=2, h=2) + approxNDCG with dropout 0.1, 6 epochs.  Dropout streams differ (counter hash vs
    Philox), so the final metrics agree within run-to-run noise, not bit for bit."""
    cpu = reference_result("transformer_cfg")
    gpu = run_on_b200(tmp_path, "transformer_cfg")
    assert gpu["native_so_loaded"]
    assert gpu["num_params"] == cpu["num_params"]
    for k in ("val_metrics/ndcg_5", "val_metrics/ndcg_10", "val_metrics/mrr_5"):
        assert abs(gpu[k] - cpu[k]) < 4e-2, (k, gpu[k], cpu[k])
    assert gpu["val_metrics/ndcg_5"] > 0.70
    print("L3 transformer: reference", cpu, "B200", gpu)
