"""Pin the CPU oracle against vectors produced by the unmodified reference (oracle/make_golden.py)."""
import ast

import numpy as np
import pytest
import torch

from oracle import losses_ref, metrics_ref, scorer_ref


def _loss_keys(golden):
    g = golden("losses")
    return list(g["keys"])


def test_losses_match_reference(golden):
    g = golden("losses")
    cases = [ast.literal_eval(str(c)) for c in g["cases"]]
    for key in g["keys"]:
        key = str(key)
        ci = int(key.split("_")[0][1:])
        name, kw = cases[ci]
        yp = torch.tensor(g[key + "_pred"]).requires_grad_(True)
        yt = torch.tensor(g[key + "_true"])
        val = losses_ref.LOSSES[name](yp, yt, **kw)
        if val.requires_grad:
            val.backward()
            grad = yp.grad.numpy()
        else:
            grad = np.zeros_like(g[key + "_grad32"])
        ref, gref = g[key + "_loss32"], g[key + "_grad32"]
        assert np.allclose(val.detach().numpy(), ref, rtol=2e-6, atol=1e-7), (key, name, kw, val.item(), ref)
        scale = max(np.abs(gref).max(), 1e-12)
        assert np.abs(grad - gref).max() <= 2e-5 * scale, (key, name, kw)


def test_listmle_matches_reference(golden):
    g = golden("listmle")
    for key in g["keys"]:
        key = str(key)
        yp = torch.tensor(g[key + "_pred"]).requires_grad_(True)
        yt = torch.tensor(g[key + "_true"])
        perm = torch.tensor(g[key + "_perm"])
        order = torch.tensor(g[key + "_order"])
        val = losses_ref.listMLE(yp, yt, perm=perm, order=order)
        val.backward()
        assert np.allclose(val.item(), g[key + "_loss32"], rtol=1e-6), key
        assert np.allclose(yp.grad.numpy(), g[key + "_grad32"], rtol=1e-5, atol=1e-7), key
        if key.endswith("distinct"):       # tie-free labels: any permutation gives the same value
            other = losses_ref.listMLE(yp.detach(), yt, perm=torch.arange(yt.shape[1]))
            assert np.allclose(other.item(), g[key + "_loss32"], rtol=2e-6), key


def test_metrics_match_reference_bit_exact(golden):
    g = golden("metrics")
    ats = [int(a) for a in g["ats"]]
    for key in g["keys"]:
        key = str(key)
        yp, yt = torch.tensor(g[key + "_pred"]), torch.tensor(g[key + "_true"])
        assert (metrics_ref.ranking(yp, yt).numpy() == g[key + "_order"]).all()
        assert np.array_equal(metrics_ref.ndcg(yp, yt, ats=ats).numpy(), g[key + "_ndcg"])
        assert np.array_equal(metrics_ref.dcg(yp, yt, ats=ats).numpy(), g[key + "_dcg"])
        assert np.array_equal(metrics_ref.mrr(yp, yt, ats=ats).numpy(), g[key + "_mrr"])
        assert np.array_equal(metrics_ref.ndcg(yp, yt).numpy(), g[key + "_ndcg_none"])
        assert np.array_equal(metrics_ref.dcg(yp, yt, ats=[3, 10], gain_function=lambda x: x).numpy(),
                              g[key + "_dcg_identity"])


def build_from_golden(g):
    meta = [int(v) for v in g["meta"]]
    F, d, N, h, dff = meta[:5]
    n_out = meta[7] if len(meta) > 7 else 1
    act = str(g["act"])
    model = scorer_ref.make_ref_model(F, [d], N, h, dff, d_output=n_out, output_activation=None if act == "None" else act)
    sd = {k[2:]: torch.tensor(g[k]) for k in g.files if k.startswith("p:")}
    assert set(sd) == set(model.state_dict()), "state_dict keys must equal the reference's"
    model.load_state_dict(sd)
    return model.eval()


@pytest.mark.parametrize("name", ["tiny", "mid", "cfg2"])
def test_scorer_matches_reference(golden, name):
    g = golden("scorer_" + name)
    model = build_from_golden(g)
    x, y = torch.tensor(g["x"]), torch.tensor(g["y"])
    mask = y == -1
    scores = model(x, mask, None)
    assert np.allclose(scores.detach().numpy(), g["scores"], rtol=1e-5, atol=2e-6)
    assert np.allclose(model.score(x, mask, None).detach().numpy(), g["scores"], rtol=1e-5, atol=2e-6)
    (scores * torch.tensor(g["w"])).sum().backward()
    for k, p in model.named_parameters():
        ref = g["g:" + k]
        assert np.abs(g.sampled(k, p.grad.numpy()) - ref).max() <= 1e-4 * max(np.abs(ref).max(), 1e-6), k


@pytest.mark.parametrize("name", ["dout4", "dout3_fc"])
def test_multi_output_scorer_matches_reference(golden, name):
    g = golden("scorer_" + name)
    model = build_from_golden(g)
    x, y = torch.tensor(g["x"]), torch.tensor(g["y"])
    mask = y == -1
    out = model(x, mask, None)
    assert out.shape == g["scores"].shape and out.dim() == 3
    assert np.allclose(out.detach().numpy(), g["scores"], rtol=1e-5, atol=2e-6)
    assert np.allclose(model.score(x, mask, None).detach().numpy(), g["score_sum"], rtol=1e-5, atol=4e-6)
    (out * torch.tensor(g["w"])).sum().backward()
    for k, p in model.named_parameters():
        ref = g["g:" + k]
        assert np.abs(p.grad.numpy() - ref).max() <= 1e-4 * max(np.abs(ref).max(), 1e-6), k


def test_ordinal_matches_reference(golden):
    g = golden("ordinal")
    for key in g["keys"]:
        key = str(key)
        n = int(key.split("_")[0][1:])
        yp = torch.tensor(g[key + "_pred"]).requires_grad_(True)
        yt = torch.tensor(g[key + "_true"])
        assert np.array_equal(losses_ref.with_ordinals(yt, n).numpy(), g[key + "_targets"]), key
        val = losses_ref.ordinal(yp, yt, n)
        val.backward()
        assert np.allclose(val.item(), g[key + "_loss32"], rtol=2e-6), key
        assert np.allclose(yp.grad.numpy(), g[key + "_grad32"], rtol=1e-5, atol=1e-7), key


def test_bce_matches_reference(golden):
    g = golden("bce")
    for key in g["keys"]:
        key = str(key)
        yp = torch.tensor(g[key + "_pred"]).requires_grad_(True)
        val = losses_ref.bce(yp, torch.tensor(g[key + "_true"]))
        val.backward()
        assert np.allclose(val.item(), g[key + "_loss32"], rtol=2e-6), key
        assert np.allclose(yp.grad.numpy(), g[key + "_grad32"], rtol=1e-5, atol=1e-7), key


@pytest.mark.parametrize("strategy", ["fixed", "learned"])
def test_scorer_with_positional_encoding_matches_reference(golden, strategy):
    g = golden("scorer_pe_" + strategy)
    F, d, N, h, dff, B, S, max_idx = [int(v) for v in g["meta"]]
    model = scorer_ref.make_ref_model(F, [d], N, h, dff, positional=(strategy, max_idx)).eval()
    sd = {k[2:]: torch.tensor(g[k]) for k in g.files if k.startswith("p:")}
    assert set(sd) == set(model.state_dict())
    model.load_state_dict(sd)
    x, y, idx = torch.tensor(g["x"]), torch.tensor(g["y"]), torch.tensor(g["idx"])
    scores = model(x, y == -1, idx)
    assert np.allclose(scores.detach().numpy(), g["scores"], rtol=1e-5, atol=2e-6)
    (scores * torch.tensor(g["w"])).sum().backward()
    for k, p in model.named_parameters():
        ref = g["g:" + k]
        assert np.abs(p.grad.numpy() - ref).max() <= 1e-4 * max(np.abs(ref).max(), 1e-6), k
