"""Generate tests/golden/*.npz from the UNMODIFIED reference (run in the build container only).

    PYTHONDONTWRITEBYTECODE=1 python oracle/make_golden.py

Imports /root/reference/allrank behind oracle/_stubs (gcsfs / tensorboardX / flatten_dict are the
only missing deps) with CUDA hidden (model_utils.get_torch_device() hard-wires cuda:0), runs the
reference on seeded inputs and stores inputs + outputs.  /root/reference does not exist on the GPU
box, so tests only ever read the committed .npz files.
"""
import os
import sys

os.environ["CUDA_VISIBLE_DEVICES"] = ""
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path[:0] = [os.path.join(HERE, "_stubs"), "/root/reference", ROOT]
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402
import torch  # noqa: E402

from allrank.models import losses as ref_losses  # noqa: E402
from allrank.models import metrics as ref_metrics  # noqa: E402
from allrank.models.model import make_model as ref_make_model  # noqa: E402
from allrank.config import TransformerConfig, PositionalEncoding  # noqa: E402
from allrank_b200.synth import make_slates, make_scores  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
os.makedirs(OUT, exist_ok=True)

LOSS_CASES = [
    ("listNet", {}),
    ("approxNDCGLoss", {}),
    ("approxNDCGLoss", {"alpha": 2.5}),
    ("lambdaLoss", {}),
    ("lambdaLoss", {"weighing_scheme": "ndcgLoss1_scheme"}),
    ("lambdaLoss", {"weighing_scheme": "ndcgLoss2_scheme"}),
    ("lambdaLoss", {"weighing_scheme": "lambdaRank_scheme"}),
    ("lambdaLoss", {"weighing_scheme": "ndcgLoss2PP_scheme"}),
    ("lambdaLoss", {"weighing_scheme": "ndcgLoss2PP_scheme", "k": 10, "mu": 5.0, "sigma": 0.7}),
    ("lambdaLoss", {"weighing_scheme": "rankNet_scheme", "reduction_log": "natural", "reduction": "mean"}),
    ("lambdaLoss", {"weighing_scheme": "rankNetWeightedByGTDiff_scheme"}),
    ("lambdaLoss", {"weighing_scheme": "rankNetWeightedByGTDiffPowed_scheme", "k": 5}),
    ("neuralNDCG", {}),
    ("neuralNDCG", {"temperature": 0.1, "k": 10}),
    ("neuralNDCG", {"powered_relevancies": False, "temperature": 3.0}),
    ("neuralNDCG_transposed", {"temperature": 0.5, "k": 5}),
    ("neuralNDCG_transposed", {"max_iter": 20, "tol": 1e-4}),
    ("neuralNDCG_transposed", {"powered_relevancies": False}),
    ("rankNet", {}),
    ("rankNet_weightByGTDiff", {}),
    ("rankNet_weightByGTDiff_pow", {}),
    ("binary_listNet", {}),
    ("pointwise_rmse", {"no_of_levels": 4}),
]
SHAPES = [(5, 7), (4, 33), (3, 120), (3, 240)]


def case_inputs(b, s, seed):
    _, y, _ = make_slates(b, s, n_features=1, seed=seed)
    if s >= 33:
        y[0] = torch.where(y[0] >= 0, torch.zeros_like(y[0]), y[0])   # one slate without relevant items
    yp = make_scores(b, s, seed=seed + 7)
    return yp, y


def run_loss(fn, yp, y, kw, dtype):
    p = yp.to(dtype).clone().requires_grad_(True)
    val = fn(p, y.to(dtype), **kw)
    if val.requires_grad:
        val.backward()
        grad = p.grad
    else:
        grad = torch.zeros_like(p)
    return val.detach(), grad


def gen_losses():
    blob = {}
    names = []
    for ci, (name, kw) in enumerate(LOSS_CASES):
        fn = getattr(ref_losses, name)
        for (b, s) in SHAPES:
            if name.startswith("neuralNDCG") and s > 120:
                continue
            key = f"c{ci}_s{s}"
            yp, y = case_inputs(b, s, seed=100 * ci + s)
            v32, g32 = run_loss(fn, yp, y, kw, torch.float32)
            blob[key + "_pred"] = yp.numpy()
            blob[key + "_true"] = y.numpy()
            blob[key + "_loss32"] = v32.numpy()
            blob[key + "_grad32"] = g32.numpy()
            if not name.startswith("neuralNDCG"):   # reference neuralNDCG builds fp32 helpers internally; no fp64 run
                v64, g64 = run_loss(fn, yp, y, kw, torch.float64)
                blob[key + "_loss64"] = v64.numpy()
                blob[key + "_grad64"] = g64.numpy()
            names.append(key)
    blob["cases"] = np.array([repr(c) for c in LOSS_CASES])
    blob["keys"] = np.array(names)
    np.savez_compressed(os.path.join(OUT, "losses.npz"), **blob)
    print("losses:", len(names), "cases")


def gen_bce():
    """bce needs probabilities and (on torch >= 2) targets in [0,1]: unpadded slates, binary labels."""
    blob = {}
    keys = []
    for (b, s) in SHAPES:
        yp, y = case_inputs(b, s, seed=700 + s)
        yt = (y > 0).float()
        prob = torch.sigmoid(yp)
        p = prob.clone().requires_grad_(True)
        val = ref_losses.bce(p, yt)
        val.backward()
        key = f"s{s}"
        blob[key + "_pred"] = prob.numpy()
        blob[key + "_true"] = yt.numpy()
        blob[key + "_loss32"] = val.detach().numpy()
        blob[key + "_grad32"] = p.grad.numpy()
        keys.append(key)
    blob["keys"] = np.array(keys)
    np.savez_compressed(os.path.join(OUT, "bce.npz"), **blob)
    print("bce:", len(keys), "cases")


def gen_listmle():
    blob = {}
    keys = []
    for (b, s) in SHAPES:
        for tie_free in (True, False):
            yp, y = case_inputs(b, s, seed=900 + s)
            if tie_free:   # distinct labels -> value independent of the (unstable) tie order
                g = torch.Generator().manual_seed(s)
                distinct = torch.rand(b, s, generator=g) * 4.0
                y = torch.where(y >= 0, distinct, y)
            torch.manual_seed(4242 + s)
            state = torch.get_rng_state()
            perm = torch.randperm(s)              # what listMLE.py:17 will draw
            torch.set_rng_state(state)
            p = yp.clone().requires_grad_(True)
            val = ref_losses.listMLE(p, y)
            val.backward()
            order = y[:, perm].sort(descending=True, dim=-1).indices   # realised tie order on this host
            key = f"s{s}_{'distinct' if tie_free else 'ties'}"
            blob[key + "_pred"] = yp.numpy()
            blob[key + "_true"] = y.numpy()
            blob[key + "_perm"] = perm.numpy()
            blob[key + "_order"] = order.numpy()
            blob[key + "_loss32"] = val.detach().numpy()
            blob[key + "_grad32"] = p.grad.numpy()
            keys.append(key)
    blob["keys"] = np.array(keys)
    np.savez_compressed(os.path.join(OUT, "listmle.npz"), **blob)
    print("listMLE:", len(keys), "cases")


def gen_metrics():
    blob = {}
    keys = []
    ats = [1, 5, 10, 30, 60, 1000]
    for (b, s) in SHAPES + [(2, 1251)]:
        yp, y = case_inputs(b, s, seed=500 + s)
        key = f"s{s}"
        blob[key + "_pred"] = yp.numpy()
        blob[key + "_true"] = y.numpy()
        blob[key + "_ndcg"] = ref_metrics.ndcg(yp, y, ats=ats).numpy()
        blob[key + "_dcg"] = ref_metrics.dcg(yp, y, ats=ats).numpy()
        blob[key + "_mrr"] = ref_metrics.mrr(yp, y, ats=ats).numpy()
        blob[key + "_ndcg_none"] = ref_metrics.ndcg(yp, y).numpy()
        blob[key + "_dcg_identity"] = ref_metrics.dcg(yp, y, ats=[3, 10], gain_function=lambda x: x).numpy()
        masked = yp.clone()
        masked[y == -1] = float("-inf")
        blob[key + "_order"] = masked.sort(descending=True, dim=-1).indices.numpy()
        keys.append(key)
    blob["ats"] = np.array(ats)
    blob["keys"] = np.array(keys)
    np.savez_compressed(os.path.join(OUT, "metrics.npz"), **blob)
    print("metrics:", len(keys), "cases")


SCORER_CASES = {
    # name: (F, fc_sizes, N, h, d_ff, B, S, output_activation)
    "tiny": (20, [32], 1, 2, 64, 3, 20, None),
    "mid": (136, [64], 2, 2, 128, 2, 50, "Tanh"),
    "cfg2": (136, [128], 2, 4, 512, 2, 240, None),
}


def gen_scorer():
    for name, (F, sizes, N, h, dff, B, S, act) in SCORER_CASES.items():
        torch.manual_seed(7)
        model = ref_make_model(
            fc_model={"sizes": list(sizes), "input_norm": False, "activation": None, "dropout": 0.0},
            transformer=TransformerConfig(N=N, d_ff=dff, h=h, positional_encoding=None, dropout=0.0),
            post_model={"d_output": 1, "output_activation": act}, n_features=F)
        # perturb the norm gains/biases and linear biases so parity exercises them
        g = torch.Generator().manual_seed(11)
        with torch.no_grad():
            for n_, p in model.named_parameters():
                if p.dim() == 1:
                    p.add_(0.1 * torch.randn(p.shape, generator=g))
        model.eval()
        x, y, idx = make_slates(B, S, n_features=F, seed=31, mean_len=0.6 * S, std_len=0.3 * S)
        mask = y == -1
        scores = model(x, mask, idx)
        w = torch.randn(scores.shape, generator=g)
        (scores * w).sum().backward()
        blob = {"x": x.numpy(), "y": y.numpy(), "scores": scores.detach().numpy(), "w": w.numpy(),
                "meta": np.array([F, sizes[0], N, h, dff, B, S]), "act": np.array(str(act))}
        for k_, v in model.state_dict().items():
            blob["p:" + k_] = v.numpy()
        for k_, p in model.named_parameters():
            blob["g:" + k_] = p.grad.numpy().copy()
        # the same with the weight of the padded items zeroed ("gv:"): what a loss that masks padded items -- every loss
        # of allrank.models.losses -- sends back, and what the packed-rows layout of allrank_b200 reproduces
        model.zero_grad()
        (model(x, mask, idx) * (w * (~mask).float())).sum().backward()
        for k_, p in model.named_parameters():
            blob["gv:" + k_] = p.grad.numpy().copy()
        if sum(p.numel() for p in model.parameters()) > COMPACT_ABOVE_PARAMS:
            blob = compact_scorer_blob(blob, init_seed=7, perturb_seed=11, slates=(31, 0.6 * S, 0.3 * S))
        np.savez_compressed(os.path.join(OUT, f"scorer_{name}.npz"), **blob)
        print("scorer", name, "scores", tuple(scores.shape))


COMPACT_ABOVE_PARAMS = 100_000
GRAD_KEEP = 1024


def compact_scorer_blob(blob, init_seed, perturb_seed, slates):
    """Keep a golden scorer file small.  The parameters and the features are not stored: tests/conftest.py rebuilds
    the parameters with allrank_b200's make_model under torch.manual_seed(init_seed) -- the reference's seeded
    initialisation, pinned by tests/test_host_model.py -- and the 1-D shift drawn from perturb_seed, and the features
    with make_slates(seed, mean_len, std_len) = `slates` (both checked here).  A gradient of more than GRAD_KEEP
    entries is kept at GRAD_KEEP fixed, seeded flat positions, stored as gi:<name>."""
    from allrank_b200.model import make_model
    F, d, N, h, dff = [int(v) for v in blob["meta"][:5]]
    act = str(blob["act"])
    torch.manual_seed(init_seed)
    model = make_model(fc_model={"sizes": [d], "input_norm": False, "activation": None, "dropout": 0.0},
                       transformer={"N": N, "d_ff": dff, "h": h, "positional_encoding": None, "dropout": 0.0},
                       post_model={"d_output": 1, "output_activation": None if act == "None" else act}, n_features=F)
    perturb_vectors(model, perturb_seed)
    for k_, v in model.state_dict().items():
        assert np.array_equal(v.numpy(), blob.pop("p:" + k_)), k_
    B, S = [int(v) for v in blob["meta"][5:7]]
    x, y, _ = make_slates(B, S, n_features=F, seed=slates[0], mean_len=slates[1], std_len=slates[2])
    assert np.array_equal(x.numpy(), blob.pop("x")) and np.array_equal(y.numpy(), blob["y"])
    out = dict(blob, init_seed=np.array(init_seed), perturb_seed=np.array(perturb_seed), slates=np.array(slates))
    for k_, v in blob.items():
        if k_.startswith("g:") and v.size > GRAD_KEEP:
            name = k_[2:]
            idx = np.sort(np.random.RandomState(0).choice(v.size, GRAD_KEEP, replace=False)).astype(np.int32)
            out["gi:" + name] = idx
            out["g:" + name] = v.reshape(-1)[idx]
            out["gv:" + name] = blob["gv:" + name].reshape(-1)[idx]
    return out


def gen_scorer_pe():
    """Scorer with positional encodings (allrank/models/positional.py): fixed and learned, max_indices < slate length
    so that the index clipping to the padding row is exercised."""
    for strategy in ("fixed", "learned"):
        torch.manual_seed(9)
        F, d, N, h, dff, B, S, max_idx = 20, 32, 2, 2, 64, 3, 20, 15
        model = ref_make_model(
            fc_model={"sizes": [d], "input_norm": False, "activation": None, "dropout": 0.0},
            transformer=TransformerConfig(N=N, d_ff=dff, h=h, dropout=0.0,
                                          positional_encoding=PositionalEncoding(strategy=strategy, max_indices=max_idx)),
            post_model={"d_output": 1, "output_activation": None}, n_features=F)
        model.eval()
        x, y, idx = make_slates(B, S, n_features=F, seed=33, mean_len=0.7 * S, std_len=0.2 * S)
        g = torch.Generator().manual_seed(12)
        idx = torch.where(idx >= 0, torch.stack([torch.randperm(S, generator=g) for _ in range(B)]), idx)
        mask = y == -1
        scores = model(x, mask, idx)
        w = torch.randn(scores.shape, generator=g)
        (scores * w).sum().backward()
        blob = {"x": x.numpy(), "y": y.numpy(), "idx": idx.numpy(), "scores": scores.detach().numpy(), "w": w.numpy(),
                "meta": np.array([F, d, N, h, dff, B, S, max_idx])}
        for k_, v in model.state_dict().items():
            blob["p:" + k_] = v.numpy()
        for k_, p in model.named_parameters():
            blob["g:" + k_] = p.grad.numpy()
        np.savez_compressed(os.path.join(OUT, f"scorer_pe_{strategy}.npz"), **blob)
        print("scorer pe", strategy, [k_ for k_ in model.state_dict() if "position" in k_])


def gen_ordinal():
    """ordinal (ordinal.py:25-50) on per-level probabilities [B,S,n]; unpadded slates only -- on torch >= 2 the
    reference's nn.BCELoss rejects the -1 targets of padded items (its own padded test fails here)."""
    blob = {}
    keys = []
    for n in (2, 4):
        for (b, s) in SHAPES:
            _, y = case_inputs(b, s, seed=1100 + s + n)
            g = torch.Generator().manual_seed(s + n)
            y = torch.where(y < 0, torch.randint(0, 5, y.shape, generator=g).float(), y)   # fill the padding
            prob = torch.sigmoid(torch.randn(b, s, n, generator=g) * 2.0)
            p = prob.clone().requires_grad_(True)
            val = ref_losses.ordinal(p, y, n)
            val.backward()
            key = f"n{n}_s{s}"
            blob[key + "_pred"] = prob.numpy()
            blob[key + "_true"] = y.numpy()
            blob[key + "_targets"] = ref_losses.with_ordinals(y, n).numpy()
            blob[key + "_loss32"] = val.detach().numpy()
            blob[key + "_grad32"] = p.grad.numpy()
            keys.append(key)
    blob["keys"] = np.array(keys)
    np.savez_compressed(os.path.join(OUT, "ordinal.npz"), **blob)
    print("ordinal:", len(keys), "cases")


def gen_scorer_multi():
    """d_output > 1 heads (model.py:104-128; the ordinal configuration: Sigmoid over n levels), with and without
    the transformer; stores forward(), score() and parameter gradients."""
    cases = {"dout4": (20, 32, 1, 2, 64, 3, 20, 4, "Sigmoid"), "dout3_fc": (20, 32, 0, 0, 0, 3, 20, 3, None)}
    for name, (F, d, N, h, dff, B, S, n_out, act) in cases.items():
        torch.manual_seed(13)
        tr = TransformerConfig(N=N, d_ff=dff, h=h, positional_encoding=None, dropout=0.0) if N else None
        model = ref_make_model(
            fc_model={"sizes": [d], "input_norm": False, "activation": None, "dropout": 0.0},
            transformer=tr, post_model={"d_output": n_out, "output_activation": act}, n_features=F)
        g = torch.Generator().manual_seed(14)
        with torch.no_grad():
            for _, p in model.named_parameters():
                if p.dim() == 1:
                    p.add_(0.1 * torch.randn(p.shape, generator=g))
        model.eval()
        x, y, idx = make_slates(B, S, n_features=F, seed=35, mean_len=0.6 * S, std_len=0.3 * S)
        mask = y == -1
        out = model(x, mask, idx)
        w = torch.randn(out.shape, generator=g)
        (out * w).sum().backward()
        blob = {"x": x.numpy(), "y": y.numpy(), "scores": out.detach().numpy(), "w": w.numpy(),
                "score_sum": model.score(x, mask, idx).detach().numpy(),
                "meta": np.array([F, d, N, h, dff, B, S, n_out]), "act": np.array(str(act))}
        for k_, v in model.state_dict().items():
            blob["p:" + k_] = v.numpy()
        for k_, p in model.named_parameters():
            blob["g:" + k_] = p.grad.numpy()
        np.savez_compressed(os.path.join(OUT, f"scorer_{name}.npz"), **blob)
        print("scorer", name, "out", tuple(out.shape))


SHIPPED_CONFIGS = [
    "reproducibility/configs/contextaware_web30k/ndcgloss2pp.json",
    "reproducibility/configs/contextaware_web30k/ndcgloss2pp_mlp.json",
    "reproducibility/configs/contextaware_web30k/ordinal.json",
    "reproducibility/configs/contextaware_web30k/ordinal_mlp.json",
    "reproducibility/configs/neuralndcg_web30k/approxndcg.json",
    "reproducibility/configs/neuralndcg_web30k/lambdarank_atmax.json",
    "reproducibility/configs/neuralndcg_web30k/neuralndcg_atmax.json",
    "scripts/local_config.json",
]
GRAD_SAMPLES = 1024


def grad_sample_index(numel):
    """Deterministic positions at which the golden file keeps a parameter gradient (all of it when small)."""
    if numel <= GRAD_SAMPLES:
        return torch.arange(numel)
    return torch.linspace(0, numel - 1, GRAD_SAMPLES).long()


def perturb_vectors(model, seed):
    """Shift every 1-D parameter (biases, norm gains) so that parity exercises them; the tests repeat this."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for _, p in model.named_parameters():
            if p.dim() == 1:
                p.add_(0.1 * torch.randn(p.shape, generator=g))


def gen_scorer_shipped():
    """Every model configuration the reference ships (reproducibility/configs/*/*.json, scripts/local_config.json),
    built by the reference's make_model from the JSON's `model` section at MSLR shape (136 features, the config's
    slate length), eval mode.  Weights are NOT stored: a seeded init reproduces the reference's bit for bit
    (tests/test_host_model.py), so the file keeps the seed, the inputs, the scores and sampled parameter gradients."""
    import json
    F, B = 136, 2
    blob = {}
    names = []
    x, y, idx = make_slates(B, 240, n_features=F, seed=41, mean_len=150, std_len=60)
    mask = y == -1
    blob["x"], blob["y"] = x.numpy(), y.numpy()
    for rel in SHIPPED_CONFIGS:
        cfg = json.load(open(os.path.join("/root/reference", rel)))
        m = cfg["model"]
        name = os.path.splitext(os.path.basename(rel))[0]
        assert cfg["data"]["slate_length"] == 240
        torch.manual_seed(77)
        tr = m["transformer"]
        tcfg = None
        if tr:
            pe = tr.get("positional_encoding")
            tcfg = TransformerConfig(N=tr["N"], d_ff=tr["d_ff"], h=tr["h"], dropout=tr["dropout"],
                                     positional_encoding=PositionalEncoding(**pe) if pe else None)
        model = ref_make_model(fc_model=dict(m["fc_model"], sizes=list(m["fc_model"]["sizes"])), transformer=tcfg,
                               post_model=dict(m["post_model"]), n_features=F)
        perturb_vectors(model, 78)
        model.eval()
        for k_, v in model.state_dict().items():       # checksum of every tensor: pins the seeded initialisation
            blob[name + ":c:" + k_] = np.array([v.double().sum().item(), v.double().abs().sum().item()])
        out = model(x, mask, idx)
        w = torch.randn(out.shape, generator=torch.Generator().manual_seed(79))
        (out * w).sum().backward()
        blob[name + ":model"] = np.array(json.dumps(m))
        blob[name + ":loss"] = np.array(json.dumps(cfg["loss"]))
        blob[name + ":scores"] = out.detach().numpy()
        blob[name + ":w"] = w.numpy()
        for k_, p in model.named_parameters():
            gi = grad_sample_index(p.numel())
            blob[name + ":g:" + k_] = p.grad.flatten()[gi].numpy()
            blob[name + ":n:" + k_] = np.array(p.grad.norm().item())
        names.append(name)
        print("shipped", name, tuple(out.shape), sum(p.numel() for p in model.parameters()), "params")
    blob["names"] = np.array(names)
    np.savez_compressed(os.path.join(OUT, "scorer_shipped_configs.npz"), **blob)


def gen_neural_sort():
    """deterministic_neural_sort and sinkhorn_scaling themselves (loss_utils.py:34-67, :8-31), which no test of the
    reference pins in the tau = 1, 50-iteration regime of BASELINE config 4: P_hat before and after the scaling."""
    from allrank.models.losses.loss_utils import deterministic_neural_sort, sinkhorn_scaling
    blob = {}
    keys = []
    for (b, s_len, tau, iters, tol) in [(4, 7, 1.0, 50, 1e-6), (3, 33, 1.0, 50, 1e-6), (3, 120, 1.0, 50, 1e-6),
                                        (3, 120, 0.1, 50, 1e-6), (3, 64, 3.0, 20, 1e-6), (2, 128, 1.0, 50, 1e-6)]:
        yp, y = case_inputs(b, s_len, seed=2100 + s_len + int(10 * tau))
        if s_len >= 33:
            y[0] = torch.where(y[0] >= 0, torch.ones_like(y[0]), y[0])   # (case_inputs zeroes slate 0: give it relevance)
        mask = y == -1
        p0 = deterministic_neural_sort(yp.unsqueeze(-1), tau=tau, mask=mask)
        p = sinkhorn_scaling(p0, mask, tol=tol, max_iter=iters)
        key = f"s{s_len}_t{tau}_i{iters}"
        blob[key + "_pred"], blob[key + "_true"] = yp.numpy(), y.numpy()
        blob[key + "_p0"], blob[key + "_p"] = p0.numpy(), p.numpy()
        blob[key + "_args"] = np.array([tau, iters, tol])
        keys.append(key)
    blob["keys"] = np.array(keys)
    np.savez_compressed(os.path.join(OUT, "neural_sort.npz"), **blob)
    print("neural_sort:", keys)


def write_corpus(path, lengths, n_features, seed):
    """A small libsvm corpus (label qid:N f:v ...), query ids deliberately not sorted, a few all-zero-label queries
    and one query with a single relevant item."""
    rng = np.random.RandomState(seed)
    qids = rng.permutation(len(lengths)) + 3
    with open(path, "w") as f:
        for qi, n in enumerate(lengths):
            labels = rng.choice(5, size=n, p=[0.6, 0.2, 0.1, 0.06, 0.04])
            if qi % 5 == 1:
                labels[:] = 0
            if qi % 5 == 2:
                labels[:] = 0
                labels[rng.randint(n)] = 1
            for d in range(n):
                feats = rng.randn(n_features).round(4)
                feats[rng.rand(n_features) < 0.2] = 0.0          # sparse entries are simply absent in libsvm
                cols = " ".join(f"{j + 1}:{v}" for j, v in enumerate(feats) if v != 0.0)
                f.write(f"{labels[d]} qid:{qids[qi]} {cols}\n")


def gen_slates():
    """LibSVMDataset + FixLength on a small corpus (dataset_loading.py:32-165): padded slates, and sampled slates under
    np.random.seed so that the oracle (same numpy calls) can be pinned exactly."""
    from allrank.data.dataset_loading import LibSVMDataset, FixLength
    path = os.path.join(OUT, "slates_corpus.txt")
    lengths = [3, 17, 25, 8, 40, 12, 31, 20, 5, 64, 1, 22]
    write_corpus(path, lengths, n_features=12, seed=77)
    ds = LibSVMDataset.from_svm_file(path)
    blob = {"lengths": np.array([len(v) for v in ds.y_by_qid]), "shape": np.array(ds.shape)}
    S = 20
    fix = FixLength(S)
    for qi in range(len(ds)):
        np.random.seed(1000 + qi)
        x, y, idx = fix((ds.X_by_qid[qi], ds.y_by_qid[qi]))
        blob[f"q{qi}_x"], blob[f"q{qi}_y"], blob[f"q{qi}_idx"] = x.astype(np.float32), y.astype(np.float32), idx
    blob["slate_length"] = np.array(S)
    # the validation transform pads everything to the longest query (:185-192)
    longest = int(ds.longest_query_length)
    fix = FixLength(longest)
    for qi in range(len(ds)):
        if len(ds.y_by_qid[qi]) < longest:
            x, y, idx = fix((ds.X_by_qid[qi], ds.y_by_qid[qi]))
            blob[f"v{qi}_x"], blob[f"v{qi}_y"], blob[f"v{qi}_idx"] = x.astype(np.float32), y.astype(np.float32), idx
    np.savez_compressed(os.path.join(OUT, "slates.npz"), **blob)
    print("slates:", len(ds), "queries, longest", longest)


def gen_init():
    """Seeded initialisation of the reference's make_model (model.py:131-151): pins construction order."""
    torch.manual_seed(123)
    model = ref_make_model(
        fc_model={"sizes": [32], "input_norm": False, "activation": None, "dropout": 0.0},
        transformer=TransformerConfig(N=2, d_ff=64, h=2, positional_encoding=None, dropout=0.0),
        post_model={"d_output": 1, "output_activation": None}, n_features=20)
    blob = {"p:" + k_: v.numpy() for k_, v in model.state_dict().items()}
    np.savez_compressed(os.path.join(OUT, "init_seed123.npz"), **blob)
    print("init:", len(blob), "tensors")


def gen_l3():
    """The reference's own run() (oracle/run_reference_main.py, on the CPU) for the two training configs of
    tests/test_gpu_l3_training.py, checked against oracle/train_ref.py driving the reference's components."""
    import json
    import subprocess
    import tempfile
    from allrank.models.model import make_model
    from allrank.training.train_utils import compute_metrics
    from oracle import train_ref

    def ref_make_model(n_features, fc_model, transformer, post_model):
        return make_model(n_features=n_features, fc_model=fc_model, post_model=post_model,
                          transformer=TransformerConfig(**transformer) if transformer else None)

    out = {}
    for name in ("baseline_cfg1", "transformer_cfg"):
        config = os.path.join(ROOT, "tests", "configs", name + ".json")
        with tempfile.TemporaryDirectory() as tmp:
            r = subprocess.run([sys.executable, os.path.join(HERE, "run_reference_main.py"), "--workdir", tmp,
                                "--config", config, "--run-id", "cpu"], stdout=subprocess.PIPE, text=True, check=True)
            res = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("RESULT ")][-1][len("RESULT "):])
            res.pop("native_so_loaded")
            with open(config) as fh:
                port = train_ref.run(json.load(fh), os.path.join(tmp, "dummy_data"), torch.device("cpu"),
                                     ref_make_model, ref_losses, compute_metrics)
        flat = {"epochs": port["epochs"], "num_params": port["num_params"]}
        for role in ("train", "val"):
            flat.update({f"{role}_metrics/{k}": v for k, v in port[role + "_metrics"].items()})
        assert flat == res, (name, flat, res)
        out[name] = res
    with open(os.path.join(OUT, "l3_reference.json"), "w") as fh:
        json.dump(out, fh, indent=1, sort_keys=True)
    print("l3:", out)


def gen_reference_api():
    """Parameter names of the reference callables allrank_b200.integration rebinds, and the padding constants."""
    import inspect
    import json
    import allrank.data.dataset_loading as ref_dl
    from allrank_b200 import integration
    names = {"allrank.models.losses": integration.LOSS_NAMES, "allrank.models.metrics": integration.METRIC_NAMES,
             "allrank.models.model": ("make_model",),
             "allrank.training.train_utils": ("metric_on_batch", "metric_on_epoch", "compute_metrics"),
             "allrank.inference.inference_utils": ("rank_slates",),
             "allrank.data.dataset_loading": ("load_libsvm_dataset", "load_libsvm_dataset_role", "load_libsvm_role",
                                              "create_data_loaders"),
             "allrank.main": ("make_model", "load_libsvm_dataset", "create_data_loaders", "CustomDataParallel")}
    sig = {}
    for mod, fns in names.items():
        m = __import__(mod, fromlist=["_"])
        sig[mod] = {n: None if inspect.isclass(getattr(m, n)) else list(inspect.signature(getattr(m, n)).parameters)
                    for n in fns}
    consts = {"PADDED_Y_VALUE": ref_dl.PADDED_Y_VALUE, "PADDED_INDEX_VALUE": ref_dl.PADDED_INDEX_VALUE}
    with open(os.path.join(OUT, "reference_api.json"), "w") as fh:
        json.dump({"signatures": sig, "dataset_loading_constants": consts}, fh, indent=1)
    print("reference api:", sum(len(v) for v in sig.values()), "callables")


if __name__ == "__main__":
    torch.set_num_threads(4)
    gens = {"losses": gen_losses, "listmle": gen_listmle, "bce": gen_bce, "ordinal": gen_ordinal, "metrics": gen_metrics,
            "scorer": gen_scorer, "scorer_pe": gen_scorer_pe, "scorer_multi": gen_scorer_multi, "scorer_shipped": gen_scorer_shipped, "neural_sort": gen_neural_sort, "slates": gen_slates, "init": gen_init,
            "l3": gen_l3, "reference_api": gen_reference_api}
    for name in (sys.argv[1:] or list(gens)):      # optionally: only the named generators
        gens[name]()
