"""Oracle restatement of the reference's training driver (TEST INFRASTRUCTURE, see oracle/__init__.py):
allrank/main.py run() -> allrank/training/train_utils.py fit() on the reference's dummy data
(allrank/data/generate_dummy_data.py), with the model factory, the loss module and the epoch metrics passed in.

Given the reference's own make_model, losses and compute_metrics it returns exactly what the reference's run() writes
to experiment_result.json (oracle/make_golden.py: gen_l3 checks this before storing tests/golden/l3_reference.json);
tests/test_gpu_l3_training.py passes allrank_b200's and compares with that stored result.  Random streams are drawn in
the reference's order: torch / numpy seeds 42, the model's initialisation, then per epoch the shuffled train loader
(twice: training pass and train metrics) and the validation slates (FixLength samples a slate of exactly the
validation length, with numpy's global stream).
"""
import os
from collections import defaultdict
from functools import partial

import numpy as np
import torch
from torch.utils.data import DataLoader, Dataset

from . import slates_ref


def write_dummy_data(path, num_queries=100, results_len=20, num_labels=5, num_features=20):
    """generate_dummy_data.py run as a script: np.random.seed(42), train then vali, libsvm files under `path`."""
    from sklearn.datasets import dump_svmlight_file
    np.random.seed(42)
    os.makedirs(path, exist_ok=True)
    roles = []
    for role in ("train", "vali"):
        X = np.random.randn(num_queries * results_len, num_features)
        y = np.maximum(0, (((X + 1) / 2).mean(axis=-1) * num_labels).astype(np.int32))
        roles.append((role, X, y, np.repeat(np.arange(0, num_queries), results_len)))
    for role, X, y, qid in roles:
        dump_svmlight_file(X, y, os.path.join(path, role + ".txt"), query_id=qid)


class Slates(Dataset):
    """LibSVMDataset with Compose([FixLength(slate_length), ToTensor()]); slate_length None = the longest query."""

    def __init__(self, svm_file, slate_length=None):
        from sklearn.datasets import load_svmlight_file
        x, y, qid = load_svmlight_file(svm_file, query_id=True)
        off = slates_ref.group_offsets(qid)
        X = x.toarray()
        self.X = [X[a:b] for a, b in zip(off[:-1], off[1:])]
        self.y = [y[a:b] for a, b in zip(off[:-1], off[1:])]
        self.n_features = X.shape[-1]
        self.slate_length = int(slate_length or max(len(v) for v in self.y))

    def __len__(self):
        return len(self.y)

    def __getitem__(self, i):
        fx, fy, idx = slates_ref.fix_length(self.X[i], self.y[i], self.slate_length)
        return (torch.from_numpy(fx).type(torch.float32), torch.from_numpy(fy).type(torch.float32),
                torch.from_numpy(idx).type(torch.long))


def parse_metrics(names):
    """config.py _parse_metrics: ["ndcg_5", "ndcg_10", "mrr_5"] -> {"ndcg": [5, 10], "mrr": [5]}."""
    out = defaultdict(list)
    for s in names:
        name, at = s.split("_")
        out[name].append(int(at))
    return dict(out)


def loss_batch(model, loss_func, xb, yb, indices, opt=None):
    loss = loss_func(model(xb, yb == slates_ref.PAD_Y, indices), yb)
    if opt is not None:
        loss.backward()
        opt.step()
        opt.zero_grad()
    return loss.item(), len(xb)


def run(config, data_path, device, make_model, losses, compute_metrics):
    """main.run() + fit() for a config without gradient clipping or early stopping within its epochs; returns
    {"epochs", "train_metrics", "val_metrics", "num_params"} as the reference's experiment result holds them."""
    torch.manual_seed(42)
    torch.cuda.manual_seed_all(42)
    np.random.seed(42)
    data = config["data"]
    train_ds = Slates(os.path.join(data_path, "train.txt"), data["slate_length"])
    val_ds = Slates(os.path.join(data_path, data["validation_ds_role"] + ".txt"))
    train_dl = DataLoader(train_ds, batch_size=data["batch_size"], shuffle=True)
    val_dl = DataLoader(val_ds, batch_size=data["batch_size"], shuffle=False)
    model = make_model(n_features=train_ds.n_features, **config["model"]).to(device)
    optimizer = getattr(torch.optim, config["optimizer"]["name"])(params=model.parameters(),
                                                                  **config["optimizer"]["args"])
    loss_func = partial(getattr(losses, config["loss"]["name"]), **config["loss"]["args"])
    scheduler = getattr(torch.optim.lr_scheduler, config["lr_scheduler"]["name"])(optimizer,
                                                                                  **config["lr_scheduler"]["args"])
    metrics = parse_metrics(config["metrics"])
    num_params = int(sum(p.numel() for p in model.parameters() if p.requires_grad))
    for epoch in range(config["training"]["epochs"]):
        model.train()
        for xb, yb, indices in train_dl:
            loss_batch(model, loss_func, xb.to(device), yb.to(device), indices.to(device), optimizer)
        train_metrics = compute_metrics(metrics, model, train_dl, device)
        model.eval()
        with torch.no_grad():
            for xb, yb, indices in val_dl:
                loss_batch(model, loss_func, xb.to(device), yb.to(device), indices.to(device))
            val_metrics = compute_metrics(metrics, model, val_dl, device)
        scheduler.step()
    return {"epochs": epoch, "num_params": num_params,
            "train_metrics": {k: float(v) for k, v in train_metrics.items()},
            "val_metrics": {k: float(v) for k, v in val_metrics.items()}}
