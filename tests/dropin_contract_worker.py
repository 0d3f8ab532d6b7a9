"""Worker of tests/test_dropin_contract.py (own process: it replaces the kernels behind `mmrec_b200.ops` for its lifetime).

INTEGRATION.md section 2 claims that `mmrec_b200.models.FREEDOM` is a drop-in for the reference's model under the
reference's `quick_start` / `Trainer` / dataloaders.  This checks the claim without a GPU and without the reference: the
package's restatement of that harness (Config, RecDataset, TrainDataLoader, EvalDataLoader, Trainer) is built exactly as
`src/utils/quick_start.py:26-74` builds the reference's, the model class is OURS, and the kernels behind `mmrec_b200.ops` are
replaced by oracle-backed CPU stand-ins (test infrastructure: the product has no CPU path).  What the reference's harness
produced around the reference's own model -- its batches, losses and `Trainer.evaluate` metrics -- was recorded in
tests/golden (make_golden.py); `Trainer.evaluate` on the dense route (full_sort_predict -> in-place mask -> torch.topk ->
TopKEvaluator) must return those metrics, and one `calculate_loss` through `Trainer._train_epoch`'s call path must return
the recorded loss."""
import json
import os
import random
import sys
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
from conftest import load_golden  # noqa: E402


class CpuCSR:
    """Stand-in for ops.CSR: a coalesced torch sparse matrix on the CPU."""

    def __init__(self, t, symmetric=False):
        self.t_, self.n_rows, self.n_cols, self.nnz, self.symmetric = t, t.shape[0], t.shape[1], t._nnz(), symmetric

    @staticmethod
    def from_coo(row, col, val, n_rows, n_cols, sum_duplicates=True, symmetric=False, seg=None, light_max=None):
        val = torch.ones(row.numel(), dtype=torch.float32) if val is None else val.to(torch.float32)
        t = torch.sparse_coo_tensor(torch.stack([row.to(torch.int64), col.to(torch.int64)]), val, (n_rows, n_cols))
        return CpuCSR(t.coalesce() if sum_duplicates else t.coalesce(), symmetric)

    @staticmethod
    def from_torch_sparse(t, symmetric=False):
        return CpuCSR(t.coalesce(), symmetric)

    def coo(self):
        i = self.t_.indices()
        return i[0], i[1], self.t_.values()

    def t(self):
        return self if self.symmetric else CpuCSR(self.t_.t().coalesce())


def install_cpu_ops():
    from oracle import mmrec_oracle as O
    from mmrec_b200 import graph, ops
    ops.CSR = graph.CSR = CpuCSR
    ops.propagate_mean = lambda A, ego, n_layers: O.propagate_mean(A.t_, ego, n_layers)
    ops.spmm = lambda A, X, base=None: torch.sparse.mm(A.t_, X) if base is None else base + torch.sparse.mm(A.t_, X)
    ops.project = lambda table, weight, bias=None, idx=None, l2_normalize=False: O.project(table, weight, bias, idx=idx, l2_normalize=l2_normalize)
    ops.score = lambda u, i, users=None: O.full_sort_scores(u, i, users if users is not None else torch.arange(u.shape[0]))

    def mask_topk(scores, mask, k, item_offset=0):                    # graph._knn, Trainer.evaluate's dense route
        assert item_offset == 0
        if mask is not None:
            scores[mask[0], mask[1]] = -1e10                            # in place, as the reference's trainer.py:305-307
        return torch.topk(scores, k, dim=-1)
    ops.mask_topk = mask_topk

    def bipartite_norm(users, items, n_users, n_items, eps=1e-7):
        return O.normalize_adj_m(torch.stack([users, items]), n_users, n_items)
    ops.bipartite_norm = bipartite_norm

    # inference-only entry points (restated from their documented formulas in include/mmrec_b200.h)
    def spmm_raw(A, X, Y=None, acc_in=None, acc_out=None, acc_div=1.0, gate_ref=None, use_plan=True, y_accumulate=False):
        y = torch.sparse.mm(A.t_, X)
        if gate_ref is not None:
            y = torch.nn.functional.cosine_similarity(y, gate_ref, dim=-1).unsqueeze(1) * y
        if acc_out is not None:
            acc_out.copy_(((y if acc_in is None else acc_in + y)) / acc_div)
        if Y is not None:
            Y.copy_(Y + y if y_accumulate else y)
    ops.spmm_raw = spmm_raw

    def gate_rows(x, weight, bias, mul=None, out=None):
        r = torch.sigmoid(torch.nn.functional.linear(x, weight, bias))
        r = r if mul is None else mul * r
        return r if out is None else out.copy_(r)
    ops.gate_rows = gate_rows

    def mgcn_fuse(img, txt, content, q_w, q_b, q_w2, gi_w, gi_b, gt_w, gt_b, want_side=False):
        lin = torch.nn.functional.linear
        att = torch.cat([lin(torch.tanh(lin(img, q_w, q_b)), q_w2), lin(torch.tanh(lin(txt, q_w, q_b)), q_w2)], dim=-1)
        w = torch.softmax(att, dim=-1)
        common = w[:, 0].unsqueeze(1) * img + w[:, 1].unsqueeze(1) * txt
        side = (torch.sigmoid(lin(content, gi_w, gi_b)) * (img - common) + torch.sigmoid(lin(content, gt_w, gt_b)) * (txt - common) + common) / 3
        return (content + side, side) if want_side else content + side
    ops.mgcn_fuse = mgcn_fuse

    def propagate_layergcn(A, ego, n_layers):
        acc, x = torch.zeros_like(ego), ego
        for _ in range(n_layers):
            x = torch.sparse.mm(A.t_, x)
            x = torch.nn.functional.cosine_similarity(x, ego, dim=-1).unsqueeze(1) * x
            acc = acc + x
        return acc
    ops.propagate_layergcn = propagate_layergcn


def harness(name, over):
    """The tiny synthetic dataset on disk, then Config -> RecDataset -> loaders the way `src/utils/quick_start.py:26-74`
    builds them, with the seed set as it sets it; the CPU stand-ins are installed last.  Returns (config, train, valid,
    test, Trainer)."""
    from mmrec_b200.common.trainer import Trainer
    from mmrec_b200.utils import synth
    from mmrec_b200.utils.configurator import Config
    from mmrec_b200.utils.dataloader import EvalDataLoader, TrainDataLoader
    from mmrec_b200.utils.dataset import RecDataset
    from mmrec_b200.utils.utils import init_seed
    data = os.path.join(tempfile.mkdtemp(prefix="mmrec_contract_"), "data")
    u, i, e, d, f = synth.SHAPES["tiny"]
    g = synth.make_graph(u, i, e, seed=0)
    v, t = synth.make_features(i, f, seed=1)
    synth.write_dataset(data, "tiny", g, v, t)
    # the dense evaluation route (full_sort_predict -> mask -> top-k) of the reference's trainer: the stand-ins restate it
    config = Config(name, "tiny", dict({"data_path": data + "/", "gpu_id": 0, "use_gpu": False, "use_fused_topk": False}, **over))
    for k in config["hyper_parameters"]:
        if isinstance(config[k], list):
            config[k] = config[k][0]
    dataset = RecDataset(config)
    tr, va, te = dataset.split()
    train_data = TrainDataLoader(config, tr, batch_size=config["train_batch_size"], shuffle=True)
    valid_data = EvalDataLoader(config, va, additional_dataset=tr, batch_size=config["eval_batch_size"])
    test_data = EvalDataLoader(config, te, additional_dataset=tr, batch_size=config["eval_batch_size"])
    init_seed(config["seed"])
    train_data.pretrain_setup()
    install_cpu_ops()
    return config, train_data, valid_data, test_data, Trainer


def main():
    config, train_data, valid_data, test_data, Trainer = harness("FREEDOM", {"n_ui_layers": 3})
    # --- OUR model class, the way utils.get_model would return it from src/models/freedom.py (INTEGRATION.md section 2)
    from mmrec_b200.models.freedom import FREEDOM
    model = FREEDOM(config, train_data).to(config["device"])
    gold = load_golden("freedom_tiny.npz")
    sd = model.state_dict()
    init_identical = all(np.array_equal(sd[k[len("param0."):]].numpy(), gold[k]) for k in gold.files if k.startswith("param0."))
    trainer = Trainer(config, model)
    valid = trainer.evaluate(valid_data)
    test = trainer.evaluate(test_data, is_test=True)
    names = [str(x) for x in gold["metric_names"]]
    want_valid = dict(zip(names, [float(x) for x in gold["metric_values"]]))
    want_test = dict(zip(names, [float(x) for x in gold["test_metric_values"]]))
    # --- one loss through the call the reference's _train_epoch makes (src/common/trainer.py:147-153), on the recorded batch
    from mmrec_b200 import graph
    model.train()
    model.masked_adj = model.pruner.adj_from_keep(torch.from_numpy(gold["prune_keep_idx"]))
    loss = model.calculate_loss(torch.from_numpy(gold["batch"]))
    loss = sum(loss) if isinstance(loss, tuple) else loss
    loss.backward()                                                 # autograd-connected to the parameters (the optimiser steps on them)
    has_grads = all(p.grad is not None for p in model.parameters())
    out = {"init_identical": bool(init_identical), "valid": {k: float(v) for k, v in valid.items()}, "want_valid": want_valid,
           "test": {k: float(v) for k, v in test.items()}, "want_test": want_test, "loss": float(loss.item()),
           "want_loss": float(np.asarray(gold["loss"]).sum()), "has_grads": bool(has_grads)}
    print("CONTRACT " + json.dumps(out))


def main_mmgcn():
    """The same for MMGCN: OUR class (no torch_geometric needed) against tests/golden/mmgcn_tiny.npz, the reference's own
    model code run under a PyG shim (tests/golden/ref_loader.py)."""
    config, train_data, valid_data, _, Trainer = harness("MMGCN", {"eval_batch_size": 128, "train_batch_size": 512})
    from mmrec_b200.models.mmgcn import MMGCN
    model = MMGCN(config, train_data).to(config["device"])
    gold = load_golden("mmgcn_tiny.npz")
    sd = model.state_dict()
    init_identical = all(np.array_equal(sd[k[len("param0."):]].numpy(), gold[k]) for k in gold.files if k.startswith("param0.")) \
        and [k for k, _ in model.named_parameters()] == [str(x) for x in gold["param_order"]] \
        and np.array_equal(model.id_embedding.detach().numpy(), gold["id_embedding"]) \
        and np.array_equal(model.v_gcn.preference.detach().numpy(), gold["v_preference"]) \
        and np.array_equal(model.t_gcn.preference.detach().numpy(), gold["t_preference"])

    def rel(a, b):
        return float(np.linalg.norm(np.asarray(a, dtype=np.float64) - b) / np.linalg.norm(b))
    model.train()
    loss = model.calculate_loss(torch.from_numpy(gold["batch"]))
    loss.backward()
    grad_rel = max(rel(p.grad.numpy(), gold["grad." + k]) for k, p in model.named_parameters() if "grad." + k in gold.files)
    model.eval()
    with torch.no_grad():
        fwd_rel = rel(model.forward().numpy(), gold["fwd"])
        sc = model.full_sort_predict([torch.from_numpy(gold["eval_users"]), torch.from_numpy(gold["eval_mask"])])
        score_err = float(np.abs(sc.numpy() - gold["scores"]).max())
    valid = Trainer(config, model).evaluate(valid_data)
    names = [str(x) for x in gold["metric_names"]]
    out = {"init_identical": bool(init_identical), "fwd_rel": fwd_rel, "loss": float(loss.item()), "want_loss": float(gold["loss"][0]),
           "grad_rel": grad_rel, "score_err": score_err, "valid": {k: float(v) for k, v in valid.items()},
           "want_valid": dict(zip(names, [float(x) for x in gold["metric_values"]]))}
    print("CONTRACT " + json.dumps(out))


def main_model(name):
    """BM3 / MGCN / LightGCN / LayerGCN: our class against the golden file of the reference's own class -- initial
    weights, `forward`, the loss on the recorded batch WITH the reference's RNG draws (BM3's always-on dropout: same
    `torch.manual_seed(4321)` stream as tests/golden/make_golden.py), first-batch scores, `Trainer.evaluate`."""
    over = {"BM3": {}, "MGCN": {}, "LightGCN": {"n_layers": [3]}, "LayerGCN": {"dropout": [0.1]}}[name]
    config, train_data, valid_data, test_data, Trainer = harness(name, dict({"eval_batch_size": 128, "train_batch_size": 512}, **over))
    import importlib
    cls = getattr(importlib.import_module("mmrec_b200.models." + name.lower()), name)
    model = cls(config, train_data).to(config["device"])
    gold = load_golden(name.lower() + "_tiny.npz")
    sd = model.state_dict()
    init_identical = all(np.array_equal(sd[k[len("param0."):]].numpy(), gold[k]) for k in gold.files if k.startswith("param0.")) \
        and [k for k, _ in model.named_parameters()] == [str(x) for x in gold["param_order"]]

    def rel(a, b):
        return float(np.linalg.norm(np.asarray(a, dtype=np.float64) - b) / max(np.linalg.norm(b), 1e-30))
    model.eval()
    with torch.no_grad():
        if name == "MGCN":
            fu, fi = model.forward(model.norm_adj)                   # no autograd: the gate / fuse / stacked-table route (a5b)
        elif name == "LayerGCN":
            model.forward_adj = model.norm_adj_matrix
            fu, fi = model.forward()
        else:
            fu, fi = model.forward()
    fwd_rel = max(rel(fu.numpy(), gold["fwd_u"]), rel(fi.numpy(), gold["fwd_i"]))
    model.train()
    torch.manual_seed(1234)
    if name == "LayerGCN":
        model.masked_adj = model.pruner.adj_from_keep(torch.from_numpy(gold["prune_keep_idx"]))
    torch.manual_seed(4321)                                          # BM3's F.dropout draws, as in make_golden.py
    model.zero_grad()
    loss = model.calculate_loss(torch.from_numpy(gold["batch"]))
    loss = sum(loss) if isinstance(loss, tuple) else loss
    loss.backward()
    named = dict(model.named_parameters())
    gmax = max(float(np.abs(gold[k]).max()) for k in gold.files if k.startswith("grad."))
    grad_ok = all(np.linalg.norm(named[k[5:]].grad.numpy().astype(np.float64) - gold[k]) < 1e-4 * np.linalg.norm(gold[k]) + 1e-7 * gmax * np.sqrt(gold[k].size)
                  for k in gold.files if k.startswith("grad."))
    model.eval()
    with torch.no_grad():
        sc = model.full_sort_predict([torch.from_numpy(gold["eval_users"]), torch.from_numpy(gold["eval_mask"])])
    score_err = float(np.abs(sc.numpy() - gold["scores"]).max() / np.abs(gold["scores"]).max())
    trainer = Trainer(config, model)
    valid = trainer.evaluate(valid_data)
    test = trainer.evaluate(test_data, is_test=True)
    names = [str(x) for x in gold["metric_names"]]
    out = {"model": name, "init_identical": bool(init_identical), "fwd_rel": fwd_rel, "loss": float(loss.item()),
           "want_loss": float(np.asarray(gold["loss"]).sum()), "grad_ok": bool(grad_ok), "score_err": score_err,
           "valid": {k: float(v) for k, v in valid.items()}, "want_valid": dict(zip(names, [float(x) for x in gold["metric_values"]])),
           "test": {k: float(v) for k, v in test.items()}, "want_test": dict(zip(names, [float(x) for x in gold["test_metric_values"]]))}
    print("CONTRACT " + json.dumps(out))


def main_traj(name):
    """Two epochs of the reference's training loop as the package restates it (`Trainer._train_epoch`, torch's Adam, the
    scheduler, the dataloader's shuffling and negative sampling) driving OUR class, against the trajectory the reference's
    loop and class produced (tests/golden/traj_*_tiny.npz: every batch, every batch loss, per-epoch metrics)."""
    # key -> (model class, overrides of make_golden.py's dump_trajectory call, golden file)
    name, over, gfile = {"LightGCN": ("LightGCN", {"n_layers": [2], "reg_weight": [1e-4]}, "traj_lightgcn_tiny.npz"),
                         "FREEDOM": ("FREEDOM", {"dropout": [0.0], "reg_weight": [1e-3]}, "traj_freedom_tiny.npz"),
                         "FREEDOM-prune": ("FREEDOM", {"dropout": [0.8], "reg_weight": [1e-3]}, "traj_freedom_prune_tiny.npz"),
                         "LayerGCN": ("LayerGCN", {"dropout": [0.1]}, "traj_layergcn_tiny.npz"),
                         "BM3": ("BM3", {}, "traj_bm3_tiny.npz"),
                         "MGCN": ("MGCN", {}, "traj_mgcn_tiny.npz")}[name]
    config, train_data, valid_data, test_data, Trainer = harness(name, dict({"eval_batch_size": 128, "train_batch_size": 512}, **over))
    config["epochs"] = 2
    import importlib
    model = getattr(importlib.import_module("mmrec_b200.models." + name.lower()), name)(config, train_data).to(config["device"])
    gold = load_golden(gfile, os.environ.get("MMREC_TRAJ_DIR"))
    trainer = Trainer(config, model)
    rec = {"batches": [], "losses": [], "valid": [], "test": []}
    orig = model.calculate_loss

    def spy(interaction):
        rec["batches"].append(interaction.numpy().copy())
        l = orig(interaction)
        rec["losses"].append(float(sum(l)) if isinstance(l, tuple) else float(l))
        return l
    model.calculate_loss = spy
    # The package's loader draws negatives in numpy batches from a generator of its own, not one `random.sample` at a time
    # (mmrec_b200/utils/dataloader.py), so where negatives are sampled the epochs replay the batches the reference's loader
    # produced.  Without negatives (BM3) the loader must reproduce them itself.  The model's draws come from torch's
    # generator, which neither loader touches, except LayerGCN's uniform pruning: it draws from Python's `random` after the
    # reference's loader did, so each epoch starts from the state recorded there.
    epochs = [train_data, train_data]
    if config["use_neg_sampling"] is not False:
        ends = np.cumsum(gold["batch_sizes"])
        parts = [torch.from_numpy(np.ascontiguousarray(p)) for p in np.split(gold["batches"], ends[:-1], axis=1)]
        first = int(gold["batches_per_epoch"][0])
        epochs = [parts[:first], parts[first:]]
    for ep in range(2):
        if "py_random_state" in gold:
            random.setstate((3, tuple(int(x) for x in gold["py_random_state"][ep]), None))
        model.pre_epoch_processing()
        trainer._train_epoch(epochs[ep], ep)
        trainer.lr_scheduler.step()
        rec["valid"].append(list(trainer.evaluate(valid_data).values()))
        rec["test"].append(list(trainer.evaluate(test_data).values()))
    batches = np.concatenate(rec["batches"], axis=1)
    out = {"model": name, "same_batches": bool(batches.shape == gold["batches"].shape and np.array_equal(batches, gold["batches"])),
           "n_batches": len(rec["losses"]), "loss_max_rel": float(np.max(np.abs(np.array(rec["losses"]) - gold["losses"]) / np.abs(gold["losses"]))),
           "metric_max_abs": float(max(np.abs(np.array(rec["valid"]) - gold["valid"]).max(), np.abs(np.array(rec["test"]) - gold["test"]).max())),
           "first_loss": rec["losses"][0], "last_loss": rec["losses"][-1], "want_last_loss": float(gold["losses"][-1])}
    print("CONTRACT " + json.dumps(out))


if __name__ == "__main__":
    arg = sys.argv[1] if len(sys.argv) > 1 else ""
    if arg.startswith("traj:"):
        main_traj(arg[5:]); sys.exit(0)
    main_mmgcn() if arg == "mmgcn" else (main_model(arg) if arg else main())
