"""Generate the golden vectors under tests/golden/ by RUNNING THE REFERENCE ITSELF.

Run once in the build container (needs /root/reference; the GPU box only sees the
committed .npz files):

    python tests/golden/make_golden.py

The reference has no tests, fixtures or known-answer vectors of its own
(SURVEY.md section 4), so the pins are outputs of the unmodified reference code
(commit e775373) on the seeded synthetic graph `tiny` of
`mmrec_b200/utils/synth.py`, torch 2.11 CPU fp32, model seed 999
(`src/configs/overall.yaml:4`).  For every model the file holds: the train
interactions, every sparse matrix the model builds, the initial parameters, the
outputs of `forward`, `calculate_loss` (+ gradients) on a recorded batch,
`full_sort_predict` on the first eval batch, the `trainer.py:304-309` mask+top-50,
and the metrics of `Trainer.evaluate`; plus a 2-epoch training trajectory with the
batches the reference's own dataloader produced.
"""
import os
import sys
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))

import ref_loader  # noqa: E402
from conftest import save_golden  # noqa: E402
from mmrec_b200.utils import synth  # noqa: E402

DATASET = "tiny"


def coo_parts(t):
    return t._indices().numpy().copy(), t._values().detach().numpy().copy()


def build(model_name, overrides):
    from utils.configurator import Config
    from utils.dataset import RecDataset
    from utils.dataloader import TrainDataLoader, EvalDataLoader
    from utils.utils import init_seed, get_model
    cfg = {"gpu_id": 0, "use_gpu": False}
    cfg.update(overrides)
    config = Config(model_name, DATASET, cfg)
    # the dataset yaml for `tiny` does not exist in the reference: reuse baby's field names
    config["inter_file_name"] = f"{DATASET}.inter"
    config["USER_ID_FIELD"], config["ITEM_ID_FIELD"] = "userID", "itemID"
    config["vision_feature_file"], config["text_feature_file"] = "image_feat.npy", "text_feat.npy"
    # collapse grid-searched lists to their first element (SURVEY Appendix C)
    for k in config["hyper_parameters"]:
        v = config[k]
        if isinstance(v, list):
            config[k] = v[0]
    dataset = RecDataset(config)
    str(dataset)  # sets inter_num (dataset.py:115), needed by the dataloaders
    tr, va, te = dataset.split()
    str(tr), str(va), str(te)
    train_data = TrainDataLoader(config, tr, batch_size=config["train_batch_size"], shuffle=True)
    valid_data = EvalDataLoader(config, va, additional_dataset=tr, batch_size=config["eval_batch_size"])
    test_data = EvalDataLoader(config, te, additional_dataset=tr, batch_size=config["eval_batch_size"])
    init_seed(config["seed"])
    train_data.pretrain_setup()
    model = get_model(model_name)(config, train_data).to(config["device"])
    return config, train_data, valid_data, test_data, model


def dump_model(model_name, overrides, out):
    from common.trainer import Trainer
    config, train_data, valid_data, test_data, model = build(model_name, overrides)
    g = {}
    inter = train_data.inter_matrix(form="coo")
    g["inter_row"], g["inter_col"] = inter.row.astype(np.int64), inter.col.astype(np.int64)
    g["n_users"], g["n_items"] = np.int64(model.n_users), np.int64(model.n_items)
    for k in ("embedding_size", "n_layers", "n_ui_layers", "n_mm_layers", "knn_k", "mm_image_weight",
              "dropout", "reg_weight", "cl_weight", "cl_loss", "train_batch_size", "feat_embed_dim"):
        if config[k] is not None:
            g["cfg_" + k] = np.float64(config[k])
    # sparse matrices the model built in __init__
    for attr in ("norm_adj", "norm_adj_matrix", "mm_adj", "R", "image_original_adj", "text_original_adj"):
        t = getattr(model, attr, None)
        if t is not None and t.is_sparse:
            g[attr + "_idx"], g[attr + "_val"] = coo_parts(t)
    if hasattr(model, "edge_values"):
        g["edge_indices"], g["edge_values"] = model.edge_indices.numpy().copy(), model.edge_values.numpy().copy()
    for k, v in model.state_dict().items():
        g["param0." + k] = v.detach().numpy().copy()
    g["param_order"] = np.array([k for k, _ in model.named_parameters()])

    # per-epoch pruning (FREEDOM / LayerGCN): record the multinomial draw too
    torch.manual_seed(1234)
    if model_name in ("FREEDOM", "LayerGCN") and model.dropout > 0:
        ev = model.edge_values
        keep_len = int(ev.size(0) * (1.0 - model.dropout))
        st = torch.get_rng_state()
        g["prune_keep_idx"] = torch.multinomial(ev, keep_len).numpy().copy()
        torch.set_rng_state(st)
    model.pre_epoch_processing()
    if getattr(model, "masked_adj", None) is not None:
        g["masked_adj_idx"], g["masked_adj_val"] = coo_parts(model.masked_adj)

    # one training batch as the reference's dataloader emits it
    import random
    random.seed(7); np.random.seed(7)
    batch = next(iter(train_data))
    train_data.pr = 0
    g["batch"] = batch.numpy().copy()

    # forward outputs (eval graph)
    model.eval()
    with torch.no_grad():
        if model_name == "FREEDOM":
            u, i = model.forward(model.norm_adj)
            um, im = model.forward(model.masked_adj)
            g["fwd_masked_u"], g["fwd_masked_i"] = um.numpy().copy(), im.numpy().copy()
        elif model_name == "MGCN":
            u, i = model.forward(model.norm_adj)
        elif model_name == "LayerGCN":
            model.forward_adj = model.norm_adj_matrix
            u, i = model.forward()
        else:
            u, i = model.forward()
        g["fwd_u"], g["fwd_i"] = u.numpy().copy(), i.numpy().copy()
        if model_name in ("FREEDOM", "BM3", "MGCN"):
            g["proj_t"] = model.text_trs(model.text_embedding.weight).numpy().copy()
            g["proj_v"] = model.image_trs(model.image_embedding.weight).numpy().copy()

    # loss + gradients on the recorded batch
    model.train()
    torch.manual_seed(4321)  # BM3's F.dropout draws
    model.zero_grad()
    loss = model.calculate_loss(batch)
    if isinstance(loss, tuple):
        loss = sum(loss)
    loss.backward()
    g["loss"] = loss.detach().numpy().reshape(-1).copy()
    for k, p in model.named_parameters():
        if p.grad is not None and p.numel() <= 300 * 64:
            g["grad." + k] = p.grad.numpy().copy()
    model.zero_grad()

    # full_sort_predict + trainer mask/top-k on the first valid batch
    model.eval()
    with torch.no_grad():
        eb = next(iter(valid_data))
        valid_data.pr = 0; valid_data.inter_pr = 0
        scores = model.full_sort_predict(eb)
        g["eval_users"], g["eval_mask"] = eb[0].numpy().copy(), eb[1].numpy().copy()
        g["scores"] = scores.numpy().copy()
        scores[eb[1][0], eb[1][1]] = -1e10
        tv, ti = torch.topk(scores, max(config["topk"]), dim=-1)
        g["topk_idx"], g["topk_val"] = ti.numpy().copy(), tv.numpy().copy()
    g["eval_pos_items"] = np.array([np.asarray(x, dtype=np.int64) for x in valid_data.get_eval_items()], dtype=object)
    trainer = Trainer(config, model)
    res = trainer.evaluate(valid_data)
    g["metric_names"] = np.array(list(res.keys()))
    g["metric_values"] = np.array([res[k] for k in res], dtype=np.float64)
    g["test_metric_values"] = np.array([v for v in trainer.evaluate(test_data).values()], dtype=np.float64)
    g["test_eval_users"] = test_data.get_eval_users().numpy().copy()
    g["test_pos_items"] = np.array([np.asarray(x, dtype=np.int64) for x in test_data.get_eval_items()], dtype=object)

    # 2-epoch trajectory with recorded batches (device-RNG-free models only are replayable on GPU)
    if model_name in ("LightGCN", "FREEDOM0"):
        pass
    save_golden(out, g)
    print(f"{model_name}: wrote {out} ({os.path.getsize(out)/1024:.0f} KiB), valid={dict(zip(g['metric_names'][:4], g['metric_values'][:4]))}")
    return config, train_data, valid_data, test_data, model


def dump_mmgcn(overrides, out):
    """MMGCN: the reference's own model code under `ref_loader.install_pyg_shim()` (torch_geometric is absent; only its
    MessagePassing('mean') primitive and `inits.uniform` are restated there).  `id_embedding` / `preference` are plain
    tensors in the reference (`mmgcn.py:57,125`), recorded beside the state_dict."""
    from common.trainer import Trainer
    ref_loader.install_pyg_shim()
    config, train_data, valid_data, test_data, model = build("MMGCN", overrides)
    g = {"n_users": np.int64(model.n_users), "n_items": np.int64(model.n_items), "cfg_reg_weight": np.float64(config["reg_weight"]),
         "cfg_embedding_size": np.float64(config["embedding_size"])}
    g["edge_index"] = model.edge_index.numpy().copy()
    for k, v in model.state_dict().items():
        g["param0." + k] = v.detach().numpy().copy()
    g["param_order"] = np.array([k for k, _ in model.named_parameters()])
    g["id_embedding"] = model.id_embedding.detach().numpy().copy()
    g["v_preference"], g["t_preference"] = model.v_gcn.preference.detach().numpy().copy(), model.t_gcn.preference.detach().numpy().copy()
    g["v_feat"], g["t_feat"] = model.v_feat.numpy().copy(), model.t_feat.numpy().copy()
    import random
    random.seed(7); np.random.seed(7)
    batch = next(iter(train_data))
    train_data.pr = 0
    g["batch"] = batch.numpy().copy()
    model.train()
    model.zero_grad()
    loss = model.calculate_loss(batch)
    loss.backward()
    g["loss"] = loss.detach().numpy().reshape(-1).copy()
    for k, p_ in model.named_parameters():
        if p_.grad is not None and p_.numel() <= 300 * 64:
            g["grad." + k] = p_.grad.numpy().copy()
    g["grad.id_embedding"] = model.id_embedding.grad.numpy().copy()
    model.eval()
    with torch.no_grad():
        rep = model.forward()
        g["fwd"] = rep.numpy().copy()
        eb = next(iter(valid_data))
        valid_data.pr = 0; valid_data.inter_pr = 0
        scores = model.full_sort_predict(eb)
        g["eval_users"], g["eval_mask"] = eb[0].numpy().copy(), eb[1].numpy().copy()
        g["scores"] = scores.numpy().copy()
        scores[eb[1][0], eb[1][1]] = -1e10
        tv, ti = torch.topk(scores, max(config["topk"]), dim=-1)
        g["topk_idx"], g["topk_val"] = ti.numpy().copy(), tv.numpy().copy()
    res = Trainer(config, model).evaluate(valid_data)
    g["metric_names"] = np.array(list(res.keys()))
    g["metric_values"] = np.array([res[k] for k in res], dtype=np.float64)
    save_golden(out, g)
    print(f"MMGCN: wrote {out} ({os.path.getsize(out)/1024:.0f} KiB), loss {float(g['loss'][0]):.6f}")


def dump_trajectory(model_name, overrides, out, epochs=2, slim=False, py_random=False):
    """Train with the reference's own Trainer; record every batch, every batch loss, per-epoch metrics.  `py_random` also
    records the state of Python's `random` at the start of each epoch: the reference's loader draws its negatives from it,
    and LayerGCN's uniform pruning (`layergcn.py:56-58`) draws from it after them."""
    import random
    from common.trainer import Trainer
    config, train_data, valid_data, test_data, model = build(model_name, overrides)
    config["epochs"] = epochs
    trainer = Trainer(config, model)
    rec = {"batches": [], "losses": [], "valid": [], "test": []}
    orig = model.calculate_loss

    def spy(interaction):
        rec["batches"].append(interaction.numpy().copy())
        l = orig(interaction)
        rec["losses"].append(float(sum(l)) if isinstance(l, tuple) else float(l))
        return l

    model.calculate_loss = spy
    for k, p in model.state_dict().items():
        rec["param0." + k] = p.detach().numpy().copy()
    batch_epoch, py_states = [], []
    for ep in range(epochs):
        state = random.getstate()
        assert state[0] == 3 and state[2] is None
        py_states.append(state[1])
        model.pre_epoch_processing()
        n0 = len(rec["batches"])
        trainer._train_epoch(train_data, ep)
        trainer.lr_scheduler.step()
        batch_epoch.append(len(rec["batches"]) - n0)
        rec["valid"].append(list(trainer.evaluate(valid_data).values()))
        rec["test"].append(list(trainer.evaluate(test_data).values()))
    g = {} if slim else {k: v for k, v in rec.items() if k.startswith("param0.")}    # slim: batches / losses / metrics only
    g["batch_sizes"] = np.array([b.shape[1] for b in rec["batches"]])
    g["batches"] = np.concatenate(rec["batches"], axis=1)
    g["batches_per_epoch"] = np.array(batch_epoch)
    g["losses"] = np.array(rec["losses"], dtype=np.float64)
    g["valid"] = np.array(rec["valid"], dtype=np.float64)
    g["test"] = np.array(rec["test"], dtype=np.float64)
    g["metric_names"] = np.array(list(trainer.evaluate(valid_data).keys()))
    for k, p in model.state_dict().items():
        if p.numel() <= 300 * 64 and not slim:
            g["paramT." + k] = p.detach().numpy().copy()
    g["learning_rate"] = np.float64(config["learning_rate"])
    if py_random:
        g["py_random_state"] = np.array(py_states, dtype=np.int64)
    save_golden(out, g)
    print(f"trajectory {model_name}: {len(rec['losses'])} batches, loss {rec['losses'][0]:.6f} -> {rec['losses'][-1]:.6f}, "
          f"valid recall@20 {g['valid'][:, list(g['metric_names']).index('recall@20')]}")


def main():
    ref_loader.install()
    tmp = tempfile.mkdtemp(prefix="mmrec_golden_")
    data_root = ref_loader.run_dir(tmp)
    u, i, e, d, f = synth.SHAPES[DATASET]
    graph = synth.make_graph(u, i, e, seed=0)
    v, t = synth.make_features(i, f, seed=1)
    synth.write_dataset(data_root, DATASET, graph, v, t)
    np.savez_compressed(os.path.join(HERE, "tiny_graph.npz"), user=graph.user, item=graph.item, label=graph.label,
                        n_users=graph.n_users, n_items=graph.n_items)
    import logging
    logging.disable(logging.CRITICAL)
    # a tiny eval batch size so that several eval batches (ragged last one) are exercised
    common = {"eval_batch_size": 128, "train_batch_size": 512}
    dump_model("FREEDOM", dict(common, n_ui_layers=3), os.path.join(HERE, "freedom_tiny.npz"))
    for fcache in os.listdir(os.path.join(data_root, DATASET)):
        if fcache.endswith(".pt"):
            os.remove(os.path.join(data_root, DATASET, fcache))
    dump_model("BM3", common, os.path.join(HERE, "bm3_tiny.npz"))
    dump_model("MGCN", common, os.path.join(HERE, "mgcn_tiny.npz"))
    dump_model("LightGCN", dict(common, n_layers=[3]), os.path.join(HERE, "lightgcn_tiny.npz"))
    dump_model("LayerGCN", dict(common, dropout=[0.1]), os.path.join(HERE, "layergcn_tiny.npz"))
    dump_mmgcn(common, os.path.join(HERE, "mmgcn_tiny.npz"))
    dump_trajectory("LightGCN", dict(common, n_layers=[2], reg_weight=[1e-4]), os.path.join(HERE, "traj_lightgcn_tiny.npz"))
    dump_trajectory("FREEDOM", dict(common, dropout=[0.0], reg_weight=[1e-3]), os.path.join(HERE, "traj_freedom_tiny.npz"))
    # CPU contract trajectories (tests/test_dropin_contract.py): per-epoch pruning, dropout and the MGCN route in the loop
    dump_trajectory("FREEDOM", dict(common, dropout=[0.8], reg_weight=[1e-3]), os.path.join(HERE, "traj_freedom_prune_tiny.npz"), slim=True)
    for fcache in os.listdir(os.path.join(data_root, DATASET)):
        if fcache.endswith(".pt"):
            os.remove(os.path.join(data_root, DATASET, fcache))
    dump_trajectory("LayerGCN", dict(common, dropout=[0.1]), os.path.join(HERE, "traj_layergcn_tiny.npz"), slim=True,
                    py_random=True)
    dump_trajectory("BM3", common, os.path.join(HERE, "traj_bm3_tiny.npz"), slim=True)
    dump_trajectory("MGCN", common, os.path.join(HERE, "traj_mgcn_tiny.npz"), slim=True)


if __name__ == "__main__":
    main()
