#!/usr/bin/env python
"""bench.py -- the hot path of MMRec on B200, measured per BASELINE.json.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --steps K --warmup W    # the reference's CPU algorithm (oracle port)

Workload (N=1): BASELINE.json configs[1] -- FREEDOM on the synthetic baby-shaped graph (20k users, 7k items,
160k train edges, d=64, 3 UI layers + 1 item-graph layer), then full-catalog scoring + mask + top-50 for every
user in batches of 4096 (`eval_batch_size`, src/configs/overall.yaml:45).  One step =
    [A] propagation   forward(norm_adj): 1 SpMM on mm_adj (fused `+h`) + 3 SpMMs on A_hat (fused layer mean)
    [B] projection    image/text Linear(4096->64) over the whole feature table (the calculate_loss form)
    [C] scoring       U x I scores + train-positive mask + top-50, all users
`value` = graph-prop edges/s = sum of nnz over the SpMMs of [A] / device time of [A]; the second half of the
metric (scored-items/s = users x items / device time of [C]) and the projection rate are in `extra`.
Timing: CUDA events on the launch stream around each section, L2 flushed (512 MiB write) before every step,
max over ranks.  `e2e` repeats [A] and [C] through the same public API with HOST buffers (pinned), copies inside
the timed region.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from mmrec_b200.utils import synth  # noqa: E402

TOPK = 50
EVAL_BATCH = 4096


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "src": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "src": "fallback (B200_PROFILING.md)"}


def ncu_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` from the committed ncu --set full capture
    (profiles/traffic.json, written by tools/summarize_ncu.py); None when no capture is recorded."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))[kernel]["dram_bytes_per_launch"]
    except Exception:
        return None


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed regions: NVML (the library nvidia-smi prints from) polled
    every 5 ms from a thread -- the device-only region of this workload lasts ~10 ms, shorter than one period of
    `nvidia-smi -lms`; falls back to the nvidia-smi loop when the NVML binding is missing."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.rows, self.proc, self.index, self.nvml, self.stop_flag = [], None, index, None, False

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            try:
                import torch
                pr = torch.cuda.get_device_properties(self.index)
                h = pynvml.nvmlDeviceGetHandleByPciBusId(f"{pr.pci_domain_id:08x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0".encode())
            except Exception:
                h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.nvml, self.h = pynvml, h
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _poll(self):
        n = self.nvml
        bits = (("hw_slowdown", getattr(n, "nvmlClocksEventReasonHwSlowdown", getattr(n, "nvmlClocksThrottleReasonHwSlowdown", 0x8))),
                ("hw_thermal_slowdown", getattr(n, "nvmlClocksEventReasonHwThermalSlowdown", getattr(n, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40))),
                ("sw_thermal_slowdown", getattr(n, "nvmlClocksEventReasonSwThermalSlowdown", getattr(n, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20))),
                ("sw_power_cap", getattr(n, "nvmlClocksEventReasonSwPowerCap", getattr(n, "nvmlClocksThrottleReasonSwPowerCap", 0x4))))
        get_reasons = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(n, "nvmlDeviceGetCurrentClocksThrottleReasons")
        while not self.stop_flag:
            try:
                sm = float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM))
                mask = int(get_reasons(self.h))
                self.rows.append((sm, [name for name, b in bits if mask & b]))
            except Exception:
                pass
            time.sleep(0.005)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.nvml:
            self.stop_flag = True
            self.t.join(timeout=1)
            if not self.rows:
                return None
            reasons = sorted({r for _, rs in self.rows for r in rs})
            return {"sm_mhz": float(np.median([sm for sm, _ in self.rows])), "sm_max_mhz": self.mx, "reasons": reasons,
                    "samples": len(self.rows), "source": "nvml, 5 ms period"}
        if not self.proc:
            return None
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        if not sm:
            return None
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm),
                "source": "nvidia-smi -lms 50"}


# ------------------------------------------------------------------------------------------------------
# workload
# ------------------------------------------------------------------------------------------------------
MODEL_OF = {"baby": "FREEDOM", "small": "FREEDOM", "tiny": "FREEDOM", "sports": "BM3", "clothing": "MGCN"}   # BASELINE.json configs[1..3]
KNN_K = 10


class Workload:
    def __init__(self, name, n_layers=3, seed=0, items_scale=1):
        self.name = name
        U, I, E, d, F = synth.SHAPES[name]
        self.g = synth.make_graph(U, I * items_scale, E * items_scale, seed)
        self.U, self.I, self.d, self.F = U, I * items_scale, d, F
        self.n_layers = n_layers
        self.tr_u, self.tr_i = self.g.train
        rng = np.random.default_rng(7)
        bound = np.sqrt(6.0 / (self.U + d))                       # xavier_uniform, freedom.py:51-52
        self.user_emb = rng.uniform(-bound, bound, (self.U, d)).astype(np.float32)
        bound = np.sqrt(6.0 / (self.I + d))
        self.item_emb = rng.uniform(-bound, bound, (self.I, d)).astype(np.float32)

    def features(self):
        """(image, text) feature tables, fp32 [I, F] each (SURVEY.md Appendix C)."""
        return synth.make_features(self.I, self.F, seed=1)

    def knn_coo(self, k=KNN_K, seed=3):
        """Synthetic stand-in for FREEDOM's mm_adj at the scaled (N-GPU) sizes, where the dense I x I similarity is
        skipped: k random neighbours per item from each modality, 0.1/0.9 weights (freedom.py:74)."""
        rng = np.random.default_rng(seed)
        rows = np.repeat(np.arange(self.I), k)
        c1, c2 = rng.integers(0, self.I, self.I * k), rng.integers(0, self.I, self.I * k)
        w = np.float32(np.float32(1.0 / np.sqrt(np.float32(k))) ** 2)
        return (np.concatenate([rows, rows]), np.concatenate([c1, c2]),
                np.concatenate([np.full(self.I * k, 0.1 * w, np.float32), np.full(self.I * k, 0.9 * w, np.float32)]))

    def eval_mask(self, lo, hi):
        m = (self.tr_u >= lo) & (self.tr_u < hi)
        order = np.argsort(self.tr_u[m], kind="stable")
        return np.stack([self.tr_u[m][order] - lo, self.tr_i[m][order]])

    def describe(self, model, n_ui, n_mm):
        return (f"{model} synthetic {self.name}: {self.U} users, {self.I} items, {len(self.tr_u)} train edges, d={self.d}, "
                f"{n_ui} UI layers + {n_mm} mm layer (cosine kNN, k={KNN_K} per modality, of the N(0,1) feature tables), "
                f"top-{TOPK} over all users")


def build_model(wl, model_name, dev, overrides=None):
    """The plugin boundary: the dataset on disk in the reference's format, then Config -> RecDataset -> loaders -> model
    class, exactly the way `quick_start` builds them (src/utils/quick_start.py:26-74)."""
    import tempfile
    from mmrec_b200.utils.configurator import Config
    from mmrec_b200.utils.dataloader import EvalDataLoader, TrainDataLoader
    from mmrec_b200.utils.dataset import RecDataset
    from mmrec_b200.utils.utils import get_model, init_seed
    tmp = tempfile.mkdtemp(prefix="mmrec_bench_")
    v, t = wl.features()
    synth.write_dataset(os.path.join(tmp, "data"), wl.name, wl.g, v, t)
    cfg = {"data_path": os.path.join(tmp, "data") + "/", "eval_batch_size": EVAL_BATCH, "use_gpu": True, "gpu_id": dev.index or 0}
    cfg.update(overrides or {})
    config = Config(model_name, wl.name, cfg)
    for key in config["hyper_parameters"]:
        if isinstance(config[key], list):
            config[key] = config[key][0]
    config["device"] = dev
    ds = RecDataset(config)
    tr, va, te = ds.split()
    train = TrainDataLoader(config, tr, batch_size=config["train_batch_size"], shuffle=True)
    test = EvalDataLoader(config, te, additional_dataset=tr, batch_size=config["eval_batch_size"])
    init_seed(config["seed"])
    train.pretrain_setup()
    model = get_model(model_name)(config, train).to(dev)
    import shutil
    shutil.rmtree(tmp, ignore_errors=True)
    return config, train, test, model


def model_graphs(model):
    """(name, CSR, applications per forward) of the sparse matrices one `forward` of the model multiplies by."""
    name = type(model).__name__
    if name == "FREEDOM":
        return [("norm_adj", model.norm_adj, model.n_ui_layers), ("mm_adj", model.mm_adj, model.n_layers)]
    if name == "BM3":
        return [("norm_adj", model.norm_adj, model.n_layers)]
    if name == "MGCN":
        return [("norm_adj", model.norm_adj, model.n_ui_layers), ("image_adj", model.image_original_adj, model.n_layers),
                ("text_adj", model.text_original_adj, model.n_layers), ("R", model.R, 2)]
    return [("norm_adj", model.norm_adj, getattr(model, "n_layers", 1))]


def forward_eval(model):
    name = type(model).__name__
    if name in ("FREEDOM", "MGCN"):
        return model.forward(model.norm_adj)
    return model.forward()


DUMP_BYTES = 64 << 20
DUMP_NAMES = {"a": "propagation", "b": "projection", "c": "topk_items", "c4096": "topk_items_batch4096"}


def dump_outputs(dump_dir, outs):
    """Write what each timed section returned to its caller as <dump_dir>/<name>.npy: `model.forward` -> propagation_<k>
    (k-th returned tensor, user then item embeddings), the two modality projections -> projection_<k>, `full_sort_topk` of
    all users -> topk_items, and of the 4096-user batches -> topk_items_batch4096 (the batches stacked).  Embeddings are
    written as float32, item indices as float64 (exact).  When together they exceed 64 MiB, each array bigger than its share
    keeps a fixed seeded sample of its rows, whose row numbers go to <name>.rows.npy."""
    arrays = {}
    for sec, out in outs.items():
        if sec == "c4096":
            arrays[DUMP_NAMES[sec]] = torch.cat(out)
        elif torch.is_tensor(out):
            arrays[DUMP_NAMES[sec]] = out
        else:
            arrays.update((f"{DUMP_NAMES[sec]}_{k}", t) for k, t in enumerate(out) if torch.is_tensor(t))
    os.makedirs(dump_dir, exist_ok=True)
    arrays = {k: t.detach().cpu().numpy() for k, t in arrays.items()}
    arrays = {k: a.astype(np.float64 if a.dtype.kind in "iu" else np.float32) for k, a in arrays.items()}
    share = DUMP_BYTES // (2 * len(arrays))                          # the other half bounds the row lists
    sample = sum(a.nbytes for a in arrays.values()) > DUMP_BYTES
    for name, a in arrays.items():
        if sample and a.nbytes > share:
            rows = np.sort(np.random.default_rng(0).choice(a.shape[0], share // a[0].nbytes, replace=False))
            np.save(os.path.join(dump_dir, name + ".rows.npy"), rows.astype(np.float64))
            a = a[rows]
        np.save(os.path.join(dump_dir, name + ".npy"), a)


def torch_gpu_comparator(model, u_users, batches_dev, flush, reps=5):
    """The reference's own formulation on the same GPU with stock PyTorch kernels -- un-coalesced COO adjacency through
    `torch.sparse.mm` per layer + `stack().mean()` (`src/models/freedom.py:164-178`), `matmul` + in-place mask +
    `torch.topk` (`freedom.py:216-220`, `src/common/trainer.py:304-309`) -- timed with CUDA events.  This is the
    "vs torch.sparse.mm" comparator BASELINE.json's config 2 names; it is context for the speed-up, not the product."""
    dev = model.user_embedding.weight.device
    U, I = model.n_users, model.n_items
    r, c, v = model.norm_adj.coo()
    adj = torch.sparse_coo_tensor(torch.stack([r, c]), v, (U + I, U + I))           # (un-coalesced flag, like the reference's)
    r, c, v = model.mm_adj.coo()
    mm = torch.sparse_coo_tensor(torch.stack([r, c]), v, (I, I))
    ego = torch.cat((model.user_embedding.weight, model.item_id_embedding.weight), dim=0).detach()
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def prop():
        h = torch.sparse.mm(mm, ego[U:])
        e, outs = ego, [ego]
        for _ in range(model.n_ui_layers):
            e = torch.sparse.mm(adj, e)
            outs.append(e)
        a = torch.stack(outs, dim=1).mean(dim=1)
        return a[:U], a[U:] + h

    def score(u_g, i_g):
        for users, mask in batches_dev:
            s = torch.matmul(u_g[users], i_g.t())
            s[mask[0], mask[1]] = -1e10
            torch.topk(s, TOPK, dim=-1)

    tA = tC = 0.0
    with torch.no_grad():
        for it in range(reps + 2):
            flush.zero_()
            e = [ev() for _ in range(4)]
            e[0].record(); u_g, i_g = prop(); e[1].record()
            e[2].record(); score(u_g, i_g); e[3].record()
            torch.cuda.synchronize()
            if it >= 2:
                tA += e[0].elapsed_time(e[1]); tC += e[2].elapsed_time(e[3])
    edges = model.n_ui_layers * adj._nnz() + mm._nnz()
    return {"what": "reference formulation with stock torch CUDA ops on this GPU (torch.sparse.mm on the un-coalesced COO, matmul + mask + "
                    "torch.topk, eval batch 4096), eager", "edges_per_sec": edges / (tA / reps * 1e-3), "prop_ms": tA / reps,
            "scored_items_per_sec": U * I / (tC / reps * 1e-3), "score_topk_ms": tC / reps}


# ------------------------------------------------------------------------------------------------------
# this repo's arm
# ------------------------------------------------------------------------------------------------------
def bench_model(wl, model_name, dev, args, flush, sampler=None, full=True, dump_dir=None):
    """One model on one workload through the model-class API.  Device-timed sections (CUDA events, each section replayed
    from a CUDA graph -- kernels of 5-70 us are shorter than a Python call --, L2 flushed before every step):
        [A] `model.forward(...)`                       propagation, the plugin call of calculate_loss / full_sort_predict
        [B] both modality projections over the whole table (ops.project on the model's tables; FREEDOM only)
        [C] `model.full_sort_topk([users, mask], 50)`  scoring + mask + top-50 of ALL users in one call
        [C4096] the same in the reference's default eval batches of 4096 users (src/configs/overall.yaml:45)
    and the end-to-end forms with pinned HOST buffers and the copies inside the timed region."""
    from mmrec_b200 import ops
    config, train, test, model = build_model(wl, model_name, dev, {"n_ui_layers": wl.n_layers} if model_name == "FREEDOM" else None)
    model.eval()
    U, I, d = model.n_users, model.n_items, wl.d
    graphs_info = model_graphs(model)
    edges = sum(g.nnz * reps for _, g, reps in graphs_info)
    spmm_bytes = sum(g.algorithmic_bytes(d) * reps for _, g, reps in graphs_info)
    score_items, score_flops = U * I, 2 * U * I * d
    all_users = torch.arange(U, device=dev)
    mask_all_h = torch.from_numpy(wl.eval_mask(0, U))
    mask_all = mask_all_h.to(dev)
    batches_h = []
    for lo in range(0, U, EVAL_BATCH):
        hi = min(U, lo + EVAL_BATCH)
        batches_h.append((torch.arange(lo, hi).pin_memory(), torch.from_numpy(wl.eval_mask(lo, hi)).pin_memory()))
    batches_dev = [(u.to(dev), m.to(dev)) for u, m in batches_h]
    has_proj = model_name == "FREEDOM" and full
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def sec_a():
        return forward_eval(model)

    def sec_b():
        return (ops.project(model.image_embedding.weight, model.image_trs.weight, model.image_trs.bias),
                ops.project(model.text_embedding.weight, model.text_trs.weight, model.text_trs.bias))

    def sec_c():
        return model.full_sort_topk([all_users, mask_all], TOPK)

    def sec_c4096():
        return [model.full_sort_topk([u, m], TOPK) for u, m in batches_dev]

    secs = [("a", sec_a)] + ([("b", sec_b)] if has_proj else []) + [("c", sec_c), ("c4096", sec_c4096)]
    graphs, n_launch = {}, {}
    side = torch.cuda.Stream()
    with torch.cuda.stream(side), torch.no_grad():
        for _ in range(2):                                           # warm every lazy init (occupancy queries, workspaces, eval cache)
            for _, fn in secs:
                fn()
        torch.cuda.synchronize()
        for name, fn in secs:
            l0 = ops.launch_count()
            gph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gph, stream=side):
                out = fn()
            graphs[name], n_launch[name] = (gph, out), ops.launch_count() - l0
    torch.cuda.synchronize()
    times = {name: 0.0 for name, _ in secs}
    steps, warm = args.steps, args.warmup
    with torch.no_grad():
        for step in range(warm + steps):
            if step == 0 and sampler is not None:
                sampler.start()
            flush.zero_()                                            # evict L2 (126 MB) between steps
            marks = []
            for name, _ in secs:
                e0, e1 = ev(), ev()
                e0.record(); graphs[name][0].replay(); e1.record()
                marks.append((name, e0, e1))
            torch.cuda.synchronize()
            if step >= warm:
                for name, e0, e1 in marks:
                    times[name] += e0.elapsed_time(e1)
    ms = {k: v / steps for k, v in times.items()}
    launches = sum(n_launch[k] for k in n_launch if k != "c4096") * steps      # (the 4096-batch variant is an extra, not part of the step)
    if dump_dir:                                                     # each replay rewrote the captured outputs: the last step's
        dump_outputs(dump_dir, {name: graphs[name][1] for name, _ in secs})

    # ---- e2e through the same model calls, HOST buffers (pinned), copies inside the timed region.  [A]: the embedding
    # tables arrive from the host (a checkpoint / parameter-server push), forward, both outputs back.  [C]: the evaluation
    # batch arrives from the host (what the loader does when the data is not device-resident), full_sort_topk, the index
    # matrix goes back to the evaluator.  Each is captured once into a CUDA graph (copies included) and replayed.
    emb_params = [p for n, p in model.named_parameters() if "embedding" in n and p.shape[1] == d]
    host_params = [p.detach().cpu().pin_memory() for p in emb_params]
    out_u = torch.empty(U, d).pin_memory(); out_i = torch.empty(I, d).pin_memory()
    users_h = torch.arange(U).pin_memory(); mask_h = mask_all_h.pin_memory()
    out_idx = torch.empty(U, TOPK, dtype=torch.int64).pin_memory()

    def e2e_a():
        for p, h in zip(emb_params, host_params):
            p.data.copy_(h, non_blocking=True)
        model.invalidate_eval_cache()
        u_g, i_g = forward_eval(model)
        out_u.copy_(u_g, non_blocking=True); out_i.copy_(i_g, non_blocking=True)

    def e2e_c():
        inter = [users_h.to(dev, non_blocking=True), mask_h.to(dev, non_blocking=True)]
        out_idx.copy_(model.full_sort_topk(inter, TOPK), non_blocking=True)

    e2e_graphs, e2e_mode = {}, "cuda graph replay (pinned H2D/D2H copies inside the graph)"
    with torch.cuda.stream(side), torch.no_grad():
        e2e_a(); e2e_c()
        torch.cuda.synchronize()
        try:
            for name, fn in (("c", e2e_c), ("a", e2e_a)):                # ("c" first: its capture must see the cached embeddings, "a" drops them)
                gph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(gph, stream=side):
                    fn()
                e2e_graphs[name] = gph
            torch.cuda.synchronize()
        except Exception as exc:                                     # noqa: BLE001
            e2e_graphs, e2e_mode = {}, f"eager ({type(exc).__name__} during graph capture)"
            torch.cuda.synchronize()
    eA = eC = 0.0
    with torch.no_grad():
        for step in range(warm + steps):
            flush.zero_()
            e = [ev() for _ in range(4)]
            e[0].record(); (e2e_graphs["a"].replay() if e2e_graphs else e2e_a()); e[1].record()
            e[2].record(); (e2e_graphs["c"].replay() if e2e_graphs else e2e_c()); e[3].record()
            torch.cuda.synchronize()
            if step >= warm:
                eA += e[0].elapsed_time(e[1]); eC += e[2].elapsed_time(e[3])
    clocks = sampler.stop() if sampler is not None else None
    h2d = sum(h.numel() * 4 for h in host_params) + users_h.numel() * 8 + mask_h.numel() * 8
    d2h = (out_u.numel() + out_i.numel()) * 4 + out_idx.numel() * 8
    res = {"model": model_name, "workload": wl.describe(model_name, *(graphs_info[0][2], graphs_info[1][2] if len(graphs_info) > 1 else 0)),
           "edges_per_step": edges, "spmm_bytes": spmm_bytes, "ms": ms, "launches": launches, "clocks": clocks,
           "e2e": {"prop_ms": eA / steps, "score_topk_ms": eC / steps, "h2d": int(h2d), "d2h": int(d2h), "mode": e2e_mode},
           "score_items": score_items, "score_flops": score_flops, "ui_bytes": graphs_info[0][1].algorithmic_bytes(d),
           "proj_bytes": 2 * (4 * I * wl.F + 4 * d * wl.F + 4 * I * d), "proj_flops": 2 * 2 * I * wl.F * d}
    if full:
        # one training step through the plugin calls: calculate_loss + backward + Adam (src/common/trainer.py:147-189)
        try:
            from mmrec_b200.common.trainer import Trainer

            def time_train(trainer):
                model.train(); model.pre_epoch_processing()
                it = iter(train)
                ts = []
                for i in range(8):
                    batch = next(it)
                    e0, e1 = ev(), ev()
                    e0.record()
                    trainer.optimizer.zero_grad()
                    loss = model.calculate_loss(batch)
                    loss = sum(loss) if isinstance(loss, tuple) else loss
                    loss.backward()
                    trainer.optimizer.step()
                    e1.record(); torch.cuda.synchronize()
                    if i >= 3:
                        ts.append(e0.elapsed_time(e1))
                return float(np.median(ts))
            # f1: FusedAdam + factored table gradient (csrc/train.cu); then the same step with torch.optim.Adam and the dense
            # [n_items, F] table gradients for comparison (eager launches on both sides, host overhead included)
            tr_fused = Trainer(config, model)
            res["train_step_ms"] = time_train(tr_fused)
            res["train_optimizer"] = type(tr_fused.optimizer).__name__
            config["fused_adam"] = False
            res["train_step_ms_torch_adam"] = time_train(Trainer(config, model))      # (its constructor takes the parameters back)
            config["fused_adam"] = None
            res["train_batch"] = int(config["train_batch_size"])
            model.eval()
        except Exception as exc:                                     # noqa: BLE001
            res["train_step_ms"] = None
            res["train_step_error"] = f"{type(exc).__name__}: {exc}"[:200]
        try:
            res["torch_gpu_comparator"] = torch_gpu_comparator(model, all_users, batches_dev, flush) if model_name == "FREEDOM" else None
        except Exception as exc:                                     # noqa: BLE001  (context only: never fail the bench line over it)
            res["torch_gpu_comparator"] = {"unavailable": f"{type(exc).__name__}: {exc}"[:200]}
    del graphs, e2e_graphs
    return res


def run_ours(args):
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus != world:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch N>1 with: python -m torch.distributed.run --nproc-per-node N bench.py --gpus N ...")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1 or args.sharded or args.workload == "xls":
        if args.dump_outputs:
            raise SystemExit("--dump-outputs writes the outputs of the single-GPU model-class path; the item-sharded driver has none")
        # the item-sharded driver; at world size 1 it is the weak-scaling baseline of the same per-GPU problem (no exchange)
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1"); os.environ.setdefault("MASTER_PORT", "29533")
        os.environ.setdefault("RANK", "0"); os.environ.setdefault("WORLD_SIZE", "1")
        dist.init_process_group("nccl", device_id=dev)
        from mmrec_b200 import sharded
        return sharded.bench_sharded(args, rank, world, dev, Workload, peaks, ClockSampler)

    model_name = args.model or MODEL_OF.get(args.workload, "FREEDOM")
    wl = Workload(args.workload, n_layers=3)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    sampler = ClockSampler(local)
    r = bench_model(wl, model_name, dev, args, flush, sampler, full=True, dump_dir=args.dump_outputs)
    K = args.steps
    ms = r["ms"]
    msA, msB, msC = ms["a"], ms.get("b", 0.0), ms["c"]
    pk = peaks()
    edges, spmm_bytes = r["edges_per_step"], r["spmm_bytes"]
    res = {
        "metric": "graph-prop edges/sec (+ full-catalog scored-items/sec in extra) @ d=64",
        "value": edges / (msA * 1e-3), "unit": "edges/s", "n_gpus": 1, "steps": K, "warmup": args.warmup,
        "ms_per_step": msA + msB + msC, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": r["workload"], "eval_batch": "all users in one full_sort_topk call (no score matrix exists, so the batch is "
                   "bounded by nothing; the reference's default of 4096 users per call is timed as extra.score_topk_ms_batch4096)",
                   "l2": "flushed (512 MiB write) before every step", "launch": "each section replayed from a CUDA graph",
                   "api": "model.forward / ops.project / model.full_sort_topk of the drop-in model class", "parallelism": "1 GPU"},
        "extra": {"prop_ms": msA, "proj_ms": msB, "score_topk_ms": msC, "score_topk_ms_batch4096": ms["c4096"],
                  "scored_items_per_sec": r["score_items"] / (msC * 1e-3),
                  "scored_items_per_sec_batch4096": r["score_items"] / (ms["c4096"] * 1e-3),
                  "projected_rows_per_sec": (2 * wl.I / (msB * 1e-3)) if msB else None,
                  "edges_per_step": edges, "scored_items_per_step": r["score_items"],
                  "train_step_ms": r.get("train_step_ms"), "train_step_ms_torch_adam": r.get("train_step_ms_torch_adam"),
                  "train_optimizer": r.get("train_optimizer"), "train_batch": r.get("train_batch"),
                  "score_path": os.environ.get("MMREC_SCORE_PATH", "auto"), "torch_gpu_comparator": r.get("torch_gpu_comparator")},
        "roofline": {"kernel": "spmm_vec_kernel<64,16> (the SpMMs of one forward: 3 x A_hat + mm_adj)", "bound": "hbm",
                     "achieved": spmm_bytes / (msA * 1e-3) / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s",
                     "frac": spmm_bytes / (msA * 1e-3) / 1e9 / pk["hbm_gbs"], "traffic": ncu_traffic("spmm_vec_kernel"), "peak_src": pk["src"],
                     "algorithmic_bytes_per_launch_ui": r["ui_bytes"]},
        "roofline_scoring": {"kernel": "cf_pass_kernel<1|2> (tcgen05 kind::f16 on fp16-rounded operands, two passes) + cf_thr / cf_final "
                                       "(+ operand packing, mask CSR)",
                             "bound": "tensor", "achieved": r["score_flops"] / (msC * 1e-3) / 1e12, "peak": pk["bf16_tflops"], "unit": "TFLOP/s",
                             "frac": r["score_flops"] / (msC * 1e-3) / 1e12 / pk["bf16_tflops"],
                             "frac_of_tf32_peak": r["score_flops"] / (msC * 1e-3) / 1e12 / (pk["bf16_tflops"] / 2),
                             "note": "peak = measured dense bf16/fp16 rate (the pipe the filter passes run on since round 2; round 1's 3xTF32 "
                                     "kernel was quoted against half of it, kept as frac_of_tf32_peak); useful flops 2*B*I*d over the whole "
                                     "section (the tensor cores execute 2x that: filter pass + candidate pass)"},
        "e2e": {"value": edges / (r["e2e"]["prop_ms"] * 1e-3), "unit": "edges/s", "h2d_bytes_per_step": r["e2e"]["h2d"],
                "d2h_bytes_per_step": r["e2e"]["d2h"], "prop_ms": r["e2e"]["prop_ms"], "score_topk_ms": r["e2e"]["score_topk_ms"],
                "scored_items_per_sec": r["score_items"] / (r["e2e"]["score_topk_ms"] * 1e-3), "launch": r["e2e"]["mode"],
                "api": "embedding tables from pinned host memory -> model.forward -> outputs to the host; evaluation batch from pinned "
                       "host memory -> model.full_sort_topk -> index matrix to the host"},
        "gpu_launches": int(r["launches"]), "clocks": r["clocks"],
    }
    if msB:
        res["roofline_projection"] = {"kernel": "project_tc_kernel + project_reduce_kernel (2 modalities)", "bound": "hbm",
                                      "achieved": r["proj_bytes"] / (msB * 1e-3) / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s",
                                      "frac": r["proj_bytes"] / (msB * 1e-3) / 1e9 / pk["hbm_gbs"], "tflops": r["proj_flops"] / (msB * 1e-3) / 1e12}
    # BASELINE.json configs[2] (BM3 / sports) and configs[3] (MGCN / clothing): the same sections through their model classes
    if args.workload == "baby" and not args.no_other_configs:
        res["extra"]["other_configs"] = {}
        for w2, m2 in (("sports", "BM3"), ("clothing", "MGCN")):
            try:
                wl2 = Workload(w2, n_layers=2)
                r2 = bench_model(wl2, m2, dev, args, flush, None, full=False)
                res["extra"]["other_configs"][f"{m2}/{w2}"] = {
                    "workload": r2["workload"], "prop_ms": r2["ms"]["a"], "edges_per_sec": r2["edges_per_step"] / (r2["ms"]["a"] * 1e-3),
                    "spmm_roofline_frac": r2["spmm_bytes"] / (r2["ms"]["a"] * 1e-3) / 1e9 / pk["hbm_gbs"],
                    "score_topk_ms": r2["ms"]["c"], "scored_items_per_sec": r2["score_items"] / (r2["ms"]["c"] * 1e-3),
                    "score_topk_ms_batch4096": r2["ms"]["c4096"],
                    "scoring_tf32_frac": r2["score_flops"] / (r2["ms"]["c"] * 1e-3) / 1e12 / (pk["bf16_tflops"] / 2),
                    "e2e_prop_ms": r2["e2e"]["prop_ms"], "e2e_score_topk_ms": r2["e2e"]["score_topk_ms"]}
                del wl2, r2
                torch.cuda.empty_cache()
            except Exception as exc:                                 # noqa: BLE001
                res["extra"]["other_configs"][f"{m2}/{w2}"] = {"unavailable": f"{type(exc).__name__}: {exc}"[:300]}
    if not args.no_cpu_baseline:
        res["cpu_baseline"] = cpu_baseline(wl, steps=3)
    print(json.dumps(res))


# ------------------------------------------------------------------------------------------------------
# CPU arm: the reference's algorithm (oracle port: same torch CPU ops in the same order as the reference)
# ------------------------------------------------------------------------------------------------------
def cpu_setup(wl, mm_layers=1, knn="features"):
    from oracle import mmrec_oracle as O
    adj = O.norm_adj_coo(wl.tr_u, wl.tr_i, wl.U, wl.I)
    mm = None
    if mm_layers:
        if knn == "features":                                        # the same item-item graph the model class builds (freedom.py:67-100)
            v, t = wl.features()
            mm = O.freedom_mm_adj(torch.from_numpy(v), torch.from_numpy(t), KNN_K, 0.1)
        else:                                                        # scaled N-GPU workloads: the synthetic neighbour lists
            kr, kc, kv = wl.knn_coo()
            mm = torch.sparse_coo_tensor(torch.from_numpy(np.stack([kr, kc])), torch.from_numpy(kv), (wl.I, wl.I), check_invariants=False)
    lo, hi = 0, min(wl.U, EVAL_BATCH)
    batch = (torch.arange(lo, hi), torch.from_numpy(wl.eval_mask(lo, hi)))          # one evaluation batch, built outside the timed region
    return O, adj, mm, torch.from_numpy(wl.user_emb), torch.from_numpy(wl.item_emb), batch


def cpu_step(O, wl, adj, mm, ue, ie, batch, mm_layers=1):
    t0 = time.perf_counter()
    u_g, i_g = O.freedom_forward(adj, mm, ue, ie, mm_layers, wl.n_layers)  # freedom.py:164-178
    t1 = time.perf_counter()
    users, mask = batch
    s = O.full_sort_scores(u_g, i_g, users)                                 # freedom.py:216-220
    O.mask_topk(s, mask, TOPK)                                              # trainer.py:304-309
    t2 = time.perf_counter()
    return t1 - t0, t2 - t1, users.numel() * wl.I


def pick_threads(O, wl, adj, mm, ue, ie, batch, mm_layers=1):
    """Give the CPU arm its best shot: torch's sparse/dense kernels at this size get slower when oversubscribed,
    so try a few thread counts (up to all host cores) on one step and keep the fastest."""
    cores = os.cpu_count() or 1
    best, best_t = 1, float("inf")
    with torch.no_grad():
        for t in sorted({min(cores, c) for c in (4, 8, 16, 32, 64, cores)}):
            torch.set_num_threads(t)
            cpu_step(O, wl, adj, mm, ue, ie, batch, mm_layers)
            a, c, _ = cpu_step(O, wl, adj, mm, ue, ie, batch, mm_layers)
            if a + c < best_t:
                best, best_t = t, a + c
    torch.set_num_threads(best)
    return best


def cpu_baseline(wl, steps=3):
    O, adj, mm, ue, ie, batch = cpu_setup(wl)
    threads = pick_threads(O, wl, adj, mm, ue, ie, batch)
    with torch.no_grad():
        cpu_step(O, wl, adj, mm, ue, ie, batch)
        ta = tc = 0.0
        sc = 0
        for _ in range(steps):
            a, c, s = cpu_step(O, wl, adj, mm, ue, ie, batch)
            ta += a; tc += c; sc += s
    edges = wl.n_layers * adj._nnz() + mm._nnz()
    return {"value": edges * steps / ta, "unit": "edges/s", "cores": threads, "kind": "port",
            "sample": f"{steps} x (FREEDOM forward on the full graph + 1 eval batch of {EVAL_BATCH} users), torch CPU fp32, "
                      f"same ops/order as the reference (oracle/mmrec_oracle.py); threads = fastest of 4/8/16/32/64/all {os.cpu_count()} host cores",
            "scored_items_per_sec": sc / tc}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # the same workload as this repo's arm at --gpus N: weak scaling = N x the items and edges
    n = max(1, args.gpus)
    wl = Workload(args.workload, n_layers=3, items_scale=n)
    O, adj, mm, ue, ie, batch = cpu_setup(wl, 1, "features" if (n == 1 and args.workload != "xls" and not args.sharded) else "synthetic")
    threads = pick_threads(O, wl, adj, mm, ue, ie, batch)
    edges = wl.n_layers * adj._nnz() + mm._nnz()
    ta = tc = 0.0
    sc = 0
    with torch.no_grad():
        for step in range(args.warmup + args.steps):
            a, c, s = cpu_step(O, wl, adj, mm, ue, ie, batch)
            if step >= args.warmup:
                ta += a; tc += c; sc += s
    K = args.steps
    value = edges * K / ta
    sample = (f"each step: FREEDOM forward on the full graph + score/mask/top-{TOPK} of ONE batch of {EVAL_BATCH} users "
              f"(bounded sample of the {wl.U}-user pass), torch CPU fp32 with {threads} threads (fastest of 4/8/16/32/64/all {os.cpu_count()} host cores)")
    if n == 1 and args.workload != "xls" and not args.sharded:
        workload = wl.describe("FREEDOM", wl.n_layers, 1)
    else:
        workload = (f"FREEDOM synthetic {wl.name} x{n} items: {wl.U} users, {wl.I} items ({wl.I // n} per GPU), {len(wl.tr_u)} train edges, "
                    f"d={wl.d}, {wl.n_layers} UI layers + 1 mm layer, top-{TOPK} over all users, eval batch {EVAL_BATCH}")
    print(json.dumps({
        "impl": "reference", "metric": "graph-prop edges/sec (+ full-catalog scored-items/sec in extra) @ d=64",
        "value": value, "unit": "edges/s", "n_gpus": args.gpus, "steps": K, "warmup": args.warmup,
        "ms_per_step": (ta + tc) / K * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload, "parallelism": f"CPU, {threads} threads"},
        "extra": {"prop_ms": ta / K * 1e3, "score_topk_ms_per_batch": tc / K * 1e3, "scored_items_per_sec": sc / tc},
        "cpu_baseline": {"value": value, "unit": "edges/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                "scored_items_per_sec": sc / tc},
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="baby", choices=list(synth.SHAPES))
    ap.add_argument("--model", default=None, help="model class (default: the one BASELINE.json pairs with the workload)")
    ap.add_argument("--sharded", action="store_true", help="run the item-sharded driver also at --gpus 1 (weak-scaling baseline)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the BM3/sports and MGCN/clothing lines in extra")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of this repo's CUDA path (--impl ours)")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
