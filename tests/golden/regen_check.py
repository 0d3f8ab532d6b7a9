"""Re-run parts of make_golden.py against a checkout of the reference (the one ref_loader.py imports) into a scratch
directory and compare with the committed golden files: a model dump, the MMGCN dump under the PyG shim and a training
trajectory -- every array bit for bit, recorded gradients to 1e-5 (CPU `index_put` backward is not run-to-run
deterministic).  Prints one `REGEN {json}` line; needs the reference, so it is run by hand when a generator changes."""
import json
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))
import make_golden as M  # noqa: E402
from conftest import load_golden  # noqa: E402
import ref_loader  # noqa: E402
from mmrec_b200.utils import synth  # noqa: E402


def main():
    ref_loader.install()
    tmp = tempfile.mkdtemp(prefix="mmrec_regen_")
    data_root = ref_loader.run_dir(tmp)
    u, i, e, d, f = synth.SHAPES["tiny"]
    g = synth.make_graph(u, i, e, seed=0)
    v, t = synth.make_features(i, f, seed=1)
    synth.write_dataset(data_root, "tiny", g, v, t)
    import logging
    logging.disable(logging.CRITICAL)
    common = {"eval_batch_size": 128, "train_batch_size": 512}
    out = os.path.join(tmp, "out")
    os.makedirs(out)
    M.dump_model("LightGCN", dict(common, n_layers=[3]), os.path.join(out, "lightgcn_tiny.npz"))
    M.dump_mmgcn(common, os.path.join(out, "mmgcn_tiny.npz"))
    M.dump_trajectory("BM3", common, os.path.join(out, "traj_bm3_tiny.npz"), slim=True)
    report = {}
    for name in ("lightgcn_tiny.npz", "mmgcn_tiny.npz", "traj_bm3_tiny.npz"):
        a, b = load_golden(name, out), load_golden(name, HERE)
        same_keys = sorted(a.files) == sorted(b.files)
        exact, worst = True, 0.0
        for k in b.files:
            x, y = a[k], b[k]
            if x.dtype == object or x.dtype.kind in "US":
                ok = len(x) == len(y) and all(np.array_equal(p, q) for p, q in zip(x, y))
            elif k.startswith("grad.") or k.startswith("paramT."):          # CPU index_put backward is not run-to-run deterministic
                err = float(np.abs(x.astype(np.float64) - y).max() / max(float(np.abs(y).max()), 1e-30))
                worst, ok = max(worst, err), err < 1e-5
            else:
                ok = x.shape == y.shape and np.array_equal(x, y)
            exact = exact and bool(ok)
        report[name] = {"same_keys": same_keys, "reproduced": exact, "worst_grad_rel": worst}
    print("REGEN " + json.dumps(report))


if __name__ == "__main__":
    main()
