"""A/B check of the CTA-pair FFN kernel (TTB_FFN_PAIR=1) against the cta_group::1 kernel (TTB_FFN_PAIR=0):
full-size bf16 forward on the golden inputs and on a larger random batch, each mode in its own process."""
import os
import subprocess
import sys
import tempfile
from pathlib import Path

import numpy as np
import torch

REPO = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(REPO))


def child(out):
    sys.path.insert(0, str(REPO / "tests"))
    from helpers import load_json, load_npz
    from translation_transformer_b200.model import B200Transformer
    from translation_transformer_b200.weights import ModelConfig, random_init_state_dict
    z, meta = load_npz("model_forward.npz"), load_json("model_forward.json")
    m = meta["meta"]["full"]
    cfg = ModelConfig(**m["config"])
    sd = random_init_state_dict(cfg, m["seed"])
    eng = B200Transformer(cfg, sd, precision="bf16", device=0)
    dev = torch.device("cuda", 0)
    src, tgt = torch.from_numpy(z["full_src"]).to(dev), torch.from_numpy(z["full_tgt"]).to(dev)
    a = eng(src, tgt).float().cpu().numpy()
    g = torch.Generator().manual_seed(7)
    V = cfg.tgt_vocab_size
    src2 = torch.randint(3, V, (37, 61), generator=g).to(dev)
    tgt2 = torch.randint(3, V, (37, 50), generator=g).to(dev)
    b = eng(src2, tgt2).float().cpu().numpy()
    # more 256-row blocks than clusters of four fit on the chip at once (second wave of clusters), ragged last block
    src3 = torch.randint(3, V, (181, 40), generator=g).to(dev)
    tgt3 = torch.randint(3, V, (181, 50), generator=g).to(dev)
    c = eng(src3, tgt3).float().cpu().numpy()
    torch.cuda.synchronize()
    np.savez(out, a=a, b=b, c=c, ref=z["full_forward_logits"])
    print("child done", out, a.shape, b.shape, c.shape, flush=True)


if __name__ == "__main__":
    if len(sys.argv) > 1:
        child(sys.argv[1])
        sys.exit(0)
    outs = {}
    with tempfile.TemporaryDirectory() as tmp:      # private to this run: several users may share the machine
        for mode in ("0", "1"):
            env = dict(os.environ, TTB_FFN_PAIR=mode, TTB_DEBUG="1")
            f = os.path.join(tmp, f"ffn_pair_{mode}.npz")
            r = subprocess.run(["timeout", "120", sys.executable, __file__, f], env=env)
            print("mode", mode, "rc", r.returncode, flush=True)
            if r.returncode != 0:
                sys.exit(1)
            with np.load(f) as z:
                outs[mode] = dict(z)
    worst = 0.0
    for k in ("a", "b", "c"):
        d = np.abs(outs["0"][k] - outs["1"][k])
        worst = max(worst, float(d.max()) if not np.isnan(d).any() else float("inf"))
        print(k, "max|pair - single| =", float(d.max()), "scale", float(np.abs(outs["0"][k]).max()), "nan", int(np.isnan(outs["1"][k]).sum()))
    ref = outs["0"]["ref"]
    for mode in ("0", "1"):
        print("mode", mode, "max|logits - fp32 golden| =", float(np.abs(outs[mode]["a"] - ref).max()), "of", float(np.abs(ref).max()))
    print("WORST", worst)
    sys.exit(0 if worst == 0.0 else 2)
