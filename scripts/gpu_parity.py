"""End-to-end parity report of the CUDA path against the golden fixtures (tests/golden/*.npz,
produced by the unmodified reference).  Prints the error of every bank / pose residual /
per-block activation so a broken layer can be bisected from one GPU run."""
import argparse
import os
import sys
import time

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

import torch  # noqa: E402

from magicdance_b200 import synth  # noqa: E402  (seeded weights + inputs)
from tests import golden_util as G  # noqa: E402
from magicdance_b200.engine import DenoiseEngine  # noqa: E402


def nchw(act_data, b, h, w):
    return act_data.float().reshape(b, h, w, -1).permute(0, 3, 1, 2)


def report(gold, key, t):
    shape = tuple(int(v) for v in gold[key + "/shape"])
    f = t.detach().float().reshape(-1).cpu()
    if tuple(t.shape) != shape:
        print(f"  {key}: SHAPE {tuple(t.shape)} vs golden {shape}")
        return 9.9
    idx = synth.sample_indices(f.numel())
    err = G.rel_l2(f[idx], torch.from_numpy(gold[key + "/sample"]))
    print(f"  {key}: rel-L2 {err:.3e}  finite={bool(torch.isfinite(f).all())}")
    return err


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--case", default="small32")
    args = ap.parse_args()
    torch.set_grad_enabled(False)
    t0 = time.time()
    sd = synth.synth_state_dict(seed=0)
    print(f"synthetic weights in {time.time() - t0:.1f}s", flush=True)
    eng = DenoiseEngine(sd, device="cuda")
    del sd
    torch.cuda.synchronize()
    print(f"engine packed in {time.time() - t0:.1f}s; mem {torch.cuda.memory_allocated() / 2**30:.2f} GiB", flush=True)
    tag = args.case
    gold = G.load(tag)
    inp = G.small32_inputs() if tag == "small32" else G.full64_inputs()
    dev = {k: v.cuda() for k, v in inp.items()}
    eps_c, bank, pose, taps = eng.apply_model(dev["x"], dev["t"], dev["context"], dev["pose"], dev["ref"], uc=False,
                                              return_parts=True)
    torch.cuda.synchronize()
    b = inp["x"].shape[0]
    worst = 0.0
    if f"{tag}/n_bank" not in gold:
        print(f"(no per-layer golden for {tag}: eps only)")
    else:
        print("bank (appearance net norm1 states):")
        for i, n1 in enumerate(bank):
            shape = tuple(int(v) for v in gold[f"{tag}/bank{i}/shape"])
            worst = max(worst, report(gold, f"{tag}/bank{i}", n1.reshape(shape)))
        print("pose residuals:")
        for i, p in enumerate(pose):
            bb, c, h, w = (int(v) for v in gold[f"{tag}/pose{i}/shape"])
            worst = max(worst, report(gold, f"{tag}/pose{i}", nchw(p, bb, h, w)))
        print("UNet (read) per-block activations:")
        for i, a in enumerate(taps):
            worst = max(worst, report(gold, f"{tag}/tap{i}", nchw(a.data, a.b, a.h, a.w)))
    e = G.rel_l2(eps_c, torch.from_numpy(gold[f"{tag}/eps_c"]))
    print(f"eps_c rel-L2 {e:.3e}")
    eps_u = eng.apply_model(dev["x"], dev["t"], dev["context"], dev["pose"], None, uc=True)
    torch.cuda.synchronize()
    e2 = G.rel_l2(eps_u, torch.from_numpy(gold[f"{tag}/eps_u"]))
    print(f"eps_u rel-L2 {e2:.3e}")
    print(f"worst intermediate {worst:.3e}; launches so far {__import__('magicdance_b200').ops.launch_count()}")


if __name__ == "__main__":
    main()
