"""Per-step time of the E/G step with the generator backward split into per-pass chains (csrc/train.cu step_g) and without
(cvg_debug_set("eg_split", 0)).

    python tools/eg_ab.py [--batch 4096] [--steps 50]

`--steps` E/G steps through the per-step API (seeded Philox noise, lambda_class 0.25, Adam update) are captured in a CUDA
graph and timed with CUDA events over 10 replays after a warm-up replay; the two settings alternate three times.  Prints
one JSON line per (round, setting) with ms per step and launches per step."""
import argparse
import json
import os
import sys

import torch

REPLAYS = 10

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=50)
    args = ap.parse_args()
    from cvae_gan_b200 import models
    from cvae_gan_b200.engine import Engine
    F_, K, Z, B = 10, 5, 128, args.batch
    torch.manual_seed(0)
    eng = Engine(F_, K, Z, max_batch=B)
    mods = [models.CVAEGANEncoderModel(F_, K), models.CVAEGANGeneratorModel(Z, K, F_),
            models.CVAEGANDiscriminatorModel(F_, K), models.CVAEGANClassifierModel(F_, K)]
    for net, m in enumerate(mods):
        eng.load_state(net, m.state_dict())
    x = torch.rand(B, F_, device="cuda")
    for rnd in range(3):
        for split in (1, 0):
            eng.debug_set("eg_split", split)
            for i in range(3):
                eng.step_g(x, 2, 0.25, seed=7, counter=2 * i)
            torch.cuda.synchronize()
            gr = torch.cuda.CUDAGraph()
            l0 = eng.launch_count()
            with torch.cuda.graph(gr):
                for i in range(args.steps):
                    eng.step_g(x, 2, 0.25, seed=7, counter=2 * i)
            launches = (eng.launch_count() - l0) / args.steps
            gr.replay()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(REPLAYS):
                gr.replay()
            b.record()
            torch.cuda.synchronize()
            print(json.dumps({"round": rnd, "eg_split": split, "batch": B,
                              "ms_per_step": a.elapsed_time(b) / (REPLAYS * args.steps),
                              "launches_per_step": launches}), flush=True)
            del gr
    eng.close()


if __name__ == "__main__":
    main()
