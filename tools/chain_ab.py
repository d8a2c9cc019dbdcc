"""Per-step-kind time of the D and C steps with the fused critic / classifier chains (csrc/chain.cuh) on and off.

    python tools/chain_ab.py [--batch 4096] [--steps 50]

`--steps` steps of one kind through the per-step API (seeded Philox noise, Adam update) are captured in a CUDA graph and
timed with CUDA events over 10 replays after a warm-up replay; the two settings alternate three times.  Prints one JSON
line per (round, setting, kind) with ms per step and launches per step."""
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
        for chain in (1, 0):
            eng.debug_set("chain", chain)
            for kind in ("d", "c"):
                step = eng.step_d if kind == "d" else eng.step_c
                for i in range(3):
                    step(x, 2, seed=7, counter=2 * i)
                torch.cuda.synchronize()
                gr = torch.cuda.CUDAGraph()
                l0 = eng.launch_count()
                with torch.cuda.graph(gr):
                    for i in range(args.steps):
                        step(x, 2, seed=7, counter=2 * i)
                launches = (eng.launch_count() - l0) / args.steps
                gr.replay()
                torch.cuda.synchronize()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(REPLAYS):
                    gr.replay()
                b.record()
                torch.cuda.synchronize()
                print(json.dumps({"round": rnd, "chain": chain, "kind": kind, "batch": B,
                                  "ms_per_step": a.elapsed_time(b) / (REPLAYS * args.steps),
                                  "launches_per_step": launches}), flush=True)
                del gr
    eng.close()


if __name__ == "__main__":
    main()
