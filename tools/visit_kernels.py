"""Device time of every kernel of an eager label visit of the bench configuration (F=10, K=5, Z=128, batch 4096), split by
step kind, from torch.profiler with CUDA activities.

    python tools/visit_kernels.py [--visits 4] [--out profiles/visit_kernels.json]

Each step kind is profiled in visits of that kind alone (loops 5,0,0 / 0,5,0 / 0,0,3), so every kernel is attributed to
its step; one full visit (5,5,3) is profiled as well.  Times are device time per visit, averaged over `--visits` visits
after two warm-up visits.  For the D and C steps it also reports the weight-gradient tail: from the end of the step's chain
kernel to the end of the step's last weight-gradient kernel, which is what the step's join waits for.  Prints a table and
writes the numbers as JSON."""
import argparse
import collections
import json
import os
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

KINDS = {"d": (5, 0, 0), "c": (0, 5, 0), "eg": (0, 0, 3), "visit": (5, 5, 3)}
CHAIN = {"d": "critic_chain_kernel", "c": "classifier_chain_kernel"}


def short(name):
    name = name.replace("void ", "").replace("cvg::", "")
    return name.split("(")[0]


def device_kernels(prof):
    out = []
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA and ev.time_range.end > ev.time_range.start:
            out.append((ev.time_range.start, ev.time_range.end, short(ev.name)))
    return sorted(out)


def dw_tail(kern, chain):
    """us from the end of each chain kernel to the end of the last weight-gradient kernel before the next chain kernel."""
    idx = [i for i, k in enumerate(kern) if k[2].startswith(chain)]
    tails = []
    for a, i in enumerate(idx):
        stop = kern[idx[a + 1]][0] if a + 1 < len(idx) else float("inf")
        ends = [k[1] for k in kern[i + 1:] if k[0] < stop and k[2].startswith("gemm_dw")]
        if ends:
            tails.append(max(ends) - kern[i][1])
    return tails


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--visits", type=int, default=4)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from torch.profiler import ProfilerActivity, profile
    from cvae_gan_b200 import models
    from cvae_gan_b200.engine import Engine
    F_, K, Z, B = 10, 5, 128, 4096
    torch.manual_seed(0)
    eng = Engine(F_, K, Z, max_batch=B)
    mods = [models.CVAEGANEncoderModel(F_, K, Z), models.CVAEGANGeneratorModel(Z, K, F_),
            models.CVAEGANDiscriminatorModel(F_, K), models.CVAEGANClassifierModel(F_, K)]
    for net, m in enumerate(mods):
        eng.load_state(net, m.state_dict())
    g = torch.Generator(device="cuda").manual_seed(0)
    tabs = [torch.rand(20000, F_, device="cuda", generator=g) for _ in range(K)]
    eng.ctl_set(seed=1234, counter=0, lambda_class=0.25)
    loss = torch.zeros(13, 4, device="cuda")
    result = {"gpu": torch.cuda.get_device_name(0), "visits": args.visits, "batch": B, "kinds": {}}
    for kind, loops in KINDS.items():
        for i in range(2):
            eng.visit(i % K, B, class_rows=tabs[i % K], loops=loops, loss_out=loss)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for i in range(args.visits):
                eng.visit(i % K, B, class_rows=tabs[i % K], loops=loops, loss_out=loss)
            torch.cuda.synchronize()
        kern = device_kernels(prof)
        per = collections.defaultdict(lambda: [0, 0.0])
        for s, e, n in kern:
            per[n][0] += 1
            per[n][1] += e - s
        rows = {n: {"launches": c / args.visits, "us": t / args.visits} for n, (c, t) in per.items()}
        rec = {"loops": loops, "kernels": dict(sorted(rows.items(), key=lambda kv: -kv[1]["us"])),
               "device_us": sum(r["us"] for r in rows.values()),
               "gemm_dw_us": sum(r["us"] for n, r in rows.items() if n.startswith("gemm_dw")),
               "span_us": (kern[-1][1] - kern[0][0]) / args.visits if kern else 0.0}
        if kind in CHAIN:
            t = dw_tail(kern, CHAIN[kind])
            rec["dw_tail_us_per_step"] = {"mean": sum(t) / len(t), "min": min(t), "max": max(t), "n": len(t)} if t else None
        result["kinds"][kind] = rec
        print(f"== {kind} {loops}: device {rec['device_us']:.1f} us/visit, gemm_dw {rec['gemm_dw_us']:.1f} us, "
              f"span {rec['span_us']:.1f} us" + (f", dW tail per step {rec['dw_tail_us_per_step']}" if kind in CHAIN else ""))
        for n, r in rec["kernels"].items():
            print(f"  {r['us']:9.1f} us  {r['launches']:5.1f} x  {n}")
    eng.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
