"""Data-parallel path on CPU (gloo, world_size 2): the sharding scheme the CUDA engine implements -
batch rows split across ranks, BatchNorm batch moments all-reduced between layers, flat gradient
all-reduce before Adam, losses summed - must reproduce the single-process result on the full batch.
Checked here on the oracle (the same algebra the NCCL path follows, train.cu `sync_stats` /
`finish_step`), plus the host-side sharding helpers (global-row-keyed draws, generation row ranges)."""
import os
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import cvae_gan_oracle as O  # noqa: E402

F_, K, B, Z = 10, 5, 32, 128


# step sequences per trainer: the CVAE-GAN's (d, c, g) and the sibling trainers' own generator steps (SURVEY 8 f4):
# p = CGAN (cgan.py:138-178), v = CVAE (cvae.py:117-166), u = VAE-GAN on unconditional networks (vae_gan.py:103-141)
SEQUENCES = {"cvae_gan": "dcgdg", "cgan": "dcpdp", "cvae": "cvcv", "vae_gan": "dudu"}


def _build(dp=None, trainer="cvae_gan"):
    g = torch.Generator().manual_seed(7)
    cfg = O.OracleConfig(batch_size=B, unconditional=(trainer == "vae_gan"))
    orc = O.OracleCVAEGAN(F_, K, cfg, dp=dp).init_like_reference(g)
    orc.make_optimizers()
    return orc


def _noise(kind, rows, g):
    out = {}
    if kind != "v":
        out["z"] = torch.randn(rows, Z, generator=g)
    if kind in ("g", "v", "u"):
        out["eps"] = torch.randn(rows, Z, generator=g)
    specs = {"d": [("d", 2)], "c": [("c", 2)], "v": [("c", 1)], "u": [("d", 1)]}.get(kind, [("d", 1), ("c", 1)])
    for prefix, n in specs:
        out[prefix + "_mask1"] = (torch.rand(n, rows, 256, generator=g) < 0.7).float()
        out[prefix + "_mask2"] = (torch.rand(n, rows, 128, generator=g) < 0.7).float()
    return out


def _inject(noise, sl):
    inj = O.InjectedNoise()
    if "z" in noise:
        inj.push("z", noise["z"][sl])
    if "eps" in noise:
        inj.push("eps", noise["eps"][sl])
    for prefix in ("d", "c"):
        if prefix + "_mask1" in noise:
            for p in range(noise[prefix + "_mask1"].shape[0]):
                inj.push(prefix + "_mask1", noise[prefix + "_mask1"][p][sl])
                inj.push(prefix + "_mask2", noise[prefix + "_mask2"][p][sl])
    return inj


def _run(orc, sl, trainer="cvae_gan"):
    g = torch.Generator().manual_seed(99)
    x = torch.rand(B, F_, generator=g)
    label = None if trainer == "vae_gan" else 3
    out = []
    for kind in SEQUENCES[trainer]:
        nz = _noise(kind, B, g)
        inj = _inject(nz, sl)
        if kind == "d":
            loss, _ = orc.step_d(x[sl], label, inj)
            out.append(orc.last_losses["d_loss"])
        elif kind == "c":
            loss, _ = orc.step_c(x[sl], label, inj)
            out.append(orc.last_losses["c_loss"])
        elif kind == "p":
            losses, _ = orc.step_g_prior(label, x[sl].shape[0], inj, 0.25)
            out.extend(losses.values())
        elif kind == "v":
            losses, _ = orc.step_g_cvae(x[sl], label, inj, 0.25)
            out.extend(losses.values())
        elif kind == "u":
            losses, _ = orc.step_g_vaegan(x[sl], inj)
            out.extend(losses.values())
        else:
            losses, _ = orc.step_g(x[sl], label, inj, 0.25)
            out.extend(losses.values())
    return out


def _worker(rank, world, port, q, trainer="cvae_gan"):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.set_num_threads(1)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    dp = O.DataParallelCtx(rank, world)
    orc = _build(dp, trainer)
    per = B // world
    losses = _run(orc, slice(rank * per, (rank + 1) * per), trainer)
    st = orc.state()
    flat = torch.cat([t.flatten().float() for n in O.NETS for t in st[n].values()])
    # a numpy copy, not the tensor: torch.multiprocessing passes tensors by file descriptor, which the parent can only
    # fetch while this process lives, and it exits right after the barrier below
    q.put((rank, losses, flat.numpy()))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("trainer", sorted(SEQUENCES))
def test_dp2_equals_single_process(trainer):
    torch.set_num_threads(1)
    single = _build(None, trainer)
    ref_losses = _run(single, slice(0, B), trainer)
    st = single.state()
    ref_flat = torch.cat([t.flatten().float() for n in O.NETS for t in st[n].values()])
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000) + 7 * sorted(SEQUENCES).index(trainer)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q, trainer)) for r in range(2)]
    for p in procs:
        p.start()
    results = [(rank, losses, torch.from_numpy(flat)) for rank, losses, flat in (q.get(timeout=300) for _ in range(2))]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for rank, losses, flat in results:
        assert losses == pytest.approx(ref_losses, rel=2e-4, abs=2e-5), rank
        # Adam normalises near-zero gradients (pre-BN biases etc.) into +-lr steps: allow 5 steps of lr
        assert torch.allclose(flat, ref_flat, rtol=1e-3, atol=5 * 2e-4 * 1.5), rank
    assert torch.equal(results[0][2], results[1][2])      # replicas stay bit-identical


def test_generation_row_ranges_partition_the_stream():
    """Generation shards with no collective: rank r takes rows [r*n/W, (r+1)*n/W) of the Philox stream."""
    n, W = 1000003, 8
    per = (n + W - 1) // W
    ranges = [(r * per, min(n, (r + 1) * per)) for r in range(W)]
    assert ranges[0][0] == 0 and ranges[-1][1] == n
    assert all(a[1] == b[0] for a, b in zip(ranges, ranges[1:]))
