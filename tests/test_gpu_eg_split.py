"""The E/G step's generator backward run as two per-pass chains (csrc/train.cu step_g) against the one two-pass chain it
replaces (cvg_debug_set("eg_split", 0)): from the same state and noise, every parameter, gradient, Adam moment, BN / SN
state, loss and workspace buffer the backward writes must be bit-identical."""
import pytest
import torch

from tests import parity as P

pytestmark = pytest.mark.gpu

# workspace buffers of the backward: (name, passes)
BUFS = [("g_dout", 2), ("g_dy0", 2), ("g_dy1", 2), ("g_dy2", 2), ("e_dml", 1), ("e_dy0", 1), ("e_dy1", 1), ("e_dy2", 1),
        ("dx", 1)]
# the split adds the pass-1 seed and the pass-1 input gradients of generator layers 3, 2 and 1
EXTRA_LAUNCHES = 4


def _snapshot(eng, B):
    out = {}
    for n in range(4):
        for which in ("params", "grads", "adam_m", "adam_v", "state"):
            out[f"{which}{n}"] = getattr(eng, which)[n].clone()
    for name, passes in BUFS:
        for pas in range(passes):
            out[f"{name}/{pas}"] = eng.debug_read(name, B, pas)
    return out


def _step(F_, K, B, split, update, lam, **cfg_kw):
    from cvae_gan_b200._lib import STEP_NO_UPDATE
    orc, eng, g = P.make_pair(F_, K, B, seed=5 + B, **cfg_kw)
    eng.debug_set("eg_split", split)
    x, y = P.make_data(F_, K, [B] * K, seed=2)
    xb = x[y == (K - 1)][:B].contiguous().cuda()
    uncond = cfg_kw.get("unconditional", False)
    h1, h2 = (cfg_kw.get("hidden") or (256, 128, 64))[:2]
    _, dev = P.draw_noise("u" if uncond else "g", B, orc.cfg.z_size, g, h1=h1, h2=h2)
    label = 0 if uncond else K - 1
    l0 = eng.launch_count()
    loss = eng.step_g(xb, label, lam, noise=dev, flags=0 if update else STEP_NO_UPDATE).clone()
    launches = eng.launch_count() - l0
    torch.cuda.synchronize()
    out = _snapshot(eng, B)
    out["loss"] = loss
    eng.close()
    return out, launches


def _assert_equal(a, b):
    assert a.keys() == b.keys()
    bad = [k for k in a if not torch.equal(a[k], b[k])]
    assert not bad, f"differ: {bad}"


def _assert_split_matches(F_, K, B, update, lam, **cfg_kw):
    split, n_split = _step(F_, K, B, 1, update, lam, **cfg_kw)
    ref, n_ref = _step(F_, K, B, 0, update, lam, **cfg_kw)
    assert n_split == n_ref + EXTRA_LAUNCHES, (n_split, n_ref)     # the split schedule ran
    _assert_equal(split, ref)


@pytest.mark.parametrize("F_,K,B", [(10, 5, 64), (10, 4, 333), (30, 5, 128), (10, 5, 4096)])
@pytest.mark.parametrize("update", [False, True])
@pytest.mark.parametrize("lam", [0.25, 0.0])
def test_eg_split_step_bit_identical(F_, K, B, update, lam):
    _assert_split_matches(F_, K, B, update, lam)


def test_eg_split_unconditional_bit_identical():
    """VAE-GAN's encoder / generator step: no label columns, no classifier term."""
    _assert_split_matches(10, 5, 256, True, 0.0, unconditional=True)


def test_eg_split_wide_bit_identical():
    """The widened model (hidden 512 / 256 / 128 in every network)."""
    _assert_split_matches(10, 5, 512, True, 0.25, hidden=(512, 256, 128))


def test_eg_split_graph_visit_bit_identical():
    """One CUDA-graph-captured label visit (5 D, 5 C, 3 E/G steps) with and without the split, replayed twice."""
    from cvae_gan_b200 import models
    from cvae_gan_b200.engine import Engine
    F_, K, B = 10, 5, 1024
    rows = torch.rand(5000, F_, generator=torch.Generator().manual_seed(0)).cuda()
    outs, launches = [], []
    for split in (1, 0):
        torch.manual_seed(3)
        eng = Engine(F_, K, 128, max_batch=B)
        mods = [models.CVAEGANEncoderModel(F_, K), models.CVAEGANGeneratorModel(128, K, F_),
                models.CVAEGANDiscriminatorModel(F_, K), models.CVAEGANClassifierModel(F_, K)]
        for net, m in enumerate(mods):
            eng.load_state(net, m.state_dict())
        eng.debug_set("eg_split", split)
        eng.ctl_set(seed=77, counter=10, lambda_class=0.25)
        loss = torch.zeros(13, 4, device="cuda")
        gr = torch.cuda.CUDAGraph()
        l0 = eng.launch_count()
        with torch.cuda.graph(gr):
            eng.visit(2, B, class_rows=rows, loops=(5, 5, 3), loss_out=loss)
        launches.append(eng.launch_count() - l0)
        gr.replay()
        gr.replay()
        torch.cuda.synchronize()
        out = _snapshot(eng, B)
        out["loss"] = loss.clone()
        outs.append(out)
        del gr
        eng.close()
    assert launches[0] == launches[1] + 3 * EXTRA_LAUNCHES, launches
    _assert_equal(outs[0], outs[1])
