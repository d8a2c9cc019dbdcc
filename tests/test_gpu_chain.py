"""The fused critic / classifier chains of the D and C steps (csrc/chain.cuh) against the layer kernels they replace
(cvg_debug_set("chain", 0)): from the same state and noise, every parameter, gradient, Adam moment, BN / SN state, loss and
workspace buffer the chains write must be bit-identical."""
import pytest
import torch

from tests import parity as P

pytestmark = pytest.mark.gpu

BUFS = {"d": ["d_a0", "d_a1", "d_a2", "d_s", "d_g0", "d_g1", "d_g2"],
        "c": ["c_a1", "c_h2", "c_a2", "c_a3", "c_logit", "c_dlogit", "c_g0", "c_g1", "c_g2"]}


def _snapshot(eng, kind, B):
    out = {}
    for n in range(4):
        for which in ("params", "grads", "adam_m", "adam_v", "state"):
            out[f"{which}{n}"] = getattr(eng, which)[n].clone()
    for name in BUFS.get(kind, []):
        for pas in (0, 1):
            out[f"{name}/{pas}"] = eng.debug_read(name, B, pas)
    return out


def _step(kind, F_, K, B, chain, update, unconditional=False):
    from cvae_gan_b200._lib import STEP_NO_UPDATE
    orc, eng, g = P.make_pair(F_, K, B, seed=11 + B, unconditional=unconditional)
    eng.debug_set("chain", chain)
    x, y = P.make_data(F_, K, [B] * K, seed=1)
    xb = x[y == (K - 1)][:B].contiguous().cuda()
    _, dev = P.draw_noise(kind, B, orc.cfg.z_size, g)
    label = 0 if unconditional else K - 1
    step = eng.step_d if kind == "d" else eng.step_c
    l0 = eng.launch_count()
    loss = step(xb, label, noise=dev, flags=0 if update else STEP_NO_UPDATE).clone()
    launches = eng.launch_count() - l0
    torch.cuda.synchronize()
    out = _snapshot(eng, kind, B)
    out["loss"] = loss
    eng.close()
    return out, launches


def _assert_equal(a, b):
    assert a.keys() == b.keys()
    bad = [k for k in a if not torch.equal(a[k], b[k])]
    assert not bad, f"differ: {bad}"


def _assert_chain_matches(kind, F_, K, B, update, unconditional=False):
    fused, n_fused = _step(kind, F_, K, B, 1, update, unconditional)
    layers, n_layers = _step(kind, F_, K, B, 0, update, unconditional)
    # the fused path ran: one chain launch instead of the critic's 8 / the classifier's 10 layer launches
    assert n_fused < n_layers, (n_fused, n_layers)
    _assert_equal(fused, layers)


# (12, 4): first-layer weight rows of 16 (critic, F + K) and 12 (classifier, F) floats take the vectorised weight loads
@pytest.mark.parametrize("F_,K,B", [(10, 5, 64), (10, 4, 333), (30, 5, 128), (12, 4, 256), (10, 5, 4096)])
@pytest.mark.parametrize("kind", ["d", "c"])
@pytest.mark.parametrize("update", [False, True])
def test_chain_step_bit_identical(kind, F_, K, B, update):
    _assert_chain_matches(kind, F_, K, B, update)


@pytest.mark.parametrize("B", [64, 333])
def test_chain_unconditional_critic_bit_identical(B):
    """VAE-GAN's critic has no label column."""
    _assert_chain_matches("d", 10, 5, B, False, unconditional=True)


def test_chain_graph_visit_bit_identical():
    """One CUDA-graph-captured label visit (5 D, 5 C, 3 E/G steps) with and without the chains."""
    from cvae_gan_b200 import models
    from cvae_gan_b200.engine import Engine
    F_, K, B = 10, 5, 1024
    rows = torch.rand(5000, F_, generator=torch.Generator().manual_seed(0)).cuda()
    outs, launches = [], []
    for chain in (1, 0):
        torch.manual_seed(3)
        eng = Engine(F_, K, 128, max_batch=B)
        mods = [models.CVAEGANEncoderModel(F_, K), models.CVAEGANGeneratorModel(128, K, F_),
                models.CVAEGANDiscriminatorModel(F_, K), models.CVAEGANClassifierModel(F_, K)]
        for net, m in enumerate(mods):
            eng.load_state(net, m.state_dict())
        eng.debug_set("chain", chain)
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
        out = _snapshot(eng, "", B)
        out["loss"] = loss.clone()
        outs.append(out)
        del gr
        eng.close()
    assert launches[0] < launches[1], launches
    _assert_equal(outs[0], outs[1])
