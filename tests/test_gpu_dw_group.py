"""The grouped weight-gradient launch of the D and C steps (launch_dw_group, gemm_dw_group_kernel) against the per-layer
launches of the layer-kernel path (cvg_debug_set("chain", 0)).  A sequence of eager steps must end with bit-identical
parameters, gradients, Adam moments, BatchNorm / spectral-norm state and losses: a slot or counter that one group (or the
classifier chain's LayerNorm sums on the same stream) left dirty would change the next step's gradients."""
import pytest
import torch

from tests import parity as P

pytestmark = pytest.mark.gpu

# launches per step saved by the chain with the grouped weight gradients: the critic chain replaces 8 layer launches by
# 1 and its 5 weight-gradient launches become 1; the classifier chain replaces 10 by 1 and its 4 become 1
SAVED = {"d": 11, "c": 12}


def _sequence(kinds, F_, K, B, chain, unconditional=False):
    orc, eng, g = P.make_pair(F_, K, B, seed=5 + B, unconditional=unconditional)
    eng.debug_set("chain", chain)
    x, y = P.make_data(F_, K, [B] * K, seed=2)
    xb = x[y == (K - 1)][:B].contiguous().cuda()
    label = 0 if unconditional else K - 1
    losses, launches = [], []
    for kind in kinds:
        _, dev = P.draw_noise(kind, B, orc.cfg.z_size, g)
        step = eng.step_d if kind == "d" else eng.step_c
        l0 = eng.launch_count()
        losses.append(step(xb, label, noise=dev).clone())
        launches.append(eng.launch_count() - l0)
    torch.cuda.synchronize()
    out = {"loss": torch.stack(losses)}
    for n in range(4):
        for which in ("params", "grads", "adam_m", "adam_v", "state"):
            out[f"{which}{n}"] = getattr(eng, which)[n].clone()
    eng.close()
    return out, launches


def _assert_group_matches(kinds, F_, K, B, unconditional=False):
    grouped, n_grouped = _sequence(kinds, F_, K, B, 1, unconditional)
    layers, n_layers = _sequence(kinds, F_, K, B, 0, unconditional)
    assert [b - a for a, b in zip(n_grouped, n_layers)] == [SAVED[k] for k in kinds], (n_grouped, n_layers)
    assert grouped.keys() == layers.keys()
    bad = [k for k in grouped if not torch.equal(grouped[k], layers[k])]
    assert not bad, f"differ: {bad}"


@pytest.mark.parametrize("F_,K,B", [(10, 5, 64), (10, 4, 333), (10, 5, 4096), (30, 5, 333)])
def test_dw_group_sequence_bit_identical(F_, K, B):
    _assert_group_matches("ddccd", F_, K, B)


@pytest.mark.parametrize("B", [64, 4096])
def test_dw_group_unconditional_critic_bit_identical(B):
    """VAE-GAN's critic: no label column in the first layer's weight gradient."""
    _assert_group_matches("ddd", 10, 5, B, unconditional=True)
