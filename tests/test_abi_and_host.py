"""CPU-side checks: the C-ABI library builds, loads and exports every symbol the header declares; host
logic (patience scan, lambda schedule, model mirrors) matches the oracle / the reference fixtures.
No compute calls are made (there is no GPU in this container)."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from oracle import cvae_gan_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from cvae_gan_b200 import _lib
    return _lib.load()


def test_library_exports_every_declared_symbol(lib):
    from cvae_gan_b200 import _lib
    header = open(os.path.join(ROOT, "include", "cvaegan_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(cvg_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations parsed"
    assert declared == set(_lib.SIGNATURES), (declared ^ set(_lib.SIGNATURES))
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.cvg_abi_version() == _lib.ABI_VERSION == 2


def test_create_fails_loudly_without_sm100(lib):
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from cvae_gan_b200 import CvgError, Engine, _lib
    cfg = _lib.CvgConfig(10, 5, 128, 64, 1, 0, 1, .1, 1, 2e-4, 2e-4, 1e-4, .5, .999, 1e-8, .1, 1e-5, 1e-5, 1e-12, .2, .3)
    h = C.c_void_p()
    assert lib.cvg_create(C.byref(cfg), C.byref(h)) != 0
    assert lib.cvg_last_error()
    with pytest.raises(CvgError):
        Engine(10, 5)          # no silent CPU path


def test_patience_scan_matches_oracle(lib):
    from cvae_gan_b200.engine import patience_scan
    g = torch.Generator().manual_seed(0)
    for p_acc, num in ((0.5, 57), (0.02, 40), (0.0, 10), (1.0, 33), (0.3, 1), (0.1, 1000)):
        keep = torch.rand(50000, generator=g) < p_acc
        assert patience_scan(keep, num) == O.patience_scan(keep, num)
    with pytest.raises(Exception, match="too short"):
        patience_scan(torch.zeros(15, dtype=torch.bool), 5)


def test_lambda_class_schedule_matches_oracle():
    from cvae_gan_b200 import lambda_class_at
    for e in (0, 1, 199, 200, 201, 350, 499, 500, 10000):
        assert lambda_class_at(e, 0.5) == O.lambda_class_schedule(e, 0.5)


def _assert_init_equal(got, ref, where):
    """Everything drawn from the seeded generator must be bit-identical.  Spectral norm's `_u` / `_v` are 15 power-iteration
    steps (torch.mv) run at construction: the BLAS code path the host CPU selects moves their last bits, so those two
    vectors are held to 1e-6.  The fixtures match bit for bit where MKL runs its AVX-512 kernels; on the same host,
    MKL_ENABLE_INSTRUCTIONS=AVX2 (or SSE4_2) moves `_u` / `_v` by up to 2e-7 (7 ulp) and nothing else."""
    if where[-1].endswith(("._u", "._v")):
        torch.testing.assert_close(got, ref, rtol=1e-5, atol=1e-6, msg=str(where))
    else:
        assert torch.equal(got, ref), where


def test_model_mirrors_reproduce_reference_init(golden_dir):
    """Same seed -> same starting parameters as the reference constructor (fixture: reference state_dicts
    right after `set_random_state(); CVAEGAN()`, see oracle/make_golden.py)."""
    import random
    from cvae_gan_b200 import models
    npz = np.load(os.path.join(golden_dir, "ref_fit_a.npz"))
    random.seed(0); np.random.seed(0); torch.manual_seed(0)
    nets = {
        "encoder": models.CVAEGANEncoderModel(10, 5, 128),
        "generator": models.CVAEGANGeneratorModel(128, 5, 10),
        "discriminator": models.CVAEGANDiscriminatorModel(10, 5),
        "classifier": models.CVAEGANClassifierModel(10, 5),
    }
    for name, mod in nets.items():
        sd = mod.state_dict()
        ref_keys = [k.split("/", 2)[2] for k in npz.files if k.startswith(f"init/{name}/")]
        assert list(sd.keys()) == ref_keys
        for k, v in sd.items():
            _assert_init_equal(v, torch.from_numpy(npz[f"init/{name}/{k}"]), (name, k))
        assert [k for k, _, _ in O.tensor_table(name, 10, 5, 128)] == ref_keys


def test_model_mirrors_keep_reference_error_behaviour():
    from cvae_gan_b200 import models
    torch.manual_seed(1)
    E = models.CVAEGANEncoderModel(10, 5)
    G = models.CVAEGANGeneratorModel(128, 5, 10)
    D = models.CVAEGANDiscriminatorModel(10, 5)
    Cm = models.CVAEGANClassifierModel(10, 5)
    with pytest.raises(ValueError):
        E(torch.zeros(4, 11), torch.zeros(4, dtype=torch.long))
    with pytest.raises(ValueError):
        E(torch.zeros(4, 10), torch.zeros(4, 2))
    with pytest.raises(ValueError):
        G(torch.zeros(4, 128), torch.zeros(4, dtype=torch.long))       # 1-D condition (cvae_gan_models.py:142)
    with pytest.raises(ValueError):
        G(torch.zeros(4, 127), torch.zeros(4, 5))
    with pytest.raises(ValueError):
        D(torch.zeros(4, 10), torch.zeros(3, dtype=torch.long))
    E.eval(); G.eval(); D.eval(); Cm.eval()
    mu, lv = E(torch.rand(4, 10), torch.tensor([0, 1, 2, 3]))
    assert mu.shape == (4, 128) and lv.shape == (4, 128)
    assert G(torch.randn(4, 128), torch.eye(5)[:4]).shape == (4, 10)
    assert D(torch.rand(4, 10), torch.tensor([1, 1, 1, 1])).shape == (4, 1)
    assert Cm(torch.rand(4, 10)).shape == (4, 5)


def test_oracle_models_equal_mirror_forward():
    """The torch mirrors (state containers) and the oracle compute the same function."""
    from cvae_gan_b200 import models
    torch.manual_seed(3)
    mods = {"encoder": models.CVAEGANEncoderModel(10, 5), "generator": models.CVAEGANGeneratorModel(128, 5, 10),
            "discriminator": models.CVAEGANDiscriminatorModel(10, 5), "classifier": models.CVAEGANClassifierModel(10, 5)}
    orc = O.OracleCVAEGAN(10, 5).load_state({k: m.state_dict() for k, m in mods.items()})
    for m in mods.values():
        m.eval()
    x = torch.rand(16, 10)
    z = torch.randn(16, 128)
    with torch.no_grad():
        assert torch.allclose(mods["generator"](z, torch.eye(5)[torch.full((16,), 2)]),
                              O.generator_forward(orc.sd["generator"], z, 2, False), atol=1e-6)
        assert torch.allclose(mods["classifier"](x), O.classifier_forward(orc.sd["classifier"], x, False), atol=1e-6)
        assert torch.allclose(mods["discriminator"](x, torch.full((16,), 1)),
                              O.discriminator_forward(orc.sd["discriminator"], x, 1, False), atol=1e-6)
        mu, lv = mods["encoder"](x, torch.full((16,), 4))
        omu, olv = O.encoder_forward(orc.sd["encoder"], x, 4, False)
        assert torch.allclose(mu, omu, atol=1e-6) and torch.allclose(lv, olv, atol=1e-6)


def test_pipeline_minmax_and_pickle_format(tmp_path):
    """Driver plumbing (scripts/train_cvae_gan.py:19-43, 131-140) on the CPU: joint min-max scaling equals sklearn's
    minmax_scale on the concatenation, the result is shifted to a zero minimum, and the pickle is the 4-tuple of numpy
    arrays the reference's tools read."""
    import pickle
    import numpy as np
    from sklearn.preprocessing import minmax_scale
    from cvae_gan_b200 import datasets as ds
    from cvae_gan_b200 import pipeline
    g = torch.Generator().manual_seed(3)
    tr = torch.randn(50, 6, generator=g) * 7 + 3
    te = torch.randn(20, 6, generator=g) * 7 + 3
    tr[:, 2] = 1.5
    te[:, 2] = 1.5                                   # constant column
    saved = (ds.tr_samples, ds.tr_labels, ds.te_samples, ds.te_labels, ds.feature_num, ds.label_num)
    try:
        ds.tr_samples, ds.te_samples = tr.clone(), te.clone()
        ds.tr_labels = torch.arange(50) % 4
        ds.te_labels = torch.arange(20) % 4
        pipeline.minmax_scale_(ds, device="cpu")
        ref = minmax_scale(torch.cat([tr, te]).numpy())
        ref = ref - ref.min()
        assert np.allclose(torch.cat([ds.tr_samples, ds.te_samples]).numpy(), ref, atol=1e-6)
        assert ds.feature_num == 6 and ds.label_num == 4
        out = str(tmp_path / "d.pkl")
        pipeline.dump_dataset(out, ds)
        with open(out, "rb") as f:
            a, b, c, d = pickle.load(f)
        assert a.shape == (50, 6) and b.shape == (50,) and c.shape == (20, 6) and d.shape == (20,)
    finally:
        ds.tr_samples, ds.tr_labels, ds.te_samples, ds.te_labels, ds.feature_num, ds.label_num = saved


def test_flag_values_match_the_header():
    """The Python constants are the header's enum values (include/cvaegan_b200.h)."""
    import re
    from cvae_gan_b200 import _lib
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "cvaegan_b200.h")).read()
    vals = {k: int(v) for k, v in re.findall(r"(CVG_(?:STEP|VISIT)_[A-Z_]+)\s*=\s*(\d+)", hdr)}
    assert vals == {"CVG_STEP_NO_UPDATE": _lib.STEP_NO_UPDATE, "CVG_STEP_LOCAL_BN": _lib.STEP_LOCAL_BN,
                    "CVG_VISIT_LAMBDA_ZERO": _lib.VISIT_LAMBDA_ZERO, "CVG_STEP_PRIOR_ONLY": _lib.STEP_PRIOR_ONLY,
                    "CVG_STEP_CVAE": _lib.STEP_CVAE}


def test_cgan_host_class_mirrors_the_reference_surface():
    """src/cgan.py:10-309: attribute and method names a caller of the reference's CGAN uses (no GPU: class level only)."""
    import cvae_gan_b200 as cg
    for name in ("fit", "_divide_samples", "_get_target_samples", "plot_loss_history", "generate_samples", "generate_qualified_samples"):
        assert callable(getattr(cg.CGAN, name)), name
    assert cg.config.gan_config.cgan_config == {"lambda_adv": 1.0, "lambda_class": 0.5, "confidence_threshold": 0.5}
    from cvae_gan_b200 import cgan, models
    assert cgan.CGANGeneratorModel is models.CVAEGANGeneratorModel      # same layers and state_dict keys (cgan_models.py)
    assert cg.CGAN._HISTORY == (("adv_loss", 2), ("class_loss", 3)) and not cg.CGAN._USES_ENCODER


def test_cvae_host_class_mirrors_the_reference_surface():
    """src/cvae.py:11-319: attribute and method names a caller of the reference's CVAE uses (no GPU: class level only)."""
    import cvae_gan_b200 as cg
    for name in ("fit", "_divide_samples", "_get_target_samples", "plot_loss_history", "generate_samples",
                 "generate_qualified_samples", "reconstruct_samples"):
        assert callable(getattr(cg.CVAE, name)), name
    assert cg.config.gan_config.cvae_config == {"lambda_recon": 1.0, "lambda_kl": 0.01, "lambda_class": 0.1,
                                                "confidence_threshold": 0.5}
    from cvae_gan_b200 import cvae, models
    assert cvae.CVAEEncoderModel is models.CVAEGANEncoderModel          # same layers and state_dict keys (cvae_models.py)
    assert cg.CVAE._HISTORY == (("recon_loss", 0), ("kl_loss", 1), ("class_loss", 3)) and not cg.CVAE._USES_CRITIC

    class _GC:
        d_loop_num, c_loop_num, g_loop_num = 5, 4, 3
    assert cg.CVAE._loops(None, _GC) == (0, 4, 3) and cg.CVAEGAN._loops(None, _GC) == (5, 4, 3)    # cvae.py:86-117: no critic steps


@pytest.mark.parametrize("cls_name,fixture,nets", [("CVAEGAN", "ref_fit_a.npz", ("encoder", "generator", "discriminator", "classifier")),
                                                   ("CGAN", "ref_cgan_a.npz", ("generator", "discriminator", "classifier")),
                                                   ("CVAE", "ref_cvae_a.npz", ("encoder", "generator", "classifier"))])
def test_host_classes_build_networks_in_the_reference_order(golden_dir, cls_name, fixture, nets):
    """Same seed -> the starting parameters of the reference class: each trainer constructs its networks in its own order
    (cvae_gan.py:19-39, cgan.py:20-34, cvae.py:19-34), which fixes the CPU-generator draws; the networks a sibling does not
    have are built afterwards without touching the stream.  Fixtures: state_dicts right after `set_random_state(); <class>()`."""
    import random
    import cvae_gan_b200 as cg
    npz = np.load(os.path.join(golden_dir, fixture))
    random.seed(0); np.random.seed(0); torch.manual_seed(0)
    built = getattr(cg, cls_name)._build_networks(10, 5, 128)
    after = torch.rand(1)
    assert sorted(built) == ["classifier", "discriminator", "encoder", "generator"]
    for name in nets:
        sd = built[name].state_dict()
        ref_keys = [k.split("/", 2)[2] for k in npz.files if k.startswith(f"init/{name}/")]
        assert list(sd.keys()) == ref_keys
        for k, v in sd.items():
            _assert_init_equal(v, torch.from_numpy(npz[f"init/{name}/{k}"]), (cls_name, name, k))
    # the extra networks did not advance the generator: the next draw is the one the reference would make
    random.seed(0); np.random.seed(0); torch.manual_seed(0)
    from cvae_gan_b200 import models
    ctor = {"encoder": lambda: models.CVAEGANEncoderModel(10, 5, 128), "generator": lambda: models.CVAEGANGeneratorModel(128, 5, 10),
            "discriminator": lambda: models.CVAEGANDiscriminatorModel(10, 5), "classifier": lambda: models.CVAEGANClassifierModel(10, 5)}
    for name in getattr(cg, cls_name)._BUILD_ORDER:
        ctor[name]()
    assert torch.equal(after, torch.rand(1))


def test_bench_flop_accounting_reproduces_the_survey_figures():
    """bench.flop_per_train_sample generalises SURVEY.md 8(d)'s minimal-work accounting to any layer widths (needed for the
    widened model); at the reference's widths it must give the SURVEY figures: 873 945 (F=10, K=5), 871 463 (OTIDS K=4),
    925 145 (F=30, K=5)."""
    import bench
    assert round(bench.flop_per_train_sample(10, 5, 128)) == 873_945 == bench.FLOP_PER_SAMPLE
    assert round(bench.flop_per_train_sample(10, 4, 128)) == 871_463
    assert round(bench.flop_per_train_sample(30, 5, 128)) == 925_145
    assert bench.flop_per_train_sample(10, 5, 128, (256, 128, 64)) == bench.flop_per_train_sample(10, 5, 128)
    assert bench.flop_per_train_sample(10, 5, 128, bench.WIDE_HIDDEN) > 10 * bench.FLOP_PER_SAMPLE


def test_vaegan_host_class_and_model_mirrors():
    """src/vae_gan.py:10-261 and src/models/vae_gan_models.py: the surface a caller of the reference's VAEGAN uses, and the
    unconditional mirrors (same keys as the CVAE-GAN's stacks, first Linear without label columns, forwards without condition)."""
    import cvae_gan_b200 as cg
    from cvae_gan_b200 import models
    for name in ("fit", "_store_samples", "_get_random_samples", "plot_loss_history", "generate_samples", "reconstruct_samples"):
        assert callable(getattr(cg.VAEGAN, name)), name
    assert cg.config.gan_config.vae_gan_config == {"lambda_recon": 1.0, "lambda_kl": 0.01, "lambda_adv": 0.1,
                                                   "confidence_threshold": 0.5}
    torch.manual_seed(2)
    E, G, D = models.VAEGANEncoderModel(10, 128), models.VAEGANGeneratorModel(128, 10), models.VAEGANDiscriminatorModel(10)
    assert E.state_dict()["encoder.0.weight"].shape == (256, 10) and G.state_dict()["main_model.0.weight"].shape == (256, 128)
    assert D.state_dict()["discriminator_network.0.parametrizations.weight.original"].shape == (256, 10)
    assert [k for k, _, _ in O.tensor_table("encoder", 10, 5, 128, unconditional=True)] == list(E.state_dict().keys())
    assert [tuple(s) for _, s, _ in O.tensor_table("discriminator", 10, 5, 128, unconditional=True)] == \
           [tuple(v.shape) for v in D.state_dict().values()]
    for m in (E, G, D):
        m.eval()
    x = torch.rand(6, 10)
    mu, lv = E(x)
    assert mu.shape == lv.shape == (6, 128) and G(mu).shape == (6, 10) and D(x).shape == (6, 1)
    with pytest.raises(ValueError):
        E(torch.zeros(4, 11))
    with pytest.raises(ValueError):
        G(torch.zeros(4, 127))
    # same arithmetic as the oracle's unconditional forwards on the same state
    sd = {k: v.detach() for k, v in E.state_dict().items()}
    mu_o, lv_o = O.encoder_forward(sd, x, None, False, None)
    assert torch.allclose(mu, mu_o, atol=1e-6) and torch.allclose(lv, lv_o, atol=1e-6)


def test_dataset_tensors_honours_the_dataset_that_is_passed_in():
    """cvae_gan.py:238-245 iterates `for sample, label in dataset`: whatever dataset is PASSED is what gets partitioned - this
    package's own Dataset (fast path), torch's TensorDataset (its `.tensors` is a tuple, not a method), a same-length subset or
    permutation of the global training set (no length heuristics), or any indexable dataset."""
    from torch.utils.data import Subset, TensorDataset
    import cvae_gan_b200 as cg
    from cvae_gan_b200.cvae_gan import dataset_tensors
    g = torch.Generator().manual_seed(5)
    x, y = torch.rand(40, 6, generator=g), torch.randint(0, 3, (40,), generator=g)
    saved = (cg.datasets.tr_samples, cg.datasets.tr_labels)
    try:
        cg.datasets.tr_samples, cg.datasets.tr_labels = x, y
        a, b = dataset_tensors(cg.datasets.TrDataset())
        assert torch.equal(a, x) and torch.equal(b, y)
        perm = torch.randperm(40, generator=g)
        a, b = dataset_tensors(TensorDataset(x[perm], y[perm]))              # same length as the globals, different rows
        assert torch.equal(a, x[perm]) and torch.equal(b, y[perm])
        a, b = dataset_tensors(Subset(TensorDataset(x, y), list(range(0, 40, 3))))
        assert torch.equal(a, x[::3]) and torch.equal(b, y[::3])

        class Plain:
            def __len__(self):
                return 5

            def __getitem__(self, i):
                return x[i + 10], int(y[i + 10])
        a, b = dataset_tensors(Plain())
        assert torch.equal(a, x[10:15]) and b.tolist() == y[10:15].tolist()
    finally:
        cg.datasets.tr_samples, cg.datasets.tr_labels = saved


def test_header_is_plain_c_and_a_c_program_links_against_the_library(lib, tmp_path):
    """The drop-in boundary is a C ABI: include/cvaegan_b200.h must compile as C99 (no C++ in the signatures) and a C program
    that includes it must link against libcvaegan_b200.so and agree with it on the ABI version and the size of CvgConfig.
    No compute call is made (no GPU here)."""
    import shutil
    import subprocess
    from cvae_gan_b200 import _lib
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no gcc")
    src = tmp_path / "abi_check.c"
    src.write_text('#include <stdio.h>\n#include "cvaegan_b200.h"\n'
                   'int main(void) {\n'
                   '  CvgConfig c; (void)c;\n'
                   '  printf("%d %d %d %d\\n", cvg_abi_version(), CVG_ABI_VERSION, cvg_config_bytes(), (int)sizeof(CvgConfig));\n'
                   '  return cvg_abi_version() == CVG_ABI_VERSION && cvg_config_bytes() == (int)sizeof(CvgConfig) ? 0 : 1;\n}\n')
    exe = tmp_path / "abi_check"
    libdir = os.path.dirname(_lib.LIB_PATH)
    subprocess.run([gcc, "-std=c99", "-Wall", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe),
                    "-L", libdir, "-l:libcvaegan_b200.so", f"-Wl,-rpath,{libdir}"], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr
    a, b, c, d = [int(v) for v in out.stdout.split()]
    assert a == b == _lib.ABI_VERSION and c == d == C.sizeof(_lib.CvgConfig)
