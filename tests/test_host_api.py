"""Host-side drop-in contract (CPU): class signatures, state_dict keys/shapes, bit-exact
schedule buffers, loud failure without a GPU, and that libmri_b200.so exports the C ABI."""
import contextlib
import ctypes
import io
import os
import pickle
import re

import pytest
import torch

from helpers import ROOT, check_schedule_against_gold, load_gold
from oracle import reference_oracle as O


def quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


def test_library_exports_every_declared_symbol():
    from mri_image_generation_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "mri_b200.h")).read()
    declared = set(re.findall(r"\b(mri_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name
    assert _lib.load().mri_abi_version() == 1


def test_gemm_args_struct_matches_header_size():
    from mri_image_generation_b200 import _lib
    # 5 pointers + 2 ints + 12 ints + 3 ints + 2 ints + 2 ints + 3 pointers + int + pointer(+pad) ...
    assert ctypes.sizeof(_lib.MriGemmArgs) % 8 == 0
    assert _lib.MriGemmArgs.bias.offset % 8 == 0 and _lib.MriGemmArgs.stats.offset % 8 == 0


@pytest.mark.parametrize("gold,path,cls", [
    ("unet3d_attn", "ddpm_3d_ldm.unet_attention", "UNet3DModelWithAttention"),
    ("unet3d", "ddpm_3d_ldm.unet", "UNet3DModel"),
    ("unet2d", "slice_cond_2d_ddpm.unet", "UNet"),
    ("unet25d", "ddpm_25d_all_modalities.unet", "UNet"),
])
def test_state_dict_keys_and_shapes_match_reference(gold, path, cls):
    import importlib
    g = load_gold(f"{gold}.pt")
    mod = importlib.import_module(f"mri_image_generation_b200.model_scripts.{path}")
    m = quiet(getattr(mod, cls), **g["kwargs"])
    got = [(k, tuple(v.shape)) for k, v in m.state_dict().items()]
    assert got == [(k, tuple(s)) for k, s in g["shapes"]]
    # picklable (mlflow.pytorch.log_model, slice_cond_2d_ddpm/model.py:320)
    pickle.loads(pickle.dumps(m))


def test_constructor_kwargs_are_exclusive():
    """metrics_both.py:154-175 tries in_channels= first and falls back on TypeError."""
    from mri_image_generation_b200.model_scripts.slice_cond_2d_ddpm.unet import UNet as U2
    from mri_image_generation_b200.model_scripts.ddpm_25d_all_modalities.unet import UNet as U25
    with pytest.raises(TypeError):
        quiet(U2, in_channels=1, out_channels=1)
    with pytest.raises(TypeError):
        quiet(U25, img_channels=1)


@pytest.mark.parametrize("name", ["linear_1000", "linear_50", "linear25_1000", "cosine_1000", "cosine_400"])
def test_diffusion_buffers_bit_exact(name):
    g = load_gold("schedules.pt")[name]
    T = g["T"]
    stub = torch.nn.Identity()
    if name.startswith("cosine"):
        from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.diffusion import GaussianDiffusionLatent3D
        d = quiet(GaussianDiffusionLatent3D, stub, 3, timesteps=T)
    elif name.startswith("linear25"):
        from mri_image_generation_b200.model_scripts.ddpm_25d_all_modalities.diffusion import GaussianDiffusion
        d = quiet(GaussianDiffusion, stub, 16, channels=4, timesteps=T)
    else:
        from mri_image_generation_b200.model_scripts.slice_cond_2d_ddpm.diffusion import GaussianDiffusion
        d = quiet(GaussianDiffusion, stub, 16, channels=1, timesteps=T)
    sd = d.state_dict()
    # the reference's formulas on this torch build, bit for bit; the reference's recorded values
    betas = O.cosine_betas(T) if name.startswith("cosine") else O.linear_betas(T)
    want = O.schedule_buffers(betas, with_snr=("snr" in g["sha"]))
    assert list(sd) == list(want)
    for k, v in sd.items():
        assert torch.equal(v, want[k]), k
    check_schedule_against_gold(sd, g)
    assert d.timesteps == T and d.betas.numel() == T


def test_cpu_inputs_fail_loudly():
    from mri_image_generation_b200 import _lib
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.diffusion import GaussianDiffusionLatent3D
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.unet import UNet3DModel
    m = UNet3DModel(3, base_channels=64)
    with pytest.raises(_lib.MriError):
        with torch.no_grad():
            m(torch.zeros(1, 3, 8, 8, 8), torch.zeros(1, dtype=torch.long))
    d = quiet(GaussianDiffusionLatent3D, m, 3, timesteps=10)
    with pytest.raises(_lib.MriError):
        d.q_sample(torch.zeros(1, 3, 8, 8, 8), torch.zeros(1, dtype=torch.long))
    with pytest.raises(_lib.MriError):
        d.sample(1, 8)


def test_product_code_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "mri_image_generation_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dp, f)).read()
                assert "reference_oracle" not in src and "import oracle" not in src and "from oracle" not in src, f


@pytest.mark.parametrize("name", ["vae_b32", "vae_b64_l8"])
def test_vae_state_dict_keys_and_shapes_match_reference(name):
    """VAE3D drop-in (ddpm_3d_ldm/vae.py:90): same keys / shapes as the reference fixture; picklable."""
    from mri_image_generation_b200.model_scripts.ddpm_3d_ldm.vae import VAE3D
    g = load_gold("vae3d.pt")[name]
    m = VAE3D(**g["kwargs"])
    got = [(k, tuple(v.shape)) for k, v in m.state_dict().items()]
    assert got == [(k, tuple(s)) for k, s in g["shapes"]]
    pickle.loads(pickle.dumps(m))


def test_data_parallel_replicas_are_refused_loudly():
    """nn.DataParallel (slice_cond_2d_ddpm/model.py:113-115) replicates the module on every forward;
    static launch programs cannot follow that.  A replica must raise a clear error (the
    supported multi-GPU path is one process per GPU), never run with another replica's buffers."""
    from mri_image_generation_b200 import _lib
    from mri_image_generation_b200.model_scripts.slice_cond_2d_ddpm.unet import UNet
    m = quiet(UNet)
    m._is_replica = True       # what torch.nn.parallel.replicate sets on every replica
    with pytest.raises(_lib.MriError, match="DataParallel"):
        m(torch.zeros(1, 1, 16, 16), torch.zeros(1, dtype=torch.long), torch.zeros(1))
