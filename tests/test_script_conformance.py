"""Static drop-in check against the reference's OWN driver scripts (the checks that parse them need
a reference checkout named by MRI_REFERENCE_DIR and skip without one).  The scripts cannot be
executed here (they import mlflow, perun, nibabel and build datasets at import time -- SURVEY.md
8c), so their source is parsed instead: every name they import from the hot-path modules must
exist in the overlay package, and every constructor / method call they make on those classes
must bind to the drop-in's signature with the same positional and keyword arguments.  (Executing the scripts needs a GPU next to the
reference: tools/run_reference_scripts.py / tests/test_gpu_scripts.py, logs under profiles/r04*.)"""
import ast
import contextlib
import importlib
import inspect
import io
import os

import pytest

REF = os.path.join(os.environ.get("MRI_REFERENCE_DIR") or "/nonexistent", "model_scripts")
needs_reference = pytest.mark.skipif(not os.path.isdir(REF), reason="needs a reference checkout (MRI_REFERENCE_DIR)")

HOT_MODULES = {"unet", "unet_attention", "diffusion", "vae"}
SCRIPTS = {
    "slice_cond_2d_ddpm": ["model.py", "show_model.py", "metrics.py"],
    "ddpm_25d_all_modalities": ["model.py", "show_model.py", "metrics.py", "generate_pseudo3d_volume.py",
                                "metrics_both.py"],
    "ddpm_3d_ldm": ["train.py", "show_model.py"],
}
METHODS = {"q_sample", "p_losses", "p_sample", "p_sample_loop", "sample", "sample_from", "p_sample_ddim",
           "sample_from_ddim", "encode_to_latent", "decode_from_latent", "encode", "decode", "reparameterize"}


def overlay(pkg, mod):
    return importlib.import_module(f"mri_image_generation_b200.model_scripts.{pkg}.{mod}")


def parse(pkg, script):
    path = os.path.join(REF, pkg, script)
    if not os.path.exists(path):
        return None
    return ast.parse(open(path).read(), filename=path)


def bind_ok(fn, n_pos, kw_names, drop_self=True):
    sig = inspect.signature(fn)
    params = list(sig.parameters.values())
    if drop_self and params and params[0].name == "self":
        sig = sig.replace(parameters=params[1:])
    try:
        sig.bind(*([None] * n_pos), **{k: None for k in kw_names})
        return True
    except TypeError:
        return False


@needs_reference
@pytest.mark.parametrize("pkg", sorted(SCRIPTS))
def test_imports_and_calls_of_reference_scripts_bind_to_the_drop_in(pkg):
    checked_imports = checked_ctor = checked_methods = 0
    for script in SCRIPTS[pkg]:
        tree = parse(pkg, script)
        if tree is None:
            continue
        classes = {}
        for node in ast.walk(tree):
            if isinstance(node, ast.ImportFrom) and node.level == 1 and node.module in HOT_MODULES:
                mod = overlay(pkg, node.module)
                for a in node.names:
                    assert hasattr(mod, a.name), f"{pkg}/{script}: from .{node.module} import {a.name}"
                    classes[a.asname or a.name] = getattr(mod, a.name)
                    checked_imports += 1
        # cross-package aliases (metrics_both.py imports both UNets under other names) are resolved
        # the same way because ImportFrom with level 2 names the sibling package explicitly
        for node in ast.walk(tree):
            if isinstance(node, ast.ImportFrom) and node.level == 2 and node.module:
                parts = node.module.split(".")
                if len(parts) == 2 and parts[1] in HOT_MODULES and parts[0] in SCRIPTS:
                    mod = overlay(parts[0], parts[1])
                    for a in node.names:
                        assert hasattr(mod, a.name), f"{pkg}/{script}: from ..{node.module} import {a.name}"
                        classes[a.asname or a.name] = getattr(mod, a.name)
                        checked_imports += 1
        all_methods = {}
        for c in classes.values():
            if inspect.isclass(c):
                for m in METHODS:
                    if hasattr(c, m):
                        all_methods.setdefault(m, []).append(getattr(c, m))
        for node in ast.walk(tree):
            if not isinstance(node, ast.Call):
                continue
            kw = [k.arg for k in node.keywords if k.arg is not None]
            if any(k.arg is None for k in node.keywords) or any(isinstance(a, ast.Starred) for a in node.args):
                continue  # **kwargs / *args forwarding: nothing to bind statically
            if isinstance(node.func, ast.Name) and node.func.id in classes and inspect.isclass(classes[node.func.id]):
                cls = classes[node.func.id]
                # metrics_both.py deliberately tries one keyword set and falls back on TypeError
                in_try = script == "metrics_both.py"
                ok = bind_ok(cls.__init__, len(node.args), kw)
                assert ok or in_try, f"{pkg}/{script}:{node.lineno} {node.func.id}({len(node.args)} args, {kw})"
                checked_ctor += 1
            elif isinstance(node.func, ast.Attribute) and node.func.attr in all_methods:
                cands = all_methods[node.func.attr]
                assert any(bind_ok(f, len(node.args), kw) for f in cands), \
                    f"{pkg}/{script}:{node.lineno} .{node.func.attr}({len(node.args)} args, {kw})"
                checked_methods += 1
    print(f"{pkg}: {checked_imports} imports, {checked_ctor} constructor calls, {checked_methods} method calls bind")
    assert checked_imports >= 2 and checked_methods >= 1


def test_attributes_read_by_the_scripts_exist():
    """diffusion.model / .timesteps / .betas / .channels / .image_size, unet.in_channels / .chs
    (SURVEY.md 8b 'Attributes read by callers')."""
    with contextlib.redirect_stdout(io.StringIO()):
        U2 = overlay("slice_cond_2d_ddpm", "unet").UNet
        G2 = overlay("slice_cond_2d_ddpm", "diffusion").GaussianDiffusion
        U3 = overlay("ddpm_3d_ldm", "unet_attention").UNet3DModelWithAttention
        G3 = overlay("ddpm_3d_ldm", "diffusion").GaussianDiffusionLatent3D
        u2 = U2(img_channels=1, base_channels=16, channel_mults=(1, 2), time_emb_dim=32)
        d2 = G2(u2, 32, channels=1, timesteps=20)
        u3 = U3(3, base_channels=16, channel_mults=(1, 2), time_emb_dim=32)
        d3 = G3(u3, 3, timesteps=20)
    assert d2.model is u2 and d2.timesteps == 20 and d2.image_size == 32 and d2.channels == 1
    assert d3.model is u3 and d3.timesteps == 20 and d3.channels == 3
    assert d2.betas.numel() == 20 and d3.betas.device.type == "cpu"
    assert u3.in_channels == 3 and list(u3.chs) == [16, 32]


@needs_reference
def test_ddp_calls_of_the_training_script_bind_to_the_overlapped_wrapper():
    """ddpm_3d_ldm/train.py wraps the UNet as `DDP(unet, device_ids=[local_rank],
    output_device=local_rank, find_unused_parameters=False)` and later unwraps `.module`: every such
    call must bind to mri_image_generation_b200.parallel.DistributedDataParallel (the drop-in whose
    all-reduce overlaps the backward launch list), so that switching is a one-line import change."""
    from mri_image_generation_b200.parallel import DistributedDataParallel
    tree = parse("ddpm_3d_ldm", "train.py")
    sig = inspect.signature(DistributedDataParallel.__init__)
    calls = [n for n in ast.walk(tree) if isinstance(n, ast.Call) and isinstance(n.func, ast.Name) and n.func.id == "DDP"]
    assert len(calls) >= 2
    for c in calls:
        args = [object()] * (1 + len(c.args))                  # self + positional
        kwargs = {k.arg: object() for k in c.keywords}
        sig.bind(*args, **kwargs)                               # raises TypeError if it does not fit
    src = open(os.path.join(REF, "ddpm_3d_ldm", "train.py")).read()
    assert ".module" in src
    assert "module" in inspect.getsource(DistributedDataParallel.__init__)
    assert hasattr(DistributedDataParallel, "no_sync") and hasattr(DistributedDataParallel, "forward")
