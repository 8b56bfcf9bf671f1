"""ORACLE -- test infrastructure only (see oracle/README.md).

Imports the reference's own Python modules from the read-only checkout at /root/reference so that the
restatements in oracle/hy3d_ref.py can be pinned against them and golden fixtures can be generated
(oracle/make_golden.py).  /root/reference does not exist on the GPU box: nothing at test run time on the
GPU depends on this file.

`import hy3dgen.shapegen` itself fails here (trimesh / skimage / diffusers are not installed), so the
sub-modules that only need torch/einops are loaded through stub parent packages (SURVEY.md section 8c).
"""
import importlib
import importlib.util
import os
import sys
import types

REF_ROOT = os.environ.get("R3G_REFERENCE", "/root/reference")
HY = os.path.join(REF_ROOT, "Hunyuan3D-2")
VGGT = os.path.join(REF_ROOT, "vggt")


def available():
    return os.path.isdir(os.path.join(HY, "hy3dgen"))


def _stub_pkg(name, path):
    if name in sys.modules:
        return sys.modules[name]
    m = types.ModuleType(name)
    m.__path__ = [path]
    sys.modules[name] = m
    return m


def _load_file(mod_name, path):
    spec = importlib.util.spec_from_file_location(mod_name, path)
    m = importlib.util.module_from_spec(spec)
    sys.modules[mod_name] = m
    spec.loader.exec_module(m)
    return m


def hunyuan_dit():
    """Hunyuan3D-2/hy3dgen/shapegen/models/denoisers/hunyuan3ddit.py (torch + einops only)."""
    return _load_file("_ref_hunyuan3ddit",
                      os.path.join(HY, "hy3dgen/shapegen/models/denoisers/hunyuan3ddit.py"))


def hunyuan_autoencoders():
    """attention_blocks / attention_processors / volume_decoders through stub packages (no skimage)."""
    base = os.path.join(HY, "hy3dgen")
    _stub_pkg("hy3dgen", base)
    _stub_pkg("hy3dgen.shapegen", os.path.join(base, "shapegen"))
    _stub_pkg("hy3dgen.shapegen.models", os.path.join(base, "shapegen/models"))
    _stub_pkg("hy3dgen.shapegen.models.autoencoders", os.path.join(base, "shapegen/models/autoencoders"))
    ab = importlib.import_module("hy3dgen.shapegen.models.autoencoders.attention_blocks")
    ap = importlib.import_module("hy3dgen.shapegen.models.autoencoders.attention_processors")
    vd = importlib.import_module("hy3dgen.shapegen.models.autoencoders.volume_decoders")
    return ab, ap, vd


def hunyuan_preprocessors():
    return _load_file("_ref_preprocessors", os.path.join(HY, "hy3dgen/shapegen/preprocessors.py"))


def hunyuan_conditioner():
    return _load_file("_ref_conditioner", os.path.join(HY, "hy3dgen/shapegen/models/conditioner.py"))


def vggt_package():
    if VGGT not in sys.path:
        sys.path.insert(0, VGGT)
    import vggt  # noqa: F401
    return importlib.import_module("vggt")


def hunyuan_scheduler():
    """schedulers.py needs three names from diffusers (absent here): minimal stand-ins that only record the
    constructor arguments as `.config`, which is all the Euler scheduler's arithmetic uses."""
    if "diffusers" not in sys.modules:
        import functools
        import inspect
        import logging as _logging

        d = types.ModuleType("diffusers")
        cu = types.ModuleType("diffusers.configuration_utils")
        su = types.ModuleType("diffusers.schedulers")
        ssu = types.ModuleType("diffusers.schedulers.scheduling_utils")
        ut = types.ModuleType("diffusers.utils")

        class ConfigMixin:
            pass

        def register_to_config(init):
            @functools.wraps(init)
            def wrapped(self, *a, **kw):
                sig = inspect.signature(init)
                bound = sig.bind(self, *a, **kw)
                bound.apply_defaults()
                self.config = types.SimpleNamespace(**{k: v for k, v in bound.arguments.items() if k != "self"})
                init(self, *a, **kw)
            return wrapped

        class SchedulerMixin:
            pass

        class BaseOutput:
            pass

        cu.ConfigMixin, cu.register_to_config = ConfigMixin, register_to_config
        ssu.SchedulerMixin = SchedulerMixin
        ut.BaseOutput = BaseOutput
        ut.logging = types.SimpleNamespace(get_logger=_logging.getLogger)
        d.configuration_utils, d.schedulers, d.utils = cu, su, ut
        su.scheduling_utils = ssu
        for m in (d, cu, su, ssu, ut):
            sys.modules[m.__name__] = m
    return _load_file("_ref_schedulers", os.path.join(HY, "hy3dgen/shapegen/schedulers.py"))
