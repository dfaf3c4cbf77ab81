"""ORACLE tooling: import the reference's OWN Python modules (read-only, from /root/reference) in a container that
lacks diffusers / accelerate / xformers / omegaconf / IPython, by installing minimal stub modules in sys.modules.

Only used by tests/golden/make_golden.py to generate the committed golden vectors, which the tests compare against.
Nothing of the reference is copied; the modules are executed in place.
"""
import importlib.machinery
import importlib.util
import os
import sys
import types

REFERENCE_ROOT = os.environ.get('MOS_REFERENCE_ROOT', '/root/reference')


def reference_available():
    return os.path.isfile(os.path.join(REFERENCE_ROOT, 'mixofshow', 'models', 'edlora.py'))


def _stub(name, **attrs):
    if name in sys.modules:
        mod = sys.modules[name]
    else:
        mod = types.ModuleType(name)
        mod.__spec__ = importlib.machinery.ModuleSpec(name, loader=None)
        mod.__path__ = []  # behave like a package so sub-imports resolve through sys.modules
        sys.modules[name] = mod
        if '.' in name:
            parent, child = name.rsplit('.', 1)
            setattr(_stub(parent), child, mod)
    for k, v in attrs.items():
        setattr(mod, k, v)
    return mod


class _Dummy:
    def __init__(self, *a, **k):
        pass


def install_stubs():
    import numpy as np
    # transformers probes `accelerate` at import time: import it BEFORE the accelerate stub exists
    import transformers
    from transformers import CLIPTextModel, CLIPTokenizer  # noqa: F401  (resolve lazy attributes now)
    if not hasattr(np, 'Inf'):
        np.Inf = np.inf  # gradient_fusion.py:59 uses np.Inf (removed in NumPy 2)

    class AttnProcessor(_Dummy):
        pass

    _stub('diffusers', StableDiffusionPipeline=_Dummy, DDPMScheduler=_Dummy, DPMSolverMultistepScheduler=_Dummy,
          AutoencoderKL=_Dummy, UNet2DConditionModel=_Dummy)
    _stub('diffusers.models', AutoencoderKL=_Dummy, UNet2DConditionModel=_Dummy, T2IAdapter=_Dummy)
    _stub('diffusers.models.attention_processor', AttnProcessor=AttnProcessor)
    _stub('diffusers.utils', deprecate=lambda *a, **k: None,
          logging=types.SimpleNamespace(get_logger=lambda name: __import__('logging').getLogger(name)))
    _stub('diffusers.utils.import_utils', is_xformers_available=lambda: False)
    _stub('diffusers.configuration_utils', FrozenDict=dict)
    _stub('diffusers.pipelines')
    _stub('diffusers.pipelines.stable_diffusion', StableDiffusionPipelineOutput=_Dummy)
    _stub('diffusers.pipelines.stable_diffusion.safety_checker', StableDiffusionSafetyChecker=_Dummy)
    _stub('diffusers.pipelines.t2i_adapter')
    _stub('diffusers.pipelines.t2i_adapter.pipeline_stable_diffusion_adapter',
          StableDiffusionAdapterPipeline=_Dummy, StableDiffusionAdapterPipelineOutput=_Dummy,
          _preprocess_adapter_image=lambda *a, **k: None)
    _stub('diffusers.schedulers', KarrasDiffusionSchedulers=_Dummy)
    _stub('diffusers.image_processor', VaeImageProcessor=_Dummy)
    _stub('accelerate')
    _stub('accelerate.logging', get_logger=lambda name, **k: __import__('logging').getLogger(name))
    _stub('accelerate.utils', set_seed=lambda *a, **k: None)
    _stub('accelerate.state', PartialState=_Dummy)
    _stub('IPython')
    _stub('IPython.display', display=lambda *a, **k: None)
    _stub('omegaconf', OmegaConf=_Dummy)
    if not hasattr(transformers, 'CLIPFeatureExtractor'):
        try:
            transformers.CLIPFeatureExtractor = transformers.CLIPImageProcessor
        except Exception:  # pragma: no cover
            transformers.CLIPFeatureExtractor = _Dummy


_loaded = {}


def load_reference_module(rel_path, name=None):
    """Execute a reference file in place (e.g. 'mixofshow/models/edlora.py') and return the module.

    This repo ships its own drop-in `mixofshow` package; while the reference file executes, any already imported
    `mixofshow*` modules are parked and /root/reference is put first on sys.path so that the reference's internal
    `from mixofshow... import ...` statements bind to the reference's files, then everything is restored."""
    if rel_path in _loaded:
        return _loaded[rel_path]
    install_stubs()
    parked = {k: sys.modules.pop(k) for k in list(sys.modules) if k == 'mixofshow' or k.startswith('mixofshow.')}
    # the reference's `mixofshow` is a namespace package (no __init__.py): a regular package of the same name anywhere
    # on sys.path would win, so hide those entries while the reference file executes
    saved_path = list(sys.path)
    sys.path[:] = [REFERENCE_ROOT] + [p for p in sys.path
                                      if not os.path.isfile(os.path.join(p or '.', 'mixofshow', '__init__.py'))]
    importlib.invalidate_caches()
    try:
        name = name or ('_ref_' + rel_path.replace('/', '_').replace('.py', ''))
        spec = importlib.util.spec_from_file_location(name, os.path.join(REFERENCE_ROOT, rel_path))
        mod = importlib.util.module_from_spec(spec)
        sys.modules[name] = mod
        spec.loader.exec_module(mod)
    finally:
        sys.path[:] = saved_path
        importlib.invalidate_caches()
        for k in [k for k in sys.modules if k == 'mixofshow' or k.startswith('mixofshow.')]:
            sys.modules['_ref_pkg_' + k] = sys.modules.pop(k)
        sys.modules.update(parked)
    _loaded[rel_path] = mod
    return mod
