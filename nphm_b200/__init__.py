"""nphm_b200 - B200-native engine for the hot path of NPHM (Neural Parametric Head Models).

The sub-packages mirror the reference's module layout (``NPHM.models.*``, ``NPHM.utils.*``) so that the
reference's ``scripts/fitting`` and ``scripts/training`` run unchanged on top of this engine after
:func:`install_as_nphm` (see INTEGRATION.md).
"""
import sys as _sys

__version__ = '0.1.0'


_MIRRORED = ('models.EnsembledDeepSDF', 'models.deepSDF', 'models.reconstruction', 'models.fitting',
             'models.iterative_root_finding', 'models.diff_operators', 'utils.reconstruction')


def _reference_package_dirs():
    """Directories of a real ``NPHM`` package on ``sys.path`` (the reference checkout's ``src/NPHM``), if any."""
    import os
    found = []
    for entry in _sys.path:
        cand = _os_path_join(entry or '.', 'NPHM')
        if os.path.isfile(_os_path_join(cand, '__init__.py')) and cand not in found:
            found.append(cand)
    return found


def _os_path_join(*a):
    import os
    return os.path.join(*a)


def set_native_training(enabled: bool = True) -> None:
    """Run first-order training through the native kernels: a ``DeepSDF`` / ``DeformationNetwork`` forward that autograd
    records (and that the layer chain supports) then runs on sm_100a, and its backward computes the weight gradients there.
    Default off, or on with the environment variable ``NPHM_NATIVE_TRAINING=1``.  Leave it off for losses that differentiate
    twice (stage-1 identity training): the native backward is first order and raises under ``create_graph=True``."""
    from . import _native
    _native.set_native_training(enabled)


def native_training() -> bool:
    """Whether :func:`set_native_training` is on."""
    from . import _native
    return _native.native_training()


def install_as_nphm(force: bool = False):
    """Register this package's mirrors under the reference's import names, so that
    ``from NPHM.models.deepSDF import DeepSDF`` (and the six other hot-path modules) resolve here, while every OTHER
    ``NPHM.*`` module - ``NPHM.env_paths``, ``NPHM.data.*``, ``NPHM.evaluation.*``, ``NPHM.models.training``,
    ``NPHM.models.loss_functions``, ``NPHM.utils.mesh_operations`` ... - keeps resolving to the reference checkout on
    ``sys.path``: the stand-in packages carry the reference's directories in their ``__path__`` and only the seven
    shadowed module names are pre-registered in ``sys.modules``.  Reference modules that import a shadowed name
    (``training.py`` -> ``NPHM.models.reconstruction``) therefore get the engine as well."""
    import importlib
    import os
    import types
    present = _sys.modules.get('NPHM')
    if present is not None and not force and not getattr(present, '_nphm_b200_alias', False):
        raise RuntimeError('a different NPHM package is already imported; pass force=True to shadow its hot-path modules')
    ref_dirs = _reference_package_dirs()
    if present is not None and not getattr(present, '_nphm_b200_alias', False):
        ref_dirs = [d for d in getattr(present, '__path__', []) if d not in ref_dirs] + ref_dirs
    root = types.ModuleType('NPHM')
    root._nphm_b200_alias = True
    root.__path__ = list(ref_dirs)
    root.__file__ = os.path.join(ref_dirs[0], '__init__.py') if ref_dirs else None
    # drop stale reference copies of the shadowed modules (and of the packages that hold them); keep everything else
    shadowed = {'NPHM', 'NPHM.models', 'NPHM.utils'} | {'NPHM.' + n for n in _MIRRORED}
    for key in list(_sys.modules):
        if key in shadowed:
            del _sys.modules[key]
    _sys.modules['NPHM'] = root
    for sub in ('models', 'utils'):
        pkg = types.ModuleType('NPHM.' + sub)
        pkg.__path__ = [os.path.join(d, sub) for d in ref_dirs if os.path.isdir(os.path.join(d, sub))]
        pkg._nphm_b200_alias = True
        _sys.modules['NPHM.' + sub] = pkg
        setattr(root, sub, pkg)
    for name in _MIRRORED:
        mod = importlib.import_module('nphm_b200.' + name)
        _sys.modules['NPHM.' + name] = mod
        sub, leaf = name.split('.')
        setattr(_sys.modules['NPHM.' + sub], leaf, mod)
    return root
