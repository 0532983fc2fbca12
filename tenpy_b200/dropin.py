"""Run the reference's own drivers on the device-resident engine (SURVEY.md section 8b, boundary B1).

The algorithms of tenpy/tenpy reach the tensor engine only through ``from ..linalg import np_conserved as npc``
(tenpy/algorithms/dmrg.py:42, mps_common.py, tebd.py, networks/mps.py, mpo.py, site.py, models/*).  :func:`install` makes
that import resolve to :mod:`tenpy_b200.linalg.np_conserved` / :mod:`tenpy_b200.linalg.charges`, so that the UNMODIFIED
reference files -- ``tenpy.algorithms.dmrg``, ``tebd``, ``mps_common``, ``truncation``, ``krylov_based``, the MPS / MPO /
Site / model classes -- run with every Array in packed HBM and every contraction, SVD, eigh, block move on the CUDA
kernels of ``libb200npc.so``::

    from tenpy_b200 import dropin
    dropin.install()                       # BEFORE the first ``import tenpy``
    import tenpy
    from tenpy.algorithms import dmrg      # the reference's file, now on the B200 engine
    M = tenpy.models.tf_ising.TFIChain({...}); psi = tenpy.networks.mps.MPS.from_product_state(...)
    dmrg.run(psi, M, {...})

How: ``sys.modules['tenpy.linalg.np_conserved']`` and ``['tenpy.linalg.charges']`` are seeded with the engine's modules
(an ``import`` statement consults ``sys.modules`` first, so ``tenpy/linalg/__init__.py:27`` picks them up), and a one-shot
import hook marks ``tenpy.tools.optimization.have_cython_functions = False`` right after that module is executed: the
reference asserts at ``tenpy/linalg/__init__.py:74`` that its ``@use_cython`` decorator ran, which it does not when its own
``np_conserved.py`` is never executed.  Nothing of the reference is modified or copied.

The speed-relevant extension of the engine -- the split-order / identity-environment effective-H matvec -- plugs into the
reference engine through the reference's own hook, the class attribute ``EffectiveH`` (tenpy/algorithms/mps_common.py:
``Sweep.EffectiveH``): :func:`fast_two_site_engine` returns a subclass of the reference's ``TwoSiteDMRGEngine`` whose
``EffectiveH`` is the reference's ``TwoSiteH`` with ``matvec`` replaced by the device-optimised contraction order.
"""
import importlib
import importlib.abc
import importlib.util
import os
import sys

__all__ = ['install', 'installed', 'reference_path', 'fast_two_site_engine']

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def reference_path():
    """where the unmodified reference lives: ``$TENPY_REFERENCE``, or the install ``oracle/_ref`` that ``build()`` makes
    from a reference checkout (oracle/reference_install.py)"""
    cands = [os.environ.get('TENPY_REFERENCE'), os.path.join(_ROOT, 'oracle', '_ref')]
    for c in cands:
        if c and os.path.isdir(os.path.join(c, 'tenpy')):
            return c
    return None


class _MarkNoCython(importlib.abc.MetaPathFinder):
    """one-shot post-import hook on ``tenpy.tools.optimization`` (see the module doc string)"""

    name = 'tenpy.tools.optimization'

    def find_spec(self, fullname, path, target=None):
        if fullname != self.name:
            return None
        sys.meta_path.remove(self)
        spec = importlib.util.find_spec(fullname)
        if spec is None:
            return None
        inner = spec.loader

        class _Loader(importlib.abc.Loader):
            def create_module(self, sp):
                return inner.create_module(sp)

            def exec_module(self, module):
                inner.exec_module(module)
                module.have_cython_functions = False      # the engine's modules carry no @use_cython hooks

        spec.loader = _Loader()
        return spec


def installed():
    npc = sys.modules.get('tenpy.linalg.np_conserved')
    return npc is not None and getattr(npc, '__name__', '') == 'tenpy_b200.linalg.np_conserved'


def install(path=None):
    """Seed the engine's modules under the reference's names; must run before the first ``import tenpy``.  `path`: the
    reference checkout / install to put on ``sys.path`` (default :func:`reference_path`).  Returns the path used."""
    if installed():
        return path or reference_path()
    if 'tenpy' in sys.modules:
        raise RuntimeError('tenpy_b200.dropin.install() has to run before the first `import tenpy`')
    from .linalg import np_conserved, charges
    sys.modules['tenpy.linalg.np_conserved'] = np_conserved
    sys.modules['tenpy.linalg.charges'] = charges
    sys.meta_path.insert(0, _MarkNoCython())
    path = path or reference_path()
    if path is not None and path not in sys.path:
        sys.path.insert(0, path)
    return path


def fast_two_site_engine():
    """The reference's ``TwoSiteDMRGEngine`` with the device-optimised effective Hamiltonian plugged in at the reference's
    own extension point ``EffectiveH``.  Call after :func:`install`."""
    if not installed():
        raise RuntimeError('call tenpy_b200.dropin.install() first')
    from tenpy.algorithms import dmrg as ref_dmrg
    from tenpy.algorithms import mps_common as ref_common
    from .algorithms.mps_common import TwoSiteH as _EngineH

    class B200TwoSiteH(ref_common.TwoSiteH):
        """reference ``TwoSiteH`` (same constructor, attributes, `combine_theta`, `update_LP` ...); `matvec` applies
        ``LP``, ``W0 W1``, ``RP`` to the split theta without the identity components of the environments where that is
        cheaper (tenpy_b200.algorithms.mps_common.TwoSiteH._matvec_split), the reference order otherwise."""

        def __init__(self, env, i0, combine=False, move_right=True):
            super().__init__(env, i0, combine, move_right)
            self._H_mpo = env.H
            self._W01 = None
            self._LHeff = getattr(self, 'LHeff', None)
            self._RHeff = getattr(self, 'RHeff', None)

        matvec_order = 'auto'

        def matvec(self, theta):
            if self.combine and self._use_split(theta):
                return self._matvec_split(theta, theta.get_leg_labels())
            return super().matvec(theta)

    # the device-optimised contraction routes of the engine's own TwoSiteH (everything but the constructor and the
    # environment updates, which stay the reference's): methods and their class-level switches, by name prefix
    take = ('_matvec_split', '_identity_env', '_dense_recipe', '_apply_W01', '_split_t2_views', '_use_split', 'deferred_check',
            'identity_check', 'identity_env', 'mpo_apply', 'SPLIT_MIN_BLOCK', 'stats')
    for name, val in vars(_EngineH).items():
        if name.startswith(take) and name not in vars(B200TwoSiteH):
            setattr(B200TwoSiteH, name, val)

    class B200TwoSiteDMRGEngine(ref_dmrg.TwoSiteDMRGEngine):
        EffectiveH = B200TwoSiteH

    return B200TwoSiteDMRGEngine
