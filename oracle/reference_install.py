#!/usr/bin/env python
"""Offline install of the unmodified reference (tenpy/tenpy) into ``oracle/_ref/``, for the tests and the benchmark arms
that run the reference's own code: its drivers on this engine (``tenpy_b200.dropin``), its engine on the host
(``bench.py --impl reference``, the ``cpu_baseline`` of the GPU arm) and the checkpoint exchange of
``tenpy_b200.tools.interop``.

The recipe copies the ``tenpy`` package of a reference checkout and compiles its Cython helper
``tenpy/linalg/_npc_helper.pyx`` the way the reference's setup.py does (C++, numpy headers, no MKL).  The checkout is taken
from ``$TENPY_REFERENCE`` or the default location below; without one the recipe leaves an existing install alone, so
that a tree built where the checkout exists keeps its install wherever it is copied to.  ``oracle/_ref/`` is a build
product and stays out of git.  ``build()`` runs this file; by hand:

    python oracle/reference_install.py
"""
import os
import shutil
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
TARGET = os.path.join(HERE, '_ref')
DEFAULT_CHECKOUT = '/root/reference'      # read-only checkout of tenpy/tenpy where the project is built
STAMP = 'INSTALLED_FROM'


def checkout():
    for c in (os.environ.get('TENPY_REFERENCE'), DEFAULT_CHECKOUT):
        if c and os.path.isdir(os.path.join(c, 'tenpy')) and os.path.realpath(c) != os.path.realpath(TARGET):
            return c
    return None


def _newest_mtime(root):
    t = 0.
    for d, dirs, files in os.walk(root):
        dirs[:] = [x for x in dirs if x != '__pycache__']
        for f in files:
            t = max(t, os.path.getmtime(os.path.join(d, f)))
    return t


def _up_to_date(src):
    stamp = os.path.join(TARGET, STAMP)
    if not os.path.exists(stamp):
        return False
    with open(stamp) as f:
        if f.read().strip() != os.path.realpath(src):
            return False
    return os.path.getmtime(stamp) >= _newest_mtime(os.path.join(src, 'tenpy'))


def _compile_helper(stage):
    """tenpy/linalg/_npc_helper.pyx -> extension module next to it (setup.py of the reference: language c++, numpy
    headers, compile-time HAVE_MKL = 0)"""
    import numpy
    from Cython.Build import cythonize
    from setuptools import Distribution, Extension
    pyx = os.path.join(stage, 'tenpy', 'linalg', '_npc_helper.pyx')
    ext = Extension('tenpy.linalg._npc_helper', [pyx], include_dirs=[numpy.get_include()], language='c++')
    mods = cythonize([ext], compiler_directives={'language_level': 3, 'embedsignature': True},
                     compile_time_env={'HAVE_MKL': 0, 'MKL_INTERFACE_LAYER': 0}, quiet=True)
    with tempfile.TemporaryDirectory() as tmp:
        cmd = Distribution({'ext_modules': mods}).get_command_obj('build_ext')
        cmd.build_lib, cmd.build_temp = stage, tmp
        cmd.ensure_finalized()
        cmd.run()


def install():
    """Install (or refresh) ``oracle/_ref``; returns its path, or None if there is neither a checkout nor an install."""
    src = checkout()
    if src is None:
        return TARGET if os.path.exists(os.path.join(TARGET, STAMP)) else None
    if _up_to_date(src):
        return TARGET
    stage = TARGET + '.partial'
    shutil.rmtree(stage, ignore_errors=True)
    shutil.copytree(os.path.join(src, 'tenpy'), os.path.join(stage, 'tenpy'), copy_function=shutil.copyfile,
                    ignore=shutil.ignore_patterns('__pycache__', '*.so', '*.c', '*.cpp'))
    for d, _, files in os.walk(stage):            # the checkout may be read-only; the install is not
        os.chmod(d, 0o755)
        for f in files:
            os.chmod(os.path.join(d, f), 0o644)
    _compile_helper(stage)
    with open(os.path.join(stage, STAMP), 'w') as f:
        f.write(os.path.realpath(src) + '\n')
    shutil.rmtree(TARGET, ignore_errors=True)
    os.rename(stage, TARGET)
    return TARGET


if __name__ == '__main__':
    path = install()
    print('[reference] %s' % (path or 'no reference checkout found; oracle/_ref not installed'))
    sys.exit(0)
