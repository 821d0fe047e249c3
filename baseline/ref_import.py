"""Import the unmodified reference (zgcr/SimpleAICV_pytorch_training_examples).

The reference lives in ``oracle/_ref`` (git-ignored), copied there by ``oracle/install_ref.sh``.
Only the golden-data generators under ``tests/golden`` and the torch baselines import it; the tests,
``smoke()`` and ``bench.py`` compare with the stored golden data instead.  ``tools.utils`` /
``tools.scripts`` import ``calflops`` and ``pycocotools`` at module level (tools/utils.py:19,
tools/scripts.py:14-15), which are not installed here; the hot path never
calls them, so empty stub modules are registered for those two names only.

TEST / BENCH INFRASTRUCTURE: the product package never imports this module.
"""
import importlib
import os
import sys
import types

_HERE = os.path.dirname(os.path.abspath(__file__))
CANDIDATES = [os.path.join(os.path.dirname(_HERE), 'oracle', '_ref')]


def root():
    for c in CANDIDATES:
        if os.path.isdir(os.path.join(c, 'SimpleAICV')):
            return c
    return None


def available():
    return root() is not None


def _ensure_path():
    r = root()
    if r is None:
        raise ImportError('reference not installed: run oracle/install_ref.sh <reference checkout>')
    if r not in sys.path:
        sys.path.insert(0, r)
    for name in ('calflops', 'pycocotools', 'pycocotools.coco', 'pycocotools.cocoeval', 'pycocotools.mask'):
        if name not in sys.modules:
            try:
                importlib.import_module(name)
            except Exception:
                m = types.ModuleType(name)
                m.calculate_flops = lambda *a, **k: (0, 0, 0)
                m.COCO = m.COCOeval = object
                sys.modules[name] = m
    return r


def module(name):
    _ensure_path()
    return importlib.import_module(name)


def backbones():
    return module('SimpleAICV.classification.backbones')
