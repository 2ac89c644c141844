"""TEST INFRASTRUCTURE: run the reference's OWN function bodies in this container.

The reference cannot be imported unmodified here (scoop, Bio, h5py and
sklearn.externals.joblib are absent), but the hot-path function bodies are pure
stdlib + numpy.  This module parses the reference source files where they lie
under /root/reference, picks the named ``FunctionDef`` nodes and ``exec``s only
those into a namespace that provides ``re, np, Counter, product, sys``.  Nothing
is copied into the repository; this is used only by ``tests/golden/make_golden.py``
to generate the committed golden vectors, which the tests compare against.
"""
from __future__ import annotations

import ast
import os
import re
import sys
from collections import Counter
from itertools import product

import numpy as np

REFERENCE_ROOT = os.environ.get("PHYLOLIGO_REFERENCE", "/root/reference")
_BIN = os.path.join(REFERENCE_ROOT, "phylopackage", "bin", "phyloligo.py")
_CORE = os.path.join(REFERENCE_ROOT, "phylopackage", "core", "phylodist.py")


def available() -> bool:
    return os.path.isfile(_BIN) and os.path.isfile(_CORE)


def _extract(path, names, namespace):
    with open(path, "r") as fh:
        tree = ast.parse(fh.read(), filename=path)
    wanted = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name in names]
    missing = set(names) - {n.name for n in wanted}
    if missing:
        raise RuntimeError("reference functions not found: %s" % sorted(missing))
    module = ast.Module(body=wanted, type_ignores=[])
    exec(compile(module, path, "exec"), namespace)
    return namespace


def load():
    """Return a dict of reference callables:
    cut_sequence_and_count_pattern, count2freq  (bin/phyloligo.py:601-661)
    posdef_check_value, KL, Eucl, JSD            (core/phylodist.py:12-68)
    """
    if not available():
        raise RuntimeError("reference checkout not mounted at %s" % REFERENCE_ROOT)
    np.seterr(divide="ignore", invalid="ignore")  # core/phylodist.py:9
    ns = {"re": re, "np": np, "Counter": Counter, "product": product, "sys": sys}
    _extract(_BIN, ["cut_sequence_and_count_pattern", "count2freq"], ns)
    _extract(_CORE, ["posdef_check_value", "KL", "Eucl", "JSD"], ns)
    return ns
