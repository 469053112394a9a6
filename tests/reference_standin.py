"""A stand-in for the upstream kernel-matrix-benchmarks package, for the harness tests that do not need its runner.

It has the layout ``bootstrap.find_reference`` looks for and the two names of ``kernel_matrix_benchmarks.datasets`` that
this repository's harness layer uses:

* ``DATASETS``, holding one of the upstream's own dataset names (its writer must survive ``datasets_ext.register``);
* ``GroundTruth``, the upstream's float64 brute force (datasets.py:81-83), restated by ``oracle.bruteforce_oracle``, which
  tests/test_oracle.py holds to the upstream's own outputs stored in tests/golden/ (rel-L2 <= 1e-12).

Its ``download`` fails the test that reaches it: the offline harness must replace it.
"""
import sys

import pytest

from kernel_matrix_benchmarks_b200.harness import bootstrap

UPSTREAM_DATASET = "product-sphere-D3-E1-M1000-N1000-inverse-distance"

DATASETS_PY = f'''
from oracle import bruteforce_oracle as _orc


def _upstream_writer(filename):
    raise AssertionError("the stand-in's own dataset writer was called")


DATASETS = {{{UPSTREAM_DATASET!r}: _upstream_writer}}


def download(src, dst):
    raise AssertionError("stand-in download reached: " + src)


class GroundTruth:
    def __init__(self, kernel, dimension, normalize_rows=False):
        self.kernel, self.normalize_rows = kernel, normalize_rows

    def prepare_data(self, source_points, target_points=None):
        self.y, self.x = source_points, target_points

    def fit(self):
        pass

    def prepare_query(self, source_signal):
        self.b = source_signal

    def query(self):
        self.res = _orc.kernel_product(self.kernel, self.y, self.x, self.b, normalize_rows=self.normalize_rows)

    def get_result(self):
        return self.res
'''


def _loaded():
    return [m for m in sys.modules if m == "kernel_matrix_benchmarks" or m.startswith("kernel_matrix_benchmarks.")]


@pytest.fixture
def standin_reference(tmp_path, monkeypatch):
    """Activate the stand-in (with the extra datasets registered); everything imported from it is dropped afterwards."""
    pkg = tmp_path / "standin" / "kernel_matrix_benchmarks"
    pkg.mkdir(parents=True)
    (pkg / "__init__.py").write_text("")
    (pkg / "runner.py").write_text("")
    (pkg / "datasets.py").write_text(DATASETS_PY)
    monkeypatch.setattr(sys, "path", list(sys.path))
    for name in _loaded():   # an upstream tree imported by an earlier test comes back after this one
        monkeypatch.delitem(sys.modules, name)
    try:
        yield bootstrap.activate(str(tmp_path / "standin"))[0]
    finally:
        for name in _loaded():
            del sys.modules[name]
