"""Drop-in boundary: the reference's own models/{classifier,segmenter,autoencoder}.py (unmodified,
as the bytecode build product oracle/_ref/pyref that build() compiles where the reference's sources
are available) run on top of sonet_b200's networks — construction on CPU, and full
set_input()/test_model() forwards on CUDA against the reference's own golden outputs. The
reference's files are not part of this repository: the CPU construction test skips where the
bytecode was not built; the CUDA test fails without it, since the built tree, oracle/_ref/
included, is what runs on the GPU machine. The module aliasing that install() does is checked
everywhere."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCRIPT = os.path.join(ROOT, "tests", "_dropin_run.py")


def _pyref_root():
    """oracle/_ref/pyref, or None when it was not built or was compiled by another interpreter."""
    sys.path.insert(0, ROOT)
    from oracle import build as obuild
    return obuild.pyref_root()


def _run(root, device):
    r = subprocess.run([sys.executable, SCRIPT, root, device], capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0 and "DROPIN_OK" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
    return r.stdout


def test_install_registers_our_modules_under_the_reference_names(tmp_path):
    """install() without a reference checkout: every hot-path module the reference's Model files
    import resolves to this package's module."""
    code = """
import sys
sys.path.insert(0, %r)
import sonet_b200.install as inst
from sonet_b200 import index_max, layers, losses, networks, operations, som
inst.install()
import index_max as a, util.som as b, models.operations as c, models.layers as d
import models.networks as e, models.losses as f
from models import networks as g
assert (a, b, c, d, e, f, g) == (index_max, som, operations, layers, networks, losses, networks)
print("INSTALL_OK")
""" % os.path.join(ROOT, "so-net_b200")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300,
                       cwd=str(tmp_path))
    assert r.returncode == 0 and "INSTALL_OK" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]


def test_reference_model_files_construct_on_our_networks():
    root = _pyref_root()
    if root is None:
        pytest.skip("oracle/_ref/pyref not built: the reference's sources were not available to build()")
    _run(root, "cpu")


@pytest.mark.gpu
def test_reference_model_files_forward_on_cuda():
    """models/classifier.py:64-105, models/segmenter.py:66-135, models/autoencoder.py:56-126 run
    unchanged on the CUDA path and reproduce the goldens the reference produced on CPU."""
    root = _pyref_root()
    if root is None:
        pytest.fail("oracle/_ref/pyref missing or compiled by another interpreter: run "
                    "__graft_entry__.build() where the reference's sources are available and ship "
                    "oracle/_ref/ with the tree")
    out = _run(root, "cuda:0")
    assert "classifier.Model ok" in out and "segmenter.Model ok" in out \
        and "autoencoder.Model ok" in out
