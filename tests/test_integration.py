"""Boundary proof through the REFERENCE's own callers (SURVEY.md 8b / 8f-3): INTEGRATION.md's snippet run verbatim, and a
Training Directory round trip through the reference's `generate.load_minimagen` after `install_as_minimagen()`.
Needs a checkout of the original MinImagen project (oracle/reference.py, $MINIMAGEN_REFERENCE) -- its own generate.py and
training.py are what is exercised, so no stored fixture can stand in for it and it skips without one; runs in a subprocess
because it re-binds sys.modules['minimagen*']."""
import json
import os
import subprocess
import sys

import pytest

from oracle import reference

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(mode):
    env = dict(os.environ)
    shims = os.path.join(ROOT, "oracle", "shims")
    env["PYTHONPATH"] = os.pathsep.join([ROOT, os.path.join(ROOT, "tests"), reference.REFERENCE_ROOT, shims,
                                         env.get("PYTHONPATH", "")])
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "_integration_script.py"), mode], env=env,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


@pytest.mark.skipif(not reference.available(), reason="reference checkout not present")
def test_reference_generate_loads_b200_classes_from_training_directory():
    res = _run("emu")
    assert res["generate_file"].startswith(reference.REFERENCE_ROOT)          # the reference's own generate.py ran
    assert res["generate_uses_b200_classes"] and res["training_uses_b200_unet"]
    assert res["loaded_type"] == "minimagen_b200.Imagen.Imagen"
    assert res["unet_types"] == ["minimagen_b200.Unet"]
    assert res["weights_equal"] and res["sample_equal"] and res["sample_finite"]
    assert res["sample_shape"] == [2, 3, 32, 32]
    # the reference's training loop (training.MinimagenTrain) trained the B200 classes and wrote loadable checkpoints
    assert res["train_weights_changed"] and res["trained_loaded_type"] == "minimagen_b200.Imagen"
    assert res["train_files"] == ["unet_0_state_20260101_000000.pth", "unet_1_state_20260101_000000.pth"]


def test_install_as_minimagen_without_reference_is_alias_only():
    """No reference on the path: `minimagen` becomes an alias package of the hot-path modules only."""
    code = ("import sys; sys.path = [p for p in sys.path if 'reference' not in p]\n"
            "import minimagen_b200 as m; pkg = m.install_as_minimagen()\n"
            "from minimagen.Unet import Unet; from minimagen.Imagen import Imagen; from minimagen import Unet as U\n"
            "import minimagen_b200.Unet as MU\n"
            "assert Unet is MU.Unet and U is MU\n"
            "try:\n    import minimagen.generate\n    raise SystemExit('unexpected: minimagen.generate importable')\n"
            "except ModuleNotFoundError:\n    pass\nprint('ok')\n")
    env = dict(os.environ, PYTHONPATH=ROOT, MINIMAGEN_REFERENCE="/nonexistent")
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=300, cwd="/tmp")
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), r.stderr[-2000:]
