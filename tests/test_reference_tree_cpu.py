"""The INTEGRATION.md modules resolve through the reference's OWN registries inside a scratch copy of the unmodified
reference package (baseline/_ref/RL; the repository does not ship it, so that test skips without it).  CPU only: class
resolution and the reference's error behaviour; construction needs a GPU (tests/test_gpu_trainer.py runs the reference
trainer loop there).  The TensorBoard tag table is compared with the reference's as recorded under tests/golden/."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))


def test_b200_modules_resolve_through_the_reference_registries():
    import reference_dropin as rd
    if rd.reference_package() is None:
        pytest.skip("no reference package on this host (baseline/_ref/RL is installed by __graft_entry__.build())")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "reference_dropin.py"), "registries"], capture_output=True,
                         text=True, timeout=300)
    assert res.returncode == 0, res.stderr[-2000:]
    out = json.loads(res.stdout.strip().splitlines()[-1])
    for k in ("sampler", "buffer", "buffer_indexed", "algorithm", "approx_container", "trainer", "reference_ids_still_registered",
              "unknown_id_raises"):
        assert out[k] is True, (k, out)


def test_trainer_tags_match_reference_table():
    """The TensorBoard tag table is a naming contract with the reference's CSV / plotting tools
    (RL/utils/tensorboard_setup.py:13-40, recorded in tests/golden/reference_tb_tags.json by make_golden.py):
    identical keys and values."""
    import numpy as np
    golden = os.path.join(ROOT, "tests", "golden")
    with open(os.path.join(golden, "reference_tb_tags.json")) as fh:
        ref = json.load(fh)
    import msacl_b200  # noqa: F401
    from msacl_b200.trainer import tb_tags
    assert ref == tb_tags
    # the loss tags the reference's own model_update returned in the recorded run are entries of the table
    recorded = {str(k) for k in np.load(os.path.join(golden, "msacl_update_TwoLink.npz"))["tb_keys"]}
    assert {ref[k] for k in ("loss_critic", "loss_lyapunov", "loss_actor")} <= recorded
