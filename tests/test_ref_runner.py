"""CPU: the CPU arm of bench.py really is the reference.  oracle/ref_runner.py (the reference's own SceneRF class from the
sources staged in oracle/_ref by oracle/build_ref.py, or a reference checkout) must reproduce a committed golden -- which
tests/golden/make_goldens.py produced from the unmodified reference -- BIT FOR BIT, and the staged copies must hash to the
digests of the unmodified reference files (tests/golden/reference_sources.npz).  Both tests need the reference's sources,
which this repository does not contain, and skip where they have not been staged."""
import hashlib
import os

import numpy as np
import pytest

from cases import RENDER_CASES, load_golden, pyramid_for
from oracle import build_ref, ref_runner


@pytest.mark.skipif(not ref_runner.available(), reason="neither oracle/_ref nor /root/reference is present")
@pytest.mark.parametrize("name", ["kitti_mini", "bf_mini"])
def test_reference_class_reproduces_golden_bit_for_bit(name):
    import torch
    cfg, seed = RENDER_CASES[name]
    g = load_golden(name)
    model = ref_runner.build_model(cfg)
    x_rgb = {k: torch.from_numpy(v) for k, v in pyramid_for(cfg, seed).items()}
    torch.manual_seed(0)                                   # make_goldens.run_render_case seeds the two RNG draws with 0
    out = ref_runner.render(model, cfg, x_rgb, torch.from_numpy(g["pixels"]), g["pixels"].shape[0])
    assert set(out) == {"depth", "color", "gaussian_means", "gaussian_stds", "weights_at_depth", "closest_pts_to_depths",
                        "loss_kl", "alphas", "som_vars", "densities", "weights", "depth_volumes"}
    for k in ("depth", "color", "gaussian_means", "gaussian_stds", "alphas", "densities", "weights", "depth_volumes", "loss_kl"):
        assert np.array_equal(out[k].numpy(), g[k]), k


@pytest.mark.skipif(not os.path.exists(os.path.join(build_ref.OUT, "MANIFEST.json")),
                    reason="reference sources not staged in oracle/_ref")
def test_staged_sources_are_the_unmodified_reference():
    g = load_golden("reference_sources")                   # sha256 of the unmodified reference files
    digests = dict(zip(g["files"].tolist(), g["sha256"].tolist()))
    assert sorted(digests) == sorted(build_ref.FILES)
    for rel, digest in digests.items():
        with open(os.path.join(build_ref.OUT, rel), "rb") as f:
            assert hashlib.sha256(f.read()).hexdigest() == digest, rel
