"""The CUDA kernels against the REFERENCE's own shader code, directly: per-pass parity like tests/test_gpu_*.py, but the CPU side of
every pass is the reference's shader source compiled for the CPU (oracle/build_refshaders.py -> oracle/_ref/shaders/*.so; its outputs
are replayed from tests/golden/reference_shader_outputs.npz.xz, see tests/oracle_runner.py) instead of the oracle's restatement of it.

The strict gates of the suite are against the oracle; tests/test_reference_shaders.py ties the oracle to these shaders on the CPU
(bit-identical but for the named deviations).  This file closes the triangle on the GPU with its own, wider gates: what separates
a kernel from the reference shader is (kernel vs oracle: rounding, <= 1e-3 of texels) + (oracle vs shader: tap positions evaluated
in texel instead of uv units, ~1e-4 of texels; RELAX: one association in the world-position helpers, amplified by temporal
accumulation to ~3e-3 of texels).  Named zz so that it runs last: it was written after the round's GPU budget was spent."""
import json
import os

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("denoiser_name,gate", [("REBLUR_DIFFUSE_SPECULAR", 0.995), ("SIGMA_SHADOW", 0.995), ("RELAX_DIFFUSE_SPECULAR", 0.98)])
def test_kernels_against_the_reference_shaders(denoiser_name, gate):
    import parity
    from raytracingdenoiser_b200 import nrd
    sbs = parity.SideBySide(getattr(nrd.Denoiser, denoiser_name), 320, 180, reference_shaders=True)
    report = sbs.run_per_pass(4)
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    with open(os.path.join(ROOT, "gpurun_out", "parity_vs_reference_shaders_%s.json" % denoiser_name), "w") as f:
        json.dump(report, f, indent=1, default=str)
    compared = [r for r in report if not r["shader"].startswith("Clear_")]
    assert compared
    worst = min(compared, key=lambda r: r["fraction"])
    print("%s: %d outputs compared with the reference shaders, worst %s %s fraction %.5f" % (denoiser_name, len(compared), worst["shader"], worst["resource"], worst["fraction"]))
    assert all(r["nonfinite"] == 0 for r in compared)
    assert worst["fraction"] >= gate, (worst["shader"], worst["resource"], worst["fraction"])
