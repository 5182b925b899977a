"""The GPU parity harness (tests/parity.py SideBySide) exercised WITHOUT a GPU: a CPU stand-in for the CUDA executor -- a second oracle
instance with its own textures behind the executor's upload / download / execute_raw interface -- takes the place of
nrd.CudaContext.  Checks the harness logic the GPU tests rely on (state synchronisation before every pass, output comparison, the
reference-shader mode of tests/test_zz_gpu_reference_shaders.py) on every CPU run."""
import pytest

import oracle_runner as orr
import parity
from raytracingdenoiser_b200 import nrd


class OracleAsExecutor(object):
    def __init__(self, sbs, variant=""):
        self.den = orr.CpuDenoiser(sbs.denoiser, sbs.w, sbs.h, identifier=sbs.identifier, instance=sbs.instance, variant=variant, common=sbs.common)
        self.instance = sbs.instance

    def upload(self, rtype, index, arr):
        self.den.resolve(rtype, index)[0][...] = arr

    def download(self, rtype, index, out):
        out[...] = self.den.resolve(rtype, index)[0]

    def execute_raw(self, ref):
        pipelines = self.instance.get_instance_desc()["pipelines"]
        self.den.run_dispatch(nrd.Dispatch(ref._obj, pipelines))


def test_harness_reports_identity_when_both_sides_are_the_oracle():
    sbs = parity.SideBySide(nrd.Denoiser.REBLUR_DIFFUSE_SPECULAR, 96, 64, executor=OracleAsExecutor)
    report = sbs.run_per_pass(3)
    assert len(report) > 30 and not sbs.failures()
    assert all(r["fraction"] == 1.0 and r["worst"] == 0.0 for r in report)


def test_harness_detects_a_different_evaluation():
    """The FMA-contracted build of the oracle as "the GPU": close, not identical -- the harness must see rounding differences."""
    sbs = parity.SideBySide(nrd.Denoiser.RELAX_DIFFUSE_SPECULAR, 96, 64, executor=lambda s: OracleAsExecutor(s, "fma"))
    report = sbs.run_per_pass(3)
    assert any(r["worst"] > 0.0 for r in report) and min(r["fraction"] for r in report) > 0.98


@pytest.mark.parametrize("denoiser_name,gate", [("REBLUR_DIFFUSE_SPECULAR", 0.995), ("SIGMA_SHADOW", 0.995), ("RELAX_DIFFUSE_SPECULAR", 0.98)])
def test_reference_shader_mode_of_the_harness(denoiser_name, gate):
    """tests/test_zz_gpu_reference_shaders.py with the oracle in the role of the kernels: same call, same gates."""
    sbs = parity.SideBySide(getattr(nrd.Denoiser, denoiser_name), 320, 180, reference_shaders=True, executor=OracleAsExecutor)
    report = sbs.run_per_pass(4)
    compared = [r for r in report if not r["shader"].startswith("Clear_")]
    assert compared and all(r["nonfinite"] == 0 for r in compared)
    worst = min(compared, key=lambda r: r["fraction"])
    assert worst["fraction"] >= gate, (worst["shader"], worst["resource"], worst["fraction"])
    assert any(r["fraction"] < 1.0 or r["worst"] > 0.0 for r in compared) or denoiser_name == "SIGMA_SHADOW"  # the shaders, not the oracle, ran on the CPU side
