"""include/nrd_b200_frontend.cuh (CUDA / C++ restatement of the reference's HLSL front-end / back-end helpers, NRD.hlsli:594-1161)
against the packers the test scene has always used (raytracingdenoiser_b200/scene.py) and independent numpy restatements."""
import os
import subprocess
import tempfile

import numpy as np
import torch

from raytracingdenoiser_b200 import scene

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run_probe():
    with tempfile.TemporaryDirectory() as tmp:
        exe = os.path.join(tmp, "probe")
        subprocess.run(["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"), "-I", "/usr/local/cuda/include", os.path.join(ROOT, "tests", "frontend_probe.cpp"),
                        "-o", exe], check=True)
        out = subprocess.run([exe], check=True, capture_output=True, text=True).stdout
    return np.array([[float(v) for v in line.split()] for line in out.strip().split("\n")], dtype=np.float64)


def test_frontend_header_matches_scene_packers_and_round_trips():
    d = _run_probe()
    assert d.shape == (400, 50)
    n, rough, mat, bits = d[:, 0:3], d[:, 3], d[:, 4], d[:, 5].astype(np.int64)
    # 1. IN_NORMAL_ROUGHNESS: same bits as scene.pack_normal_roughness (octahedral + R10G10B10A2 quantisation)
    ref = scene.pack_normal_roughness(torch.tensor(n, dtype=torch.float32), torch.tensor(rough, dtype=torch.float32), torch.tensor(mat, dtype=torch.float32)).numpy().astype(np.int64) & 0xFFFFFFFF
    diff = np.zeros(len(bits), dtype=np.int64)
    for shift, mask in ((0, 1023), (10, 1023), (20, 1023), (30, 3)):
        diff = np.maximum(diff, np.abs(((bits >> shift) & mask) - ((ref >> shift) & mask)))
    assert (diff == 0).mean() > 0.98 and diff.max() <= 1          # a code exactly on a rounding boundary may flip (fp32 vs torch op order)
    # 2. unpack: unit normal within the 10-bit octahedral error, roughness within 1/1023, material exact
    un = d[:, 6:9]
    assert np.allclose(np.linalg.norm(un, axis=1), 1.0, atol=1e-5)
    assert (np.sum(un * n, axis=1) > 1.0 - 2e-5).all()
    assert np.abs(d[:, 9] - rough).max() <= 0.5 / 1023 + 1e-6 and np.array_equal(np.rint(d[:, 10]), mat)
    # 3. REBLUR radiance: YCoCg + normalised hit distance = scene.pack_reblur (before the fp16 store)
    rad, hit, viewz, nh = d[:, 11:14], d[:, 14], d[:, 15], d[:, 16]
    t = lambda a: torch.tensor(a, dtype=torch.float32)
    ref = scene.pack_reblur(t(rad), t(hit), t(viewz), t(rough), torch.zeros(len(hit), dtype=torch.bool)).float().numpy()
    assert np.allclose(d[:, 17:21], ref, rtol=1.5e-3, atol=1e-4)
    a, b, c, dd = scene.HIT_DIST_PARAMS
    norm = (a + np.abs(viewz) * b) * (1.0 + (c - 1.0) * np.clip(np.exp2(dd * rough * rough), 0, 1))
    assert np.allclose(nh, np.clip(hit / norm, 0, 1), rtol=1e-5, atol=1e-6)
    assert np.allclose(d[:, 49], nh * norm, rtol=1e-5)                                     # REBLUR_GetHitDist inverts it
    assert np.allclose(d[:, 21:24], rad, rtol=1e-5, atol=1e-5)                             # YCoCg round trip
    # 4. RELAX: linear radiance + world-space hit distance
    assert np.allclose(d[:, 24:28], np.concatenate([rad, hit[:, None]], axis=1), rtol=1e-6)
    # 5. SIGMA penumbra: 0 where NoL <= 0, NRD_FP16_MAX on a miss, distance * tan(radius) / 2 otherwise; local light variant
    docc, pen, pen2 = d[:, 28], d[:, 29], d[:, 30]
    exp = np.where(docc >= 65504.0, 65504.0, np.minimum(docc * 0.004625 * 0.5, 32768.0))
    assert np.allclose(pen, exp, rtol=1e-5)
    assert np.allclose(pen2, np.where(docc >= 65504.0, 65504.0, np.minimum(2.0 * docc / np.maximum(100.0 - docc, 1e-6) * 0.5, 32768.0)), rtol=1e-5)
    assert np.array_equal(d[:, 45], (docc >= 65504.0).astype(np.float64)) and d[:, 46].max() <= 1.0
    # 6. SH / SG carrier: colour and direction survive pack -> unpack; SH diffuse resolve along the light direction = 1.5 x luma-scaled colour
    dirn = d[:, 31:34]
    assert np.allclose(d[:, 37:40], rad, rtol=1e-4, atol=1e-5) and np.allclose(d[:, 40:43], dirn, atol=1e-4)
    y = rad @ np.array([0.25, 0.5, 0.25])
    assert np.allclose(d[:, 47], dirn[:, 0] * y, rtol=1e-5, atol=1e-6) and (d[:, 48] == 0).all()
    assert np.allclose(d[:, 34:37], rad * 1.5, rtol=2e-4, atol=1e-4)
    # 7. material factors stay in [0.02, 1]
    assert d[:, 43].min() >= 0.02 - 1e-6 and d[:, 43].max() <= 1.0 + 1e-6 and d[:, 44].min() >= 0.02 - 1e-6 and d[:, 44].max() <= 1.0 + 1e-6


def test_frontend_header_compiles_as_cuda_device_code():
    """nvcc -c of a kernel that calls the helpers on the device (cross-compiles here, no GPU needed)."""
    src = '#include "nrd_b200_frontend.cuh"\n' \
          "__global__ void k(float4* o, const float3* n, const float* r) { int i = threadIdx.x; float4 p = nrd_frontend::NRD_FrontEnd_PackNormalAndRoughness(n[i], r[i], 1.0f);\n" \
          "  float4 q = nrd_frontend::REBLUR_FrontEnd_PackRadianceAndNormHitDist(n[i], nrd_frontend::REBLUR_FrontEnd_GetNormHitDist(r[i], 3.0f, make_float4(3, 0.1f, 20, -25), r[i]));\n" \
          "  nrd_frontend::NRD_SG sg = nrd_frontend::SG_Create(n[i], n[i], r[i]); float3 c = nrd_frontend::NRD_SG_ResolveSpecular(sg, n[i], n[i], r[i]);\n" \
          "  o[i] = make_float4(p.x + q.x + c.x, p.y + q.w, (float)nrd_frontend::nrdPackR10G10B10A2(p), nrd_frontend::SIGMA_FrontEnd_PackPenumbra(r[i], 0.01f)); }\n"
    with tempfile.TemporaryDirectory() as tmp:
        cu = os.path.join(tmp, "t.cu")
        open(cu, "w").write(src)
        r = subprocess.run(["/usr/local/cuda/bin/nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-I", os.path.join(ROOT, "include"), "-c", cu, "-o",
                            os.path.join(tmp, "t.o")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_frontend_header_equals_the_reference_nrd_hlsli():
    """The same probe compiled twice: against include/nrd_b200_frontend.cuh, and against the reference's OWN Shaders/Include/NRD.hlsli
    through the C++ HLSL shim (oracle/build_refshaders.py build_frontend_probe -> oracle/_ref/shaders/frontend_probe_ref, whose table
    is recorded in tests/golden/frontend_probe_reference.npz by tests/golden/make_reference_golden.py).  Same inputs, same 50 columns:
    packers, unpackers, hit-distance normalisation, SH / SG carriers and resolves, material factors, SIGMA penumbra / translucency.
    Bit-identical except the SG direction and the material factors, which agree to 2 ulp (a * rsqrt(dot) against a / length, the
    environment-term polynomial).  Both tables print float32 values with %.9g (exact) and column 5 as an integer."""
    mine = _run_probe()
    g = np.load(os.path.join(ROOT, "tests", "golden", "frontend_probe_reference.npz"))
    ref = np.insert(g["values"].astype(np.float64), 5, g["bits"].astype(np.float64), axis=1)
    assert mine.shape == ref.shape == (400, 50)
    mine = np.insert(np.delete(mine, 5, axis=1).astype(np.float32).astype(np.float64), 5, mine[:, 5], axis=1)
    loose = {40, 41, 42, 43, 44}
    for c in range(50):
        if c in loose:
            assert np.allclose(mine[:, c], ref[:, c], rtol=5e-7, atol=1e-7), c
        else:
            assert np.array_equal(mine[:, c], ref[:, c]), c
