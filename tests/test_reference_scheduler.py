"""Row a1 pinned against the reference's OWN host code.

oracle/_ref/libnrd_ref.so is built by oracle/Makefile.ref from the reference's Source/*.cpp (NRD v4.14.0, untouched) with every
NRD_EMBEDS_* option off and MathLib's ml.h replaced by the documented shim in oracle/ref_shim/.  What that library answers to the
calls below is recorded in tests/golden/reference_scheduler.json.xz (tests/golden/make_reference_golden.py, where the reference
sources are present); the tests drive the product scheduler (libnrd_b200.so) through the same nine NRD entry points with the same
inputs and demand IDENTICAL output: InstanceDesc (pipelines, shader names, resource ranges, pools, descriptor counts), and for
every frame the dispatch list -- order, names, identifiers, pipeline indices, resources (descriptor type, resource type, pool
index after ping-pong), grids, constantBufferDataSize, constantBufferDataMatchesPreviousDispatch and a 64-bit digest of the
constant bytes (with the reference library present, every constant field by name).

What this pins and what it cannot: everything above is NVIDIA's code talking, except the values the reference computes with
MathLib alone, which come out of the shim (a restatement with the same semantics as csrc/hostmath.h, so they agree by
construction): SHIM_DEPENDENT lists those constant fields; they are compared too, but agreement there proves nothing about the
real MathLib.  All other fields (sizes, scales, thresholds, frame counters, blur radii, checkerboard/perf/validation flags,
history resets, ...) are pinned for real.
"""
import ctypes as C
import hashlib
import json
import lzma
import os
import re

import numpy as np
import pytest

from raytracingdenoiser_b200 import nrd, scene

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_LIB = os.path.join(ROOT, "oracle", "_ref", "libnrd_ref.so")
GOLDEN = os.path.join(ROOT, "tests", "golden", "reference_scheduler.json.xz")
RECORD_ENV = "NRD_B200_RECORD_REFERENCE_SCHEDULER"  # "1": drive oracle/_ref/libnrd_ref.so and record it (make_reference_golden.py)

# constant-block fields whose value depends on shimmed MathLib functions (matrix inverses / products, DecomposeProjection,
# Sequence::Weyl1D / Bayer4x4, Geometry::GetRotator / CombineRotators, Rotate)
SHIM_DEPENDENT = {"gWorldToClip", "gViewToClip", "gViewToWorld", "gWorldToViewPrev", "gWorldToClipPrev", "gWorldPrevToWorld", "gWorldToView", "gRotatorPre",
                  "gRotator", "gRotatorPost", "gFrustum", "gFrustumPrev", "gCameraDelta", "gViewVectorWorld", "gViewVectorWorldPrev", "gOrthoMode", "gUnproject",
                  "gMinRectDimMulUnproject", "gFrustumRight", "gFrustumUp", "gFrustumForward", "gPrevFrustumRight", "gPrevFrustumUp", "gPrevFrustumForward",
                  "gLightDirectionView"}


def _digest(b):
    return hashlib.sha1(b).hexdigest()[:16]


def _plain(x):
    """JSON-shaped copy (enums -> ints, tuples -> lists): how a recorded answer is stored and compared."""
    return json.loads(json.dumps(x))


class _Recorded(object):
    """Stand-in for the reference library's nrd.Instance: in RECORD_ENV mode it drives oracle/_ref/libnrd_ref.so and records every
    answer under `session`; otherwise it replays tests/golden/reference_scheduler.json.xz, answer by answer, for the same calls."""
    log = {}
    _answers = None

    def __init__(self, session, denoisers):
        self.session, self.calls = session, []
        if os.environ.get(RECORD_ENV) == "1":
            try:
                self.inst = nrd.Instance(denoisers, lib=_ref_lib())
            except nrd.NrdError:
                self.log[session] = [["CreateInstance", "raise"]]
                raise
            self.log[session] = self.calls
        else:
            if _Recorded._answers is None:
                _Recorded._answers = _golden()
            if session not in self._answers:
                raise AssertionError("no recorded reference answer for %s (tests/golden/make_reference_golden.py records them)" % session)
            self.inst, self.replay = None, list(self._answers[session])
            if self.replay[0] == ["CreateInstance", "raise"]:
                raise nrd.NrdError("CreateInstance", nrd.Result.INVALID_ARGUMENT)

    def _call(self, what, fn, encode=_plain):
        if self.inst is not None:
            v = fn()
            self.calls.append([what, encode(v)])
            return v
        name, v = self.replay.pop(0)
        assert name == what, (self.session, "calls differ from the recorded ones", name, what)
        return v

    def get_instance_desc(self):
        return self._call("desc", lambda: self.inst.get_instance_desc())

    def set_denoiser_settings(self, identifier, settings, check=True):
        key = "settings %d %s" % (identifier, _digest(C.string_at(C.addressof(settings), C.sizeof(settings))))
        return self._call(key, lambda: self.inst.set_denoiser_settings(identifier, settings, check=check), int)

    def set_common_settings(self, cs, check=True):
        key = "common %s" % _digest(C.string_at(C.addressof(cs), C.sizeof(cs)))
        return self._call(key, lambda: self.inst.set_common_settings(cs, check=check), int)

    def get_compute_dispatches_raw(self, ids):
        return self._call("raw %s" % list(ids), lambda: self.inst.get_compute_dispatches_raw(ids)[:1], lambda v: [int(v[0])])

    def get_compute_dispatches(self, ids):
        rows = self._call("dispatches %s" % list(ids), lambda: self.inst.get_compute_dispatches(ids),
                          lambda ds: [[d.name, d.identifier, _plain(d.resources), d.pipelineIndex, d.shaderFileName, d.gridWidth, d.gridHeight,
                                       d.constantsMatchPrevious, len(d.constants), _digest(d.constants)] for d in ds])
        if self.inst is not None:
            return rows
        out = []
        for r in rows:
            d = _RecordedDispatch()
            (d.name, d.identifier, res, d.pipelineIndex, d.shaderFileName, d.gridWidth, d.gridHeight, d.constantsMatchPrevious, d.size, d.digest) = r
            d.resources = [tuple(x) for x in res]
            out.append(d)
        return out

    def destroy(self):
        if self.inst is not None:
            self.inst.destroy()


class _RecordedDispatch(object):
    """A dispatch of the reference as recorded: the constant bytes are represented by their size and digest."""


_REF = {}


def _ref_lib():
    if "lib" not in _REF:
        _REF["lib"] = nrd.bind_nrd_api(C.CDLL(REF_LIB))
    return _REF["lib"]


def _library_answers():
    lib = _ref_lib()
    d = lib.GetLibraryDesc().contents
    return {"version": [d.versionMajor, d.versionMinor, d.versionBuild, d.normalEncoding, d.roughnessEncoding],
            "resourceTypeStrings": [lib.GetResourceTypeString(i).decode() for i in range(len(nrd.ResourceType))],
            "denoiserStrings": [lib.GetDenoiserString(i).decode() for i in range(len(nrd.Denoiser))],
            "supportedDenoisers": sorted(int(d.supportedDenoisers[i]) for i in range(d.supportedDenoisersNum))}


def save_recording():
    """Writes what _Recorded recorded (in RECORD_ENV mode), and the library's own descriptions, to GOLDEN."""
    log = dict(_Recorded.log, library=_library_answers())
    with lzma.open(GOLDEN, "wt", preset=9 | lzma.PRESET_EXTREME) as f:
        json.dump(log, f, sort_keys=True)


def _golden():
    with lzma.open(GOLDEN, "rt") as f:
        return json.load(f)


def _library():
    if os.environ.get(RECORD_ENV) == "1":
        return _library_answers()
    return _golden()["library"]


def _fields(struct_name):
    """(name, offset, size) of every member of a constant block, parsed from csrc/constants.h (4-byte scalars and arrays)."""
    src = open(os.path.join(ROOT, "raytracingdenoiser_b200", "csrc", "constants.h")).read()
    body = re.search(r"struct alignas\(16\) %s\s*\{(.*?)\n\};" % struct_name, src, re.S).group(1)
    out, off = [], 0
    for m in re.finditer(r"^\s*(float|uint32_t|int32_t)\s+(\w+)(?:\[(\d+)\])?;", body, re.M):
        n = int(m.group(3) or 1)
        out.append((m.group(2), off, 4 * n))
        off += 4 * n
    return out


FIELDS = {"REBLUR": _fields("ReblurConstants"), "RELAX": _fields("RelaxConstants"), "SIGMA": _fields("SigmaConstants")}


def _common(f, w, h, variant):
    cs = nrd.CommonSettings()
    if variant == "ortho":
        P = np.zeros((4, 4), dtype=np.float32)
        P[0, 0], P[1, 1], P[2, 2], P[2, 3], P[3, 3] = 0.1, 0.1 * w / h, 0.01, 0.0, 1.0
    else:
        P = scene.perspective_lh(60.0 if variant != "fov45" else 45.0, w / float(h))
    if variant == "rh":   # right-handed projection and view: the scheduler converts to left-handed (InstanceImpl.cpp:392-408)
        P = P.copy()
        P[:, 2] = -P[:, 2]
    eye = (0.3 * f, 1.7, -4.0 + 0.05 * f)
    V = scene.look_at_lh(eye, 0.02 * f, -0.1)
    Vp = scene.look_at_lh((0.3 * (f - 1), 1.7, -4.0 + 0.05 * (f - 1)), 0.02 * (f - 1), -0.1) if f else V
    if variant == "rh":
        V, Vp = V.copy(), Vp.copy()
        V[2, :], Vp[2, :] = -V[2, :], -Vp[2, :]
    for k, m in (("viewToClipMatrix", P), ("viewToClipMatrixPrev", P), ("worldToViewMatrix", V), ("worldToViewMatrixPrev", Vp)):
        for i, v in enumerate(scene.colmajor(m)):
            getattr(cs, k)[i] = v
    rw, rh = (w, h) if variant != "dynres" else (w * 3 // 4, h * 2 // 3)
    for k in ("resourceSize", "resourceSizePrev"):
        getattr(cs, k)[0], getattr(cs, k)[1] = w, h
    for k in ("rectSize", "rectSizePrev"):
        getattr(cs, k)[0], getattr(cs, k)[1] = rw, rh
    if variant == "dynres" and f == 2:
        cs.rectSizePrev[0], cs.rectSizePrev[1] = w, h   # the rect changed since the previous frame
        cs.rectOrigin[0], cs.rectOrigin[1] = 16, 8
    cs.motionVectorScale[0], cs.motionVectorScale[1], cs.motionVectorScale[2] = 1.0 / w, 1.0 / h, 1.0
    cs.timeDeltaBetweenFrames = 16.6667 if variant != "slow" else 41.0
    cs.frameIndex = f
    if variant == "jitter":
        cs.cameraJitter[0], cs.cameraJitter[1] = 0.25 * ((f % 2) * 2 - 1), -0.125
        cs.cameraJitterPrev[0], cs.cameraJitterPrev[1] = 0.25 * (((f + 1) % 2) * 2 - 1), 0.125
    if variant == "restart" and f == 2:
        cs.accumulationMode = int(nrd.AccumulationMode.RESTART)
    if variant == "clear" and f == 2:
        cs.accumulationMode = int(nrd.AccumulationMode.CLEAR_AND_RESTART)
    if variant == "validation":
        cs.enableValidation = True
        cs.splitScreen = 0.5
    if variant == "inputs":
        cs.isHistoryConfidenceAvailable = True
        cs.isDisocclusionThresholdMixAvailable = True
        cs.isBaseColorMetalnessAvailable = True
        cs.isMotionVectorInWorldSpace = True
        cs.viewZScale = 2.0
        cs.denoisingRange = 1000.0
    return cs


COMMON_VARIANTS = ["default", "fov45", "ortho", "rh", "dynres", "slow", "jitter", "restart", "clear", "validation", "inputs"]


def _settings_variants(den):
    name = den.name
    if name.startswith("REBLUR"):
        yield "defaults", None
        yield "spatial_only", nrd.ReblurSettings(maxAccumulatedFrameNum=0, maxFastAccumulatedFrameNum=0, maxStabilizedFrameNum=0, historyFixFrameNum=0,
                                                 diffusePrepassBlurRadius=0.0, specularPrepassBlurRadius=0.0)
        yield "perf_hitdist3x3_checkerboard", nrd.ReblurSettings(enablePerformanceMode=True, hitDistanceReconstructionMode=int(nrd.HitDistanceReconstructionMode.AREA_3X3),
                                                                 checkerboardMode=int(nrd.CheckerboardMode.WHITE), enableAntiFirefly=True)
        yield "tuned", nrd.ReblurSettings(maxAccumulatedFrameNum=63, maxFastAccumulatedFrameNum=3, maxStabilizedFrameNum=10, historyFixFrameNum=2, historyFixBasePixelStride=8,
                                          maxBlurRadius=15.0, minBlurRadius=2.0, lobeAngleFraction=0.3, roughnessFraction=0.2, planeDistanceSensitivity=0.05,
                                          hitDistanceReconstructionMode=int(nrd.HitDistanceReconstructionMode.AREA_5X5), checkerboardMode=int(nrd.CheckerboardMode.BLACK),
                                          minMaterialForDiffuse=1.0, minMaterialForSpecular=2.0, usePrepassOnlyForSpecularMotionEstimation=True,
                                          hitDistanceParameters=nrd.HitDistanceParameters(A=2.0, B=0.2, C=10.0, D=-15.0))
    elif name.startswith("RELAX"):
        yield "defaults", None
        s = nrd.RelaxSettings()
        s.atrousIterationNum, s.enableRoughnessEdgeStopping, s.historyFixFrameNum, s.diffusePrepassBlurRadius, s.enableAntiFirefly = 3, False, 2, 0.0, True
        yield "three_iterations_antifirefly", s
        s = nrd.RelaxSettings()
        s.atrousIterationNum, s.hitDistanceReconstructionMode, s.checkerboardMode = 8, int(nrd.HitDistanceReconstructionMode.AREA_5X5), int(nrd.CheckerboardMode.BLACK)
        s.diffuseMaxAccumulatedFrameNum, s.specularMaxFastAccumulatedFrameNum, s.depthThreshold, s.specularVarianceBoost = 50, 2, 0.01, 1.5
        yield "eight_iterations_hitdist_checkerboard", s
    elif name == "REFERENCE":
        yield "defaults", None
        yield "short", nrd.ReferenceSettings(maxAccumulatedFrameNum=2)
    else:
        yield "defaults", None
        yield "no_stabilization", nrd.SigmaSettings(maxStabilizedFrameNum=0, lightDirection=[0.3, -0.8, 0.5])
        yield "long_history", nrd.SigmaSettings(maxStabilizedFrameNum=40, planeDistanceSensitivity=0.1, lightDirection=[0.0, -1.0, 0.0])


def _family(shader):
    return shader.split("_")[0] if shader.split("_")[0] in FIELDS else None


def _diff_constants(p, q):
    """names of the constant fields that differ between two dispatches of the same pass"""
    a, b = np.frombuffer(p.constants, dtype=np.uint8), np.frombuffer(q.constants, dtype=np.uint8)
    fam = _family(p.shaderFileName)
    bad = []
    covered = np.zeros(len(a), dtype=bool)
    for name, off, size in FIELDS.get(fam, []):
        if off + size <= len(a):
            covered[off:off + size] = True
            if not np.array_equal(a[off:off + size], b[off:off + size]):
                bad.append(name)
    if not np.array_equal(a[~covered], b[~covered]):
        bad.append("<bytes beyond the shared block>")
    return bad


def _constants_differ(p, q):
    """What differs between the constants of a product dispatch and the reference's: field names where the reference library
    answered, else whether the recorded size / digest differ."""
    if isinstance(q, _RecordedDispatch):
        return [] if (len(p.constants), _digest(p.constants)) == (q.size, q.digest) else ["<constant bytes (recorded size %d, digest %s)>" % (q.size, q.digest)]
    return (["<size %d vs %d>" % (len(p.constants), len(q.constants))] if len(p.constants) != len(q.constants) else []) + _diff_constants(p, q)


def _compare_streams(den, sname, settings, variant, frames=3, w=1920, h=1080):
    a, b = nrd.Instance([(7, den)]), _Recorded("stream %s %s %s" % (den.name, sname, variant), [(7, den)])
    assert _plain(a.get_instance_desc()) == _plain(b.get_instance_desc())
    if settings is not None:
        assert a.set_denoiser_settings(7, settings) == b.set_denoiser_settings(7, settings)
    checked = {"dispatches": 0, "pinned_fields": set(), "shim_fields": set()}
    for f in range(frames):
        cs = _common(f, w, h, variant)
        assert a.set_common_settings(cs, check=False) == b.set_common_settings(cs, check=False)
        xa, xb = a.get_compute_dispatches([7]), b.get_compute_dispatches([7])
        assert [d.name for d in xa] == [d.name for d in xb], (den.name, variant, f)
        for p, q in zip(xa, xb):
            for attr in ("name", "identifier", "resources", "pipelineIndex", "shaderFileName", "gridWidth", "gridHeight", "constantsMatchPrevious"):
                assert getattr(p, attr) == getattr(q, attr), (den.name, variant, f, p.name, attr, getattr(p, attr), getattr(q, attr))
            assert not _constants_differ(p, q), (den.name, variant, f, p.name, _constants_differ(p, q))
            checked["dispatches"] += 1
            for name, off, size in FIELDS.get(_family(p.shaderFileName), []):
                if off + size <= len(p.constants):
                    checked["shim_fields" if name in SHIM_DEPENDENT else "pinned_fields"].add(name)
    a.destroy()
    b.destroy()
    return checked


SUPPORTED = ["REBLUR_DIFFUSE", "REBLUR_SPECULAR", "REBLUR_DIFFUSE_SPECULAR", "RELAX_DIFFUSE", "RELAX_SPECULAR", "RELAX_DIFFUSE_SPECULAR", "SIGMA_SHADOW", "SIGMA_SHADOW_TRANSLUCENCY", "REFERENCE"]


@pytest.mark.parametrize("denoiser_name", SUPPORTED)
def test_dispatch_stream_identical_to_reference_host_code(denoiser_name):
    den = getattr(nrd.Denoiser, denoiser_name)
    total, pinned = 0, set()
    for sname, settings in _settings_variants(den):
        for variant in COMMON_VARIANTS:
            c = _compare_streams(den, sname, settings, variant)
            total += c["dispatches"]
            pinned |= c["pinned_fields"]
    assert (total > 300 and len(pinned) >= 18) or (denoiser_name == "REFERENCE" and total >= 40), (total, len(pinned))   # SIGMA has 20 fields that do not depend on MathLib, REBLUR 60


def test_library_desc_and_strings_match_reference():
    ref = _library()
    mine = nrd.get_library_desc()
    assert ref["version"] == [mine["versionMajor"], mine["versionMinor"], mine["versionBuild"], mine["normalEncoding"], mine["roughnessEncoding"]]
    # Documented deviation: the reference's resource-name table (Source/Wrapper.cpp:58-95) is not in the order of its own enum
    # (NRDDescs.h:43-137), e.g. enumerator 3 = IN_DIFF_CONFIDENCE is named "IN_DIFF_RADIANCE_HITDIST".  The product returns the
    # enumerator's own name; the two tables hold the same strings.
    ref_names = ref["resourceTypeStrings"]
    my_names = [nrd.get_resource_type_string(i) for i in range(len(nrd.ResourceType))]
    assert my_names == [t.name for t in nrd.ResourceType] and sorted(ref_names) == sorted(my_names)
    assert ref_names[:3] == my_names[:3] and ref_names[3] != my_names[3]
    assert ref["denoiserStrings"] == [nrd.get_denoiser_string(i) for i in range(len(nrd.Denoiser))]
    # every denoiser the product advertises is one the reference has, and creating an unadvertised one fails loudly
    assert {int(x) for x in mine["supportedDenoisers"]} <= set(ref["supportedDenoisers"])


def test_two_denoisers_in_one_instance_share_the_transient_pool_like_the_reference():
    dens = [(1, nrd.Denoiser.SIGMA_SHADOW), (2, nrd.Denoiser.REBLUR_DIFFUSE_SPECULAR), (5, nrd.Denoiser.RELAX_DIFFUSE_SPECULAR)]
    a, b = nrd.Instance(dens), _Recorded("transient pool", dens)
    assert _plain(a.get_instance_desc()) == _plain(b.get_instance_desc())
    for f in range(3):
        cs = _common(f, 1280, 720, "default")
        a.set_common_settings(cs)
        b.set_common_settings(cs)
        for ids in ([1, 2, 5], [5], [2, 1]):
            xa, xb = a.get_compute_dispatches(ids), b.get_compute_dispatches(ids)
            assert len(xa) == len(xb)
            for p, q in zip(xa, xb):
                assert (p.name, p.identifier, p.resources, p.pipelineIndex, p.gridWidth, p.gridHeight, p.constantsMatchPrevious) == (
                    q.name, q.identifier, q.resources, q.pipelineIndex, q.gridWidth, q.gridHeight, q.constantsMatchPrevious), (f, ids, p.name)
                assert not _constants_differ(p, q), (f, ids, p.name, _constants_differ(p, q))


def test_error_codes_match_reference():
    for inst in (nrd.Instance([(3, nrd.Denoiser.SIGMA_SHADOW)]), _Recorded("error codes", [(3, nrd.Denoiser.SIGMA_SHADOW)])):
        cs = _common(0, 640, 360, "default")
        cs.viewZScale = 0.0
        try:
            r = inst.set_common_settings(cs, check=False)
        except Exception:
            r = None
        results = [r]
        cs = _common(0, 640, 360, "default")
        inst.set_common_settings(cs)
        results.append(inst.set_denoiser_settings(99, nrd.SigmaSettings(), check=False))
        results.append(inst.get_compute_dispatches_raw([])[0])
        results.append(inst.get_compute_dispatches_raw([42])[0])
        if not isinstance(inst, _Recorded):
            mine = results
        else:
            assert mine == results, (mine, results)
    with pytest.raises(nrd.NrdError):
        nrd.Instance([(0, nrd.Denoiser.SIGMA_SHADOW), (0, nrd.Denoiser.SIGMA_SHADOW)])
    with pytest.raises(nrd.NrdError):
        _Recorded("duplicate identifiers", [(0, nrd.Denoiser.SIGMA_SHADOW), (0, nrd.Denoiser.SIGMA_SHADOW)])
