"""Test infrastructure: a CPU "RHI" that executes the product scheduler's DispatchDesc[] on the oracle (oracle/liboracle.so).

It plays the role of the application / integration layer of the reference: it creates the pool textures the InstanceDesc
asks for (as numpy arrays), binds resources in DispatchDesc order and runs each dispatch through `oracle_dispatch`.
Only tests/, __graft_entry__.smoke() and bench.py's CPU legs may import this.
"""
import ctypes as C
import hashlib
import io
import lzma
import os

import numpy as np

from raytracingdenoiser_b200 import nrd

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_ORACLE_PATH = os.path.join(_ROOT, "oracle", "liboracle.so")


class OracleTexture(C.Structure):
    _fields_ = [("data", C.c_void_p), ("width", C.c_int32), ("height", C.c_int32), ("pitchBytes", C.c_int32), ("format", C.c_int32), ("firstRow", C.c_int32),
                ("originX", C.c_int32), ("originY", C.c_int32)]


_oracle = {}


def host_threads():
    """Threads the oracle may really use: the affinity mask capped by the cgroup CPU quota.  A container that sees 128 cores through
    sched_getaffinity may be throttled to 16 of them; an OpenMP team of 128 then thrashes (measured: 3-8x slower oracle passes)."""
    import math
    affinity = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    quota = None
    try:
        parts = open("/sys/fs/cgroup/cpu.max").read().split()  # cgroup v2: "<quota|max> <period>"
        if parts and parts[0] != "max":
            quota = float(parts[0]) / float(parts[1])
    except Exception:
        try:
            q, per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read()), float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    return affinity if quota is None else max(1, min(affinity, int(math.ceil(quota))))


def oracle_lib(variant=""):
    """variant "": the oracle (no FMA contraction); "fma": the same sources compiled with contraction allowed -- a second
    IEEE-legal evaluation; "uv": the same sources with the uv of every bilinear fetch moved by one float ulp (oracle/hlsl.h);
    "src": the reference's association order in the one helper where the oracle's differs (oracle/relax.cpp, used by
    tests/test_reference_shaders.py).  The fma / uv variants are used only to measure the rounding-noise floor of the temporal passes and chains (tests/parity.py)."""
    if variant not in _oracle:
        path = _ORACLE_PATH if not variant else _ORACLE_PATH.replace("liboracle.so", "liboracle_%s.so" % variant)
        if not os.path.exists(path):
            from raytracingdenoiser_b200 import build
            build.build_oracle(force=True)
        lib = C.CDLL(path)
        lib.oracle_dispatch.argtypes = [C.c_char_p, C.c_void_p, C.c_int, C.POINTER(OracleTexture), C.c_int, C.c_int, C.c_int]
        lib.oracle_dispatch.restype = C.c_int
        lib.oracle_num_threads.restype = C.c_int
        lib.oracle_set_num_threads.argtypes = [C.c_int]
        lib.oracle_set_num_threads.restype = None
        if not os.environ.get("OMP_NUM_THREADS"):
            lib.oracle_set_num_threads(host_threads())  # (each library build carries its own OpenMP setting)
        _oracle[variant] = lib
    return _oracle[variant]


_NP = {nrd.Format.R8_UNORM: (np.uint8, 1), nrd.Format.R8_UINT: (np.uint8, 1), nrd.Format.RG8_UNORM: (np.uint8, 2), nrd.Format.RGBA8_UNORM: (np.uint8, 4),
       nrd.Format.R16_UINT: (np.uint16, 1), nrd.Format.R16_SFLOAT: (np.float16, 1), nrd.Format.RGBA16_SFLOAT: (np.float16, 4), nrd.Format.R32_UINT: (np.uint32, 1),
       nrd.Format.R32_SFLOAT: (np.float32, 1), nrd.Format.R10_G10_B10_A2_UNORM: (np.uint32, 1), nrd.Format.RGBA32_SFLOAT: (np.float32, 4)}


_REFSHADERS = {}

# The reference's pass shaders compiled for the CPU (oracle/_ref/shaders, built only where the reference sources are present) are
# not part of the repository.  What the tests need of them is recorded in tests/golden/reference_shader_outputs.npz.xz by
# tests/golden/make_reference_golden.py: for every dispatch the tests run, keyed by a hash of its input state (shader,
# constants, grid, rect origin, every bound texture), the texels where the shader's outputs differ from the oracle's and a hash of
# each output.  run_reference_shader() replays a record: it runs the oracle's pass, writes the recorded texels over it and checks the
# result against the recorded hash, so the tests see the shader's exact output.  A dispatch that was not recorded, or an oracle
# whose output has changed since the recording, is an error, not a silent fall-back.
REFERENCE_GOLDEN = os.path.join(_ROOT, "tests", "golden", "reference_shader_outputs.npz.xz")  # (an .npz, xz-compressed)
RECORD_ENV = "NRD_B200_RECORD_REFERENCE_SHADERS"  # "1": run the compiled shaders and record them (make_reference_golden.py)
_recorded = {}
_golden = {}


def _recording():
    return os.environ.get(RECORD_ENV) == "1"


def _golden_records():
    if not _golden:
        with lzma.open(REFERENCE_GOLDEN) as f:
            z = np.load(io.BytesIO(f.read()))
        _golden["shaders"] = set(str(s) for s in z["shaders"])
        _golden["index"] = {bytes(k): i for i, k in enumerate(z["keys"])}
        for k in ("out_start", "out_sha", "diff_start", "diff_index", "value_start", "diff_value"):
            _golden[k] = z[k]
    return _golden


def _shader_name(shader_file_name):
    return shader_file_name[:-3] if shader_file_name.endswith(".cs") else shader_file_name


def has_reference_shader(shader_file_name):
    """Whether the reference has a compiled pass shader for this dispatch (the Clear_* passes have none)."""
    if _recording():
        return os.path.exists(reference_shader_path(shader_file_name))
    return _shader_name(shader_file_name) in _golden_records()["shaders"]


def _texels(arr):
    """(texels, bytes per texel) uint8 view of a texture (writes go through to it)."""
    return arr.reshape(arr.shape[0] * arr.shape[1], -1).view(np.uint8)


def _digest(arr):
    return hashlib.sha1(np.ascontiguousarray(arr).tobytes()).digest()[:8]


def save_reference_recording(path=REFERENCE_GOLDEN):
    """Writes what run_reference_shader() recorded (in RECORD_ENV mode) to `path`."""
    keys = sorted(_recorded)
    out_start, out_sha, diff_start, value_start, diff_index, diff_value = [0], [], [0], [0], [], []
    for k in keys:
        for sha, idx, val in _recorded[k]:
            out_sha.append(np.frombuffer(sha, dtype=np.uint8))
            diff_index.append(np.diff(idx, prepend=0))  # (gaps compress better than positions)
            diff_value.append(val.T.reshape(-1))         # byte planes: the XOR of nearly equal values is zero in its high bytes
            diff_start.append(diff_start[-1] + len(idx))
            value_start.append(value_start[-1] + val.size)
        out_start.append(len(out_sha))
    built = sorted(f[:-3] for f in os.listdir(os.path.dirname(reference_shader_path("x"))) if f.endswith(".so"))
    buf = io.BytesIO()
    np.savez(buf, keys=np.array([np.frombuffer(k, dtype=np.uint8) for k in keys]).reshape(-1, 8), shaders=np.array(built),
             out_start=np.array(out_start, dtype=np.int32), out_sha=np.array(out_sha).reshape(-1, 8),
             diff_start=np.array(diff_start, dtype=np.int64), value_start=np.array(value_start, dtype=np.int64),
             diff_index=np.concatenate(diff_index).astype(np.int32), diff_value=np.concatenate(diff_value).astype(np.uint8))
    with lzma.open(path, "wb", preset=9 | lzma.PRESET_EXTREME) as f:
        f.write(buf.getvalue())


def reference_shader_path(shader_file_name):
    return os.path.join(_ROOT, "oracle", "_ref", "shaders", _shader_name(shader_file_name) + ".so")


def reference_shader_lib(shader_file_name):
    """The reference's own shader source of one pass, compiled for the CPU by oracle/build_refshaders.py (only where the reference
    sources are present; used to record tests/golden/reference_shader_outputs.npz.xz)."""
    path = reference_shader_path(shader_file_name)
    if path not in _REFSHADERS:
        lib = C.CDLL(path)
        lib.refshader_dispatch.restype = C.c_int
        lib.refshader_dispatch.argtypes = [C.c_void_p, C.c_int, C.POINTER(OracleTexture), C.c_int, C.c_int, C.c_int]
        _REFSHADERS[path] = lib
    return _REFSHADERS[path]


def alloc(fmt, w, h):
    dt, ch = _NP[nrd.Format(fmt)]
    return np.zeros((h, w, ch) if ch > 1 else (h, w), dtype=dt)


class CpuDenoiser(object):
    """Mirror of harness.GpuDenoiser on the CPU: same scheduler (the product's), oracle passes, numpy textures."""

    def __init__(self, denoiser, width, height, identifier=0, settings=None, user_formats=None, instance=None, variant="", common=None):
        from raytracingdenoiser_b200 import harness
        self.width, self.height, self.identifier = width, height, identifier
        self.lib = oracle_lib(variant)
        self.instance = instance or nrd.Instance([(identifier, denoiser)])
        if settings is not None and instance is None:
            self.instance.set_denoiser_settings(identifier, settings)
        desc = self.instance.get_instance_desc()
        self.permanent = [alloc(f, (width + ds - 1) // ds, (height + ds - 1) // ds) for f, ds in desc["permanentPool"]]
        self.transient = [alloc(f, (width + ds - 1) // ds, (height + ds - 1) // ds) for f, ds in desc["transientPool"]]
        self.formats = {"permanent": [f for f, _ in desc["permanentPool"]], "transient": [f for f, _ in desc["transientPool"]]}
        self.user = {}
        self.user_fmt = {}
        self.rect_origin = (0, 0)  # CommonSettings::rectOrigin of the frame being run (set by denoise() / the parity harness)
        for name in harness.denoiser_resources(denoiser, common):
            fmt = harness.user_format(denoiser, name)[0]
            self.user[name] = alloc(fmt, width, height)
            self.user_fmt[name] = fmt

    def resolve(self, rtype, index):
        if rtype == nrd.ResourceType.PERMANENT_POOL:
            return self.permanent[index], self.formats["permanent"][index]
        if rtype == nrd.ResourceType.TRANSIENT_POOL:
            return self.transient[index], self.formats["transient"][index]
        name = nrd.ResourceType(rtype).name
        return self.user[name], self.user_fmt[name]

    def set_inputs(self, frame, rect_origin=(0, 0)):
        """Writes the frame's inputs into the user textures.  A frame smaller than the textures (dynamic resolution) goes to the
        top-left corner -- or, for the guide inputs an application binds from its G-buffer, to rect_origin (WithRectOrigin)."""
        from raytracingdenoiser_b200 import harness
        for name, arr in self.user.items():
            if name.startswith("IN_"):
                src = frame[name]
                src = src.cpu().numpy() if hasattr(src, "cpu") else np.asarray(src)
                src = src.view(arr.dtype).reshape((src.shape[0], src.shape[1]) + arr.shape[2:])
                ox, oy = rect_origin if name in harness.RECT_ORIGIN_INPUTS else (0, 0)
                arr[oy:oy + src.shape[0], ox:ox + src.shape[1]] = src

    def run_dispatch(self, d, lib=None):
        lib = lib or self.lib
        texs = (OracleTexture * len(d.resources))()
        keep = []
        from raytracingdenoiser_b200 import harness
        for i, (_, rtype, index) in enumerate(d.resources):
            arr, fmt = self.resolve(rtype, index)
            keep.append(arr)
            texs[i].originX = texs[i].originY = 0
            if nrd.ResourceType(rtype).name in harness.RECT_ORIGIN_INPUTS:
                texs[i].originX, texs[i].originY = self.rect_origin  # WithRectOrigin (Common.hlsli:200-205)
            texs[i].data = arr.ctypes.data
            texs[i].height, texs[i].width = arr.shape[0], arr.shape[1]
            texs[i].pitchBytes = arr.strides[0]
            texs[i].format = int(fmt)
            texs[i].firstRow = 0
        # the reported size is the reference's sizeof() (not padded to a 16-byte register); the oracle copies whole registers
        buf = C.create_string_buffer(d.constants, (len(d.constants) + 15) // 16 * 16) if d.constants else None
        r = lib.oracle_dispatch(d.shaderFileName.encode(), buf, len(d.constants), texs, len(d.resources), d.gridWidth, d.gridHeight)
        if r != 0:
            raise RuntimeError("oracle_dispatch(%s) failed with %d" % (d.shaderFileName, r))

    def _textures(self, d):
        from raytracingdenoiser_b200 import harness
        texs = (OracleTexture * len(d.resources))()
        keep = []
        for i, (_, rtype, index) in enumerate(d.resources):
            arr, fmt = self.resolve(rtype, index)
            keep.append(arr)
            texs[i].originX = texs[i].originY = 0
            if nrd.ResourceType(rtype).name in harness.RECT_ORIGIN_INPUTS:
                texs[i].originX, texs[i].originY = self.rect_origin
            texs[i].data = arr.ctypes.data
            texs[i].height, texs[i].width = arr.shape[0], arr.shape[1]
            texs[i].pitchBytes = arr.strides[0]
            texs[i].format = int(fmt)
            texs[i].firstRow = 0
        return texs, keep

    def _state_key(self, d):
        h = hashlib.sha1(d.shaderFileName.encode() + bytes(d.constants))
        h.update(np.array([d.gridWidth, d.gridHeight, self.rect_origin[0], self.rect_origin[1]], dtype=np.int64).tobytes())
        for _, rtype, index in d.resources:
            arr, fmt = self.resolve(rtype, index)
            h.update(np.array((int(rtype), int(fmt)) + arr.shape, dtype=np.int64).tobytes())
            h.update(np.ascontiguousarray(arr).tobytes())
        return h.digest()[:8]

    def run_reference_shader(self, d):
        """Executes the dispatch as the REFERENCE's own shader source compiled for the CPU (oracle/build_refshaders.py) computes it:
        replayed from tests/golden/reference_shader_outputs.npz.xz, or -- in RECORD_ENV mode -- run from oracle/_ref/shaders/<shader>.so
        and recorded."""
        outs = [self.resolve(rtype, index)[0] for dtype, rtype, index in d.resources if dtype == nrd.DescriptorType.STORAGE_TEXTURE]
        key = self._state_key(d)
        if _recording():
            before = [a.copy() for a in outs]
            self.run_dispatch(d, oracle_lib())
            mine = [a.copy() for a in outs]
            for a, b in zip(outs, before):
                a[...] = b
            lib = reference_shader_lib(d.shaderFileName)
            texs, keep = self._textures(d)
            buf = C.create_string_buffer(d.constants, (len(d.constants) + 15) // 16 * 16)
            r = lib.refshader_dispatch(buf, len(d.constants), texs, len(d.resources), d.gridWidth, d.gridHeight)
            if r != 0:
                raise RuntimeError("refshader_dispatch(%s) failed with %d" % (d.shaderFileName, r))
            record = []
            for a, m in zip(outs, mine):
                t, tm = _texels(a), _texels(m)
                idx = np.nonzero((t != tm).any(axis=1))[0].astype(np.int32)
                record.append((_digest(a), idx, t[idx] ^ tm[idx]))
            _recorded[key] = record
            return
        g = _golden_records()
        i = g["index"].get(key)
        if i is None:
            raise RuntimeError("%s: no recorded reference-shader output for this input state (inputs, scheduler or an earlier oracle pass changed "
                               "since tests/golden/reference_shader_outputs.npz.xz was recorded)" % d.shaderFileName)
        self.run_dispatch(d, oracle_lib())
        first, last = g["out_start"][i], g["out_start"][i + 1]
        assert last - first == len(outs), (d.shaderFileName, last - first, len(outs))
        for a, o in zip(outs, range(first, last)):
            t = _texels(a)
            idx = np.cumsum(g["diff_index"][g["diff_start"][o]:g["diff_start"][o + 1]])
            t[idx] ^= g["diff_value"][g["value_start"][o]:g["value_start"][o + 1]].reshape(t.shape[1], len(idx)).T
            if _digest(a) != g["out_sha"][o].tobytes():
                raise RuntimeError("%s: the oracle's output changed since tests/golden/reference_shader_outputs.npz.xz was recorded; the "
                                   "reference shader's output cannot be reproduced from it" % d.shaderFileName)

    def run_both(self, d):
        """Runs the dispatch twice on the same state -- the oracle's pass, then the reference's own shader -- and returns
        [(resource label, format, oracle output, reference-shader output, texture before the pass)] for every texture the pass writes.  The oracle's
        outputs stay in place (the chain continues on the oracle's state)."""
        outs = [(i, rtype, index) for i, (dtype, rtype, index) in enumerate(d.resources) if dtype == nrd.DescriptorType.STORAGE_TEXTURE]
        before = {i: self.resolve(rtype, index)[0].copy() for i, rtype, index in outs}
        self.run_dispatch(d)
        mine = {i: self.resolve(rtype, index)[0].copy() for i, rtype, index in outs}
        for i, rtype, index in outs:
            self.resolve(rtype, index)[0][...] = before[i]
        self.run_reference_shader(d)
        res = []
        for i, rtype, index in outs:
            arr, fmt = self.resolve(rtype, index)
            res.append(("%s[%d]" % (nrd.ResourceType(rtype).name, index), fmt, mine[i], arr.copy(), before[i]))
            arr[...] = mine[i]
        return res

    def denoise(self, common_settings, on_dispatch=None):
        self.rect_origin = (int(common_settings.rectOrigin[0]), int(common_settings.rectOrigin[1]))
        self.instance.set_common_settings(common_settings)
        dispatches = self.instance.get_compute_dispatches([self.identifier])
        for i, d in enumerate(dispatches):
            if on_dispatch:
                on_dispatch(i, d, "before")
            self.run_dispatch(d)
            if on_dispatch:
                on_dispatch(i, d, "after")
        return dispatches


def compare(a, b, fmt, rel=1e-3, abs_tol=1e-4, layout=None):
    """Per-channel parity metric of SURVEY.md 8(d): returns (fraction of texels within tolerance, worst excess factor)."""
    fmt = nrd.Format(fmt)
    if layout == "reblur_data2":
        # REBLUR PackData2 (REBLUR_Common.hlsli:59-70): bits 0-7 occlusion flags (exact), 8-15 virtual history amount
        # (UNORM8, 1 LSB), 16-31 curvature as FP16 (relative tolerance)
        a64, b64 = a.astype(np.int64), b.astype(np.int64)
        ok = (a64 & 0xFF) == (b64 & 0xFF)
        ok &= np.abs(((a64 >> 8) & 0xFF) - ((b64 >> 8) & 0xFF)) <= 1
        ca = ((a64 >> 16) & 0xFFFF).astype(np.uint16).view(np.float16).astype(np.float64)
        cb = ((b64 >> 16) & 0xFFFF).astype(np.uint16).view(np.float16).astype(np.float64)
        ca, cb = np.nan_to_num(ca, nan=1e30, posinf=1e30, neginf=-1e30), np.nan_to_num(cb, nan=1e30, posinf=1e30, neginf=-1e30)
        err, tol = np.abs(ca - cb), 2e-3 * np.maximum(np.abs(ca), np.abs(cb)) + abs_tol
        ok &= err <= tol
        return float(ok.mean()), float((err / tol).max())
    if fmt in (nrd.Format.RGBA16_SFLOAT, nrd.Format.R16_SFLOAT, nrd.Format.R32_SFLOAT, nrd.Format.RGBA32_SFLOAT):
        x, y = a.astype(np.float64), b.astype(np.float64)
        x = np.nan_to_num(x, nan=1e30, posinf=1e30, neginf=-1e30)
        y = np.nan_to_num(y, nan=1e30, posinf=1e30, neginf=-1e30)
        tol = rel * np.maximum(np.abs(x), np.abs(y)) + abs_tol
        err = np.abs(x - y)
        ok = err <= tol
        if ok.ndim == 3:
            ok_px = ok.all(axis=2)
        else:
            ok_px = ok
        worst = float((err / tol).max()) if err.size else 0.0
        return float(ok_px.mean()), worst
    if fmt == nrd.Format.R10_G10_B10_A2_UNORM:
        d = np.zeros(a.shape, dtype=np.int64)
        for shift, mask in ((0, 1023), (10, 1023), (20, 1023), (30, 3)):
            d = np.maximum(d, np.abs(((a.astype(np.int64) >> shift) & mask) - ((b.astype(np.int64) >> shift) & mask)))
        return float((d <= 1).mean()), float(d.max())
    if fmt == nrd.Format.R16_UINT:  # REBLUR internal data: 6 + 6 + 4 bits
        d = np.zeros(a.shape, dtype=np.int64)
        for shift, mask in ((0, 63), (6, 63), (12, 15)):
            d = np.maximum(d, np.abs(((a.astype(np.int64) >> shift) & mask) - ((b.astype(np.int64) >> shift) & mask)))
        return float((d <= 1).mean()), float(d.max())
    if fmt == nrd.Format.R32_UINT:
        same = a == b
        return float(same.mean()), float((~same).sum())
    d = np.abs(a.astype(np.int64) - b.astype(np.int64))
    ok = d <= 1
    if ok.ndim == 3:
        ok = ok.all(axis=2)
    return float(ok.mean()), float(d.max())


def _excess_map(a, b, fmt, rel, abs_tol, layout=None):
    """Per-texel error in units of the tolerance (max over channels), and a mask of non-finite kernel values where the oracle is finite."""
    fmt = nrd.Format(fmt)
    if layout == "reblur_data2":
        a64, b64 = a.astype(np.int64), b.astype(np.int64)
        ex = np.where((a64 & 0xFF) == (b64 & 0xFF), 0.0, 1e9)
        ex = np.maximum(ex, np.abs(((a64 >> 8) & 0xFF) - ((b64 >> 8) & 0xFF)).astype(np.float64))
        ca = ((a64 >> 16) & 0xFFFF).astype(np.uint16).view(np.float16).astype(np.float64)
        cb = ((b64 >> 16) & 0xFFFF).astype(np.uint16).view(np.float16).astype(np.float64)
        bad = np.isfinite(ca) & ~np.isfinite(cb)
        ca, cb = np.nan_to_num(ca, nan=1e30, posinf=1e30, neginf=-1e30), np.nan_to_num(cb, nan=1e30, posinf=1e30, neginf=-1e30)
        ex = np.maximum(ex, np.abs(ca - cb) / (2e-3 * np.maximum(np.abs(ca), np.abs(cb)) + abs_tol))
        return ex, bad
    if fmt in (nrd.Format.RGBA16_SFLOAT, nrd.Format.R16_SFLOAT, nrd.Format.R32_SFLOAT, nrd.Format.RGBA32_SFLOAT):
        x, y = a.astype(np.float64), b.astype(np.float64)
        bad = np.isfinite(x) & ~np.isfinite(y)
        x = np.nan_to_num(x, nan=1e30, posinf=1e30, neginf=-1e30)
        y = np.nan_to_num(y, nan=1e30, posinf=1e30, neginf=-1e30)
        ex = np.abs(x - y) / (rel * np.maximum(np.abs(x), np.abs(y)) + abs_tol)
        if ex.ndim == 3:
            ex, bad = ex.max(axis=2), bad.any(axis=2)
        return ex, bad
    ai, bi = a.astype(np.int64), b.astype(np.int64)
    if fmt == nrd.Format.R10_G10_B10_A2_UNORM:
        fields = ((0, 1023), (10, 1023), (20, 1023), (30, 3))
    elif fmt == nrd.Format.R16_UINT:
        fields = ((0, 63), (6, 63), (12, 15))
    elif fmt == nrd.Format.R32_UINT:
        return np.where(ai == bi, 0.0, 1e9), np.zeros(a.shape[:2], dtype=bool)
    else:
        d = np.abs(ai - bi).astype(np.float64)
        return (d.max(axis=2) if d.ndim == 3 else d), np.zeros(a.shape[:2], dtype=bool)
    d = np.zeros(a.shape, dtype=np.float64)
    for shift, mask in fields:
        d = np.maximum(d, np.abs(((ai >> shift) & mask) - ((bi >> shift) & mask)))
    return d, np.zeros(a.shape[:2], dtype=bool)


def outliers(a, b, fmt, rel=1e-3, abs_tol=1e-4, max_excess=10.0, layout=None, list_limit=16):
    """Outlier gate of tests/parity.py: (number of texels further off than max_excess x tolerance, [[x, y, excess], ...] of the
    worst `list_limit`, number of texels that are non-finite in `b` but finite in `a`).  LSB-compared formats count a texel
    as an outlier when it is more than max_excess LSBs off."""
    ex, bad = _excess_map(a, b, fmt, rel, abs_tol, layout)
    mask = ex > max_excess
    n = int(mask.sum())
    where = []
    if n:
        ys, xs = np.nonzero(mask)
        order = np.argsort(-ex[ys, xs])[:list_limit]
        where = [[int(xs[i]), int(ys[i]), float(min(ex[ys[i], xs[i]], 1e9))] for i in order]
    return n, where, int(bad.sum())
