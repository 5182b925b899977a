"""Shared machinery of the GPU parity tests: run the oracle and the CUDA executor side by side on one nrd.Instance.

per-pass parity ("hard gate", SURVEY.md 8(d)): before every dispatch the CUDA context's textures are overwritten with the
oracle's state, the SAME DispatchDesc is executed by both, and every texture the pass writes is compared.
sequence parity ("statistical gate"): both executors run the whole chain on their own state for N frames.
"""
import ctypes as C

import numpy as np

import oracle_runner as orr
from raytracingdenoiser_b200 import harness, nrd, scene

# tolerance of north_star: 1e-3 relative (+1e-4 absolute floor); >= 99.9 % of texels within it.
# Outlier gate (SURVEY.md 8(d) "no pixel worse than 10x tolerance ... list outliers by cause"): a texel further off than
# MAX_EXCESS x tolerance is only ever a *decision flip* -- a tap whose pre-floor() coordinate, or a step()/compare operand, sits
# within rounding distance of its threshold, so that oracle and kernel legitimately pick different texels / branches (the chain
# feeds 1-rpp noise, a different texel is a different value, not a slightly different one).  Such texels are budgeted, not
# tolerated silently: at most OUTLIER_BUDGET of the texels of an output (and never fewer than OUTLIER_FLOOR allowed, so that tiny
# test frames are not failed by a single flip), every one is listed in the report with its position, and non-finite values
# (NaN / Inf where the oracle is finite) are never accepted.
REL, ABS, MIN_FRACTION, MAX_EXCESS = 1e-3, 1e-4, 0.999, 10.0
OUTLIER_BUDGET, OUTLIER_FLOOR = 5e-5, 4


def _scene_device(width, height, device):
    """Big frames are ray-cast on the GPU (input generation only; both executors get the same bytes): a 4K frame takes over a
    minute with torch on the CPU."""
    return "cuda:%d" % device if width * height > 1000000 else "cpu"


class _NoCuda(object):
    """Stand-in for the torch module when the harness runs on a CPU executor (tests/test_parity_harness.py)."""
    class cuda(object):
        @staticmethod
        def synchronize():
            pass


class SideBySide(object):
    def __init__(self, denoiser, width, height, settings=None, device=0, identifier=0, noise_floor=False, floor_passes=("TemporalAccumulation",), common=None, frame_fn=None, reference_shaders=False, executor=None):
        """executor: None = the CUDA executor (nrd.CudaContext); tests/test_parity_harness.py passes a CPU stand-in with the same
        upload / download / execute_raw methods to exercise this harness without a GPU.
        reference_shaders=True: the CPU side of every pass that has one is the REFERENCE's own shader source compiled for the CPU
        (oracle/build_refshaders.py; tests/oracle_runner.py run_reference_shader) instead of the oracle's restatement -- the kernels
        are compared with the reference's code directly, and the chain continues on the reference's state.
        frame_fn(frame, f) -> frame: transformation of the scene's frame f before either executor sees it (checkerboarded inputs).
        noise_floor=True: the dispatches whose shader name contains one of `floor_passes` are also run, on the same re-synchronised
        inputs, by two perturbed builds of the oracle -- "fma" (FMA contraction allowed: a second IEEE-legal evaluation of the same
        expressions) and "uv" (the uv of every bilinear fetch moved by one float ulp: the sub-texel position a shader hands to the
        sampler is only known to ulp(uv) * size = 2.4e-4 texel at 4K; the kernels merge the bilinear taps of the CatRom filter with
        exact weights).  Their disagreement with the oracle is the rounding-noise floor of the pass.  A pass whose floor is below
        the plain gate (RELAX temporal accumulation: acos of nearly parallel vectors, sigma of cancelling moments, CatRom history
        of the second moment across a contrast edge) is held to its floor instead -- the kernel must agree with the oracle at
        least as well as the oracle agrees with itself."""
        import torch
        self.denoiser, self.w, self.h, self.identifier, self.common = denoiser, width, height, identifier, common
        self.frame_fn = frame_fn
        self.reference_shaders = reference_shaders
        self.cpu = orr.CpuDenoiser(denoiser, width, height, identifier=identifier, settings=settings, common=common)
        self.instance = self.cpu.instance
        self.floor_passes = tuple(floor_passes)
        self.cpu_alt = [orr.CpuDenoiser(denoiser, width, height, identifier=identifier, instance=self.instance, variant=v, common=common) for v in ("fma", "uv")] if noise_floor else []
        self.report = []
        if executor is not None:
            self.ctx, self.torch, self.dev_user = executor(self), _NoCuda, {}
            self.scene = scene.Scene(width, height, device="cpu")
            return
        self.ctx = nrd.CudaContext(self.instance, width, height, device=device)
        self.torch = torch
        self.dev_user = {}
        for name in harness.denoiser_resources(denoiser, common):
            fmt, dtype, ch = harness.user_format(denoiser, name)
            t = torch.zeros((height, width, ch) if ch > 1 else (height, width), dtype=dtype, device="cuda:%d" % device)
            self.dev_user[name] = t
            self.ctx.set_user_texture(getattr(nrd.ResourceType, name), t.data_ptr(), t.stride(0) * t.element_size(), fmt)
        self.scene = scene.Scene(width, height, device=_scene_device(width, height, device))
        self.report = []

    def _cpu_run(self, d):
        if self.reference_shaders and orr.has_reference_shader(d.shaderFileName):
            self.cpu.run_reference_shader(d)
        else:
            self.cpu.run_dispatch(d)

    def _scene_frame(self, sc, f):
        fr = sc.frame(f, harness.radiance_mode(self.denoiser))
        return self.frame_fn(fr, f) if self.frame_fn else fr

    def _has_floor(self, d):
        return any(k in d.shaderFileName for k in self.floor_passes)

    def _sync_to_gpu(self, d):
        for _, rtype, index in d.resources:
            arr, _ = self.cpu.resolve(rtype, index)
            self.ctx.upload(rtype, index, np.ascontiguousarray(arr))

    def _compare_outputs(self, frame, d):
        for dtype_, rtype, index in d.resources:
            if dtype_ != nrd.DescriptorType.STORAGE_TEXTURE:
                continue
            ref, fmt = self.cpu.resolve(rtype, index)
            got = np.empty_like(ref)
            self.ctx.download(rtype, index, got)
            layout = "reblur_data2" if ("REBLUR" in d.shaderFileName and "TemporalAccumulation" in d.shaderFileName and fmt == nrd.Format.R32_UINT) else None
            frac, worst = orr.compare(ref, got, fmt, REL, ABS, layout=layout)
            n_out, where, nonfinite = orr.outliers(ref, got, fmt, REL, ABS, MAX_EXCESS, layout=layout)
            rec = {"frame": frame, "pass": d.name, "shader": d.shaderFileName, "resource": "%s[%d]" % (nrd.ResourceType(rtype).name, index),
                   "format": nrd.Format(fmt).name, "fraction": frac, "worst": worst, "texels": int(ref.shape[0] * ref.shape[1]),
                   "outliers": n_out, "outlier_budget": outlier_budget(ref.shape[0] * ref.shape[1]), "outliers_at": where, "nonfinite": nonfinite,
                   "outlier_cause": "decision flip (tap texel / step threshold within rounding distance)" if n_out else None,
                   "min_fraction": MIN_FRACTION}
            if self.cpu_alt and self._has_floor(d):
                for alt_den in self.cpu_alt:
                    alt, _ = alt_den.resolve(rtype, index)
                    rec["floor_fraction"] = min(rec.get("floor_fraction", 1.0), orr.compare(ref, alt, fmt, REL, ABS, layout=layout)[0])
                    rec["floor_outliers"] = max(rec.get("floor_outliers", 0), orr.outliers(ref, alt, fmt, REL, ABS, MAX_EXCESS, layout=layout)[0])
                # held to the floor where the floor is below the plain gate
                rec["min_fraction"] = min(MIN_FRACTION, rec["floor_fraction"])
                rec["outlier_budget"] = max(rec["outlier_budget"], rec["floor_outliers"])
            self.report.append(rec)

    def _frame(self, f, rect_fn):
        """(scene frame, CommonSettings, rectOrigin) of frame f.  rect_fn(f) -> (originX, originY, width, height): dynamic resolution,
        the scene is rendered at the rect size into textures of the context's (resource) size."""
        if rect_fn is None:
            fr = self._scene_frame(self.scene, f)
            return fr, harness.make_common_settings(fr, self.w, self.h, f, common=self.common), (0, 0)
        ox, oy, rw, rh = rect_fn(f)
        prev = rect_fn(f - 1) if f > 0 else (ox, oy, rw, rh)
        if (rw, rh) not in self._scenes:
            self._scenes[(rw, rh)] = scene.Scene(rw, rh, device=_scene_device(rw, rh, 0))
        fr = self._scene_frame(self._scenes[(rw, rh)], f)
        common = dict(self.common or {})
        common.update(resourceSize=(self.w, self.h), resourceSizePrev=(self.w, self.h), rectSizePrev=(prev[2], prev[3]), rectOrigin=(ox, oy))
        return fr, harness.make_common_settings(fr, rw, rh, f, common=common), (ox, oy)

    def run_per_pass(self, frames, first_frame=0, warmup=0, rect_fn=None):
        """Hard gate.  Returns the list of per-(frame, pass, output) comparison records.  `warmup` frames are run by the oracle
        alone first (histories long enough for the steady-state branches); the kernels start from the oracle's state anyway."""
        self._scenes = {}
        if rect_fn is not None:
            return self._run_per_pass_rects(frames, rect_fn)
        for f in range(first_frame, first_frame + warmup):
            fr = self._scene_frame(self.scene, f)
            self.cpu.set_inputs(fr)
            self.cpu.denoise(harness.make_common_settings(fr, self.w, self.h, f, common=self.common))
            if f == first_frame:
                self.cpu.set_inputs(fr)
        first_frame += warmup
        for f in range(first_frame, first_frame + frames):
            fr = self._scene_frame(self.scene, f)
            self.cpu.set_inputs(fr)
            cs = harness.make_common_settings(fr, self.w, self.h, f, common=self.common)
            self.instance.set_common_settings(cs)
            r, raw, n = self.instance.get_compute_dispatches_raw([self.identifier])
            assert r == nrd.Result.SUCCESS
            pipelines = self.instance.get_instance_desc()["pipelines"]
            # the frame's inputs are on the device before its first pass, like in an application: REBLUR ClassifyTiles decodes
            # IN_NORMAL_ROUGHNESS into the executor's guide surface although its DispatchDesc only binds IN_VIEWZ
            for name, arr in self.cpu.user.items():
                if name.startswith("IN_"):
                    self.ctx.upload(getattr(nrd.ResourceType, name), 0, np.ascontiguousarray(arr))
            for i in range(n):
                d = nrd.Dispatch(raw[i], pipelines)
                self._sync_to_gpu(d)
                floor = self.cpu_alt and self._has_floor(d)
                if floor:
                    for alt_den in self.cpu_alt:
                        for _, rtype, index in d.resources:
                            alt_den.resolve(rtype, index)[0][...] = self.cpu.resolve(rtype, index)[0]
                self.ctx.execute_raw(C.byref(raw[i]))
                self.torch.cuda.synchronize()
                self._cpu_run(d)
                if floor:
                    for alt_den in self.cpu_alt:
                        alt_den.run_dispatch(d)
                self._compare_outputs(f, d)
            if f == 0:
                self.cpu.set_inputs(fr)  # the frame-0 clears also zero IN_MV (reference quirk), restore it
        return self.report

    def _run_per_pass_rects(self, frames, rect_fn):
        for f in range(frames):
            fr, cs, origin = self._frame(f, rect_fn)
            for c in [self.cpu] + self.cpu_alt:
                c.rect_origin = origin
            self.cpu.set_inputs(fr, rect_origin=origin)
            self.instance.set_common_settings(cs)
            r, raw, n = self.instance.get_compute_dispatches_raw([self.identifier])
            assert r == nrd.Result.SUCCESS
            pipelines = self.instance.get_instance_desc()["pipelines"]
            for name, arr in self.cpu.user.items():
                if name.startswith("IN_"):
                    self.ctx.upload(getattr(nrd.ResourceType, name), 0, np.ascontiguousarray(arr))
            for i in range(n):
                d = nrd.Dispatch(raw[i], pipelines)
                self._sync_to_gpu(d)
                self.ctx.execute_raw(C.byref(raw[i]))
                self.torch.cuda.synchronize()
                self._cpu_run(d)
                self._compare_outputs(f, d)
            if f == 0:
                self.cpu.set_inputs(fr, rect_origin=origin)  # the frame-0 clears also zero IN_MV (reference quirk), restore it
        return self.report

    def failures(self):
        return [r for r in self.report if r["fraction"] < r["min_fraction"] or r["outliers"] > r["outlier_budget"] or r["nonfinite"]]

    def describe_failures(self, limit=40):
        return "\n".join("f%d %s %s %s frac=%.5f (gate %.5f) worst=%.1f outliers=%d/%d nonfinite=%d" % (
            r["frame"], r["shader"], r["resource"], r["format"], r["fraction"], r["min_fraction"], r["worst"], r["outliers"], r["outlier_budget"], r["nonfinite"])
                         for r in self.failures()[:limit])


def outlier_budget(texels):
    return max(OUTLIER_FLOOR, int(OUTLIER_BUDGET * texels))


def run_sequence(denoiser, width, height, frames, settings=None, device=0, noise_floor=False):
    """Statistical gate: independent end-to-end runs; returns {output name: (fraction within tolerance, PSNR dB)}.
    noise_floor=True additionally runs the FMA-contracted build of the oracle on the same frames and returns
    {name: (fraction, PSNR, floor fraction)}: `floor` is how far two IEEE-legal CPU evaluations of the same math drift apart --
    the chains are chaotic (step functions on noisy data feed back through the history), so this, not 100 %, is the yardstick."""
    import torch
    sc = scene.Scene(width, height, device=_scene_device(width, height, device))
    cpu = orr.CpuDenoiser(denoiser, width, height, settings=settings)
    cpu_fma = orr.CpuDenoiser(denoiser, width, height, settings=settings, variant="fma") if noise_floor else None
    gpu = harness.GpuDenoiser(denoiser, width, height, device=device, settings=settings)
    for f in range(frames):
        fr = sc.frame(f, harness.radiance_mode(denoiser))
        cs = harness.make_common_settings(fr, width, height, f)
        for c in (cpu, cpu_fma):
            if c is not None:
                c.set_inputs(fr)
                c.denoise(cs)
                if f == 0:
                    c.set_inputs(fr)
        gpu.set_inputs(fr)
        gpu.denoise(cs)
    torch.cuda.synchronize()
    out = {}
    for name, t in gpu.outputs().items():
        ref = cpu.user[name]
        got = t.cpu().numpy().view(ref.dtype).reshape(ref.shape)
        frac, _ = orr.compare(ref, got, cpu.user_fmt[name], REL, ABS)
        assert np.isfinite(got.astype(np.float64)).all() or not np.isfinite(ref.astype(np.float64)).all(), "non-finite texels in " + name
        a, b = ref.astype(np.float64), got.astype(np.float64)
        mse = float(((a - b) ** 2).mean())
        peak = float(max(np.abs(a).max(), 1e-6))
        psnr = 10.0 * np.log10(peak * peak / mse) if mse > 0 else 200.0
        out[name] = (frac, psnr)
        if cpu_fma is not None:
            out[name] = (frac, psnr, orr.compare(ref, cpu_fma.user[name], cpu.user_fmt[name], REL, ABS)[0])
    gpu.destroy()
    return out
