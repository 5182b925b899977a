#!/usr/bin/env python
"""TEST INFRASTRUCTURE.  Compiles the reference's OWN compute-shader sources for the CPU, from where they lie under
/root/reference/Shaders, into oracle/_ref/shaders/<pass>.so -- so that the oracle's restatement of a pass can be checked against
the code it restates (tests/test_reference_shaders.py).  No reference source is copied into the repository; the only outputs are
the shared objects (and the generated vector header) under the git-ignored oracle/_ref/.

Recipe per pass (one translation unit each; constants / resources / groupshared memory are globals of the shader):
  1. gcc -E -P -x c -undef -nostdinc            the C preprocessor resolves the shader's #includes and macros where they lie
        -include oracle/refshader/nrd_macros.h   (NRD.hlsli's "custom engine" resource macros, entry point name)
        -I oracle/refshader                      ("ml.hlsli": MathLib is an external dependency absent from /root/reference)
  2. fix_hlsl()                                  the HLSL constructs that are not C++ *syntax*, patched in the stream:
        [numthreads] / [unroll] / ... attributes, ": SV_*" semantics, out / inout parameters -> references,
        float literals get an f suffix (HLSL literals are float, C++ ones double), groupshared -> static
  3. g++ -x c++ -include oracle/refshader/hlsl_cpp.h -shared     HLSL language semantics as a C++ header (vectors with swizzles,
        intrinsics, textures on the oracle's hlsl::Tex, thread groups with barriers)
The shader math itself is compiled untouched.  What is NOT the reference here: MathLib (restated, oracle/mathlib.h), the texture
unit (oracle/hlsl.h) and the float evaluation of the C++ compiler (no FMA contraction, IEEE division / sqrt).

usage: python oracle/build_refshaders.py [pass ...]      (needs /root/reference: this container only; oracle/_ref/ travels)"""
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("NRD_REFERENCE", "/root/reference")
SHIM = os.path.join(ROOT, "oracle", "refshader")
OUT = os.path.join(ROOT, "oracle", "_ref", "shaders")
GEN = os.path.join(ROOT, "oracle", "_ref", "refshader")

def pass_list():
    """Every pass shader of the denoisers the product supports (PipelineDesc::shaderFileName minus ".cs"), from the shader
    sources that exist.  Not built: Clear_* (trivial) and *_Validation (debug overlay, needs MathLib's text renderer)."""
    out = []
    for f in sorted(os.listdir(os.path.join(REF, "Shaders", "Source"))):
        if not f.endswith(".cs.hlsl"):
            continue
        n = f[:-len(".cs.hlsl")]
        if n.startswith("Clear_") or n.endswith("_Validation"):
            continue
        if any(k in n for k in ("Occlusion", "Sh_", "DirectionalOcclusion")):  # denoisers the product does not implement
            continue
        if n.startswith(("REBLUR_", "RELAX_", "SIGMA_", "REFERENCE_")):
            out.append(n)
    return out


ENTRY = """
} // namespace refshader (opened by oracle/refshader/hlsl_cpp.h)
extern "C" __attribute__((visibility("default"))) int refshader_dispatch(const void* constants, int constantsSize, const OracleTexture* textures, int texturesNum, int gridW, int gridH)
{
    return refshader::RefShaderDispatchC(refshader::refshader_main, REFSHADER_NUMTHREADS_X, REFSHADER_NUMTHREADS_Y, constants, constantsSize, textures, texturesNum, gridW, gridH);
}
"""

FLOAT_LITERAL = re.compile(r"(?<![\w.])((?:\d+\.\d*|\.\d+)(?:[eE][-+]?\d+)?|\d+[eE][-+]?\d+)(?![\w.])")
ATTRIBUTE = re.compile(r"\[\s*(?:unroll|loop|branch|flatten|fastopt|allow_uav_condition|numthreads)\s*(?:\([^\]]*\))?\s*\]")
SEMANTIC = re.compile(r":\s*SV_\w+")
OUT_PARAM = re.compile(r"\b(?:inout|out)\s+((?:const\s+)?[A-Za-z_]\w*)\s+(?=[A-Za-z_])")
IN_PARAM = re.compile(r"([(,]\s*)in\s+(?=[A-Za-z_]\w*\s+[A-Za-z_])")


def fix_hlsl(text):
    text = ATTRIBUTE.sub("", text)
    text = SEMANTIC.sub("", text)
    text = OUT_PARAM.sub(r"\1& ", text)
    text = IN_PARAM.sub(r"\1", text)
    text = FLOAT_LITERAL.sub(r"\1f", text)
    text = re.sub(r"\bgroupshared\b", "static", text)
    # a vector initialised from a texture fetch: HLSL replicates a one-channel fetch (float2 data = gIn_Penumbra[ pixelPos ];),
    # a vector fetch is taken as it is (hlsl_cpp.h _fetch_init)
    text = re.sub(r"\b(float[234])\s+(\w+)\s*=\s*(gIn_\w+\s*\[[^\]]*\])\s*;", r"\1 \2 = _fetch_init<\1>(\3);", text)
    # x.xxx on a scalar (HLSL: float3(x)) -- also harmless on a vector
    text = re.sub(r"((?<![\w.])\d[\d.]*(?:[eE][-+]?\d+)?f)\s*\.(x{2,4})\b", r"_splat_\2(\1)", text)
    text = re.sub(r"(?<![\w.\])])([A-Za-z_]\w*)\.(x{2,4})\b", r"_splat_\2(\1)", text)
    # NAME.x where NAME may be a scalar variable (REBLUR_FAST_TYPE)
    text = re.sub(r"(?<![\w.\])])([A-Za-z_]\w*)\.x\b(?!\s*\()", r"_comp_x(\1)", text)
    return text


def build(name, keep_source=False):
    os.makedirs(OUT, exist_ok=True)
    os.makedirs(GEN, exist_ok=True)
    gen = os.path.join(GEN, "hlsl_vec_gen.h")
    if not os.path.exists(gen) or os.path.getmtime(gen) < os.path.getmtime(os.path.join(SHIM, "gen_vec.py")):
        with open(gen, "w") as f:
            subprocess.run([sys.executable, os.path.join(SHIM, "gen_vec.py")], stdout=f, check=True)
    src = os.path.join(REF, "Shaders", "Source", name + ".cs.hlsl")
    wrapper = '#include "%s"\n%s' % (src, ENTRY)
    cpp = subprocess.run(["gcc", "-E", "-P", "-x", "c", "-undef", "-nostdinc", "-include", os.path.join(SHIM, "nrd_macros.h"), "-I", SHIM,
                          "-I", os.path.join(REF, "Shaders", "Include"), "-I", os.path.join(REF, "Shaders", "Resources"),
                          "-DNRD_NORMAL_ENCODING=2", "-DNRD_ROUGHNESS_ENCODING=1", "-"], input=wrapper, capture_output=True, text=True)
    if cpp.returncode != 0:
        raise RuntimeError("preprocessing %s failed:\n%s" % (name, cpp.stderr[-4000:]))
    # the group size is what the entry point's [numthreads( x, y, 1 )] says (macros are expanded by now)
    m = re.search(r"\[\s*numthreads\s*\(([^,\]]+),([^,\]]+),", cpp.stdout)
    if not m:
        raise RuntimeError("no [numthreads] in " + name)
    text = fix_hlsl(cpp.stdout).replace("REFSHADER_NUMTHREADS_X", "(" + m.group(1).strip() + ")").replace("REFSHADER_NUMTHREADS_Y", "(" + m.group(2).strip() + ")")
    if keep_source:  # debugging aid only: the stream is reference text, it must stay under the git-ignored oracle/_ref/
        with open(os.path.join(OUT, name + ".ii"), "w") as f:
            f.write(text)
    so = os.path.join(OUT, name + ".so")
    cxx = subprocess.run(["g++", "-x", "c++", "-std=c++17", "-O1", "-fPIC", "-shared", "-w", "-ffp-contract=off", "-fvisibility=hidden", "-mavx2", "-mf16c",
                          "-include", os.path.join(SHIM, "hlsl_cpp.h"), "-I", GEN, "-o", so, "-"], input=text, capture_output=True, text=True)
    if cxx.returncode != 0:
        with open("/tmp/refshader_errors.txt", "w") as f:
            f.write(cxx.stderr)
        raise RuntimeError("compiling %s failed (full log: /tmp/refshader_errors.txt):\n%s" % (name, cxx.stderr[:3000]))
    return so


FRONTEND_PRELUDE = """
// tests/frontend_probe.cpp is written against include/nrd_b200_frontend.cuh; the same text is compiled here against the reference's
// NRD.hlsli: these few names map the probe's helpers onto HLSL
inline float3 f3(float x, float y, float z) { return float3(x, y, z); }
inline float4 f4(float x, float y, float z, float w) { return float4(x, y, z, w); }
inline float3 normalize3(float3 v) { return normalize(v); }
typedef uint uint32_t;
inline uint nrdPackR10G10B10A2(float4 p)
{
    uint8_t texel[4];
    hlsl::Tex t; t.data = texel; t.w = t.h = 1; t.pitch = 4; t.fmt = hlsl::R10_G10_B10_A2_UNORM;
    t.store(0, 0, O(p));
    uint v;
    memcpy(&v, texel, 4);
    return v;
}
inline float4 nrdUnpackR10G10B10A2(uint v)
{
    uint8_t texel[4];
    memcpy(texel, &v, 4);
    hlsl::Tex t; t.data = texel; t.w = t.h = 1; t.pitch = 4; t.fmt = hlsl::R10_G10_B10_A2_UNORM;
    return S(t.load(0, 0));
}
"""


def build_frontend_probe():
    """tests/frontend_probe.cpp (the probe of include/nrd_b200_frontend.cuh) compiled a second time -- against the reference's own
    NRD.hlsli through the shim -- into oracle/_ref/shaders/frontend_probe_ref: same inputs, same columns, reference code."""
    os.makedirs(OUT, exist_ok=True)
    probe = open(os.path.join(ROOT, "tests", "frontend_probe.cpp")).read()
    body = probe[probe.index("static unsigned lcg"):].replace("int main()", "int probe_main()")
    wrapper = '#include "%s"\n%s\n%s\n}\nint main() { return refshader::probe_main(); }\n' % (os.path.join(REF, "Shaders", "Include", "NRD.hlsli"), FRONTEND_PRELUDE, body)
    cpp = subprocess.run(["gcc", "-E", "-P", "-x", "c", "-undef", "-nostdinc", "-include", os.path.join(SHIM, "nrd_macros.h"), "-I", SHIM,
                          "-I", os.path.join(REF, "Shaders", "Include"), "-DNRD_NORMAL_ENCODING=2", "-DNRD_ROUGHNESS_ENCODING=1", "-"], input=wrapper, capture_output=True, text=True)
    if cpp.returncode != 0:
        raise RuntimeError("preprocessing the front-end probe failed:\n%s" % cpp.stderr[-3000:])
    exe = os.path.join(OUT, "frontend_probe_ref")
    cxx = subprocess.run(["g++", "-x", "c++", "-std=c++17", "-O1", "-w", "-ffp-contract=off", "-mavx2", "-mf16c", "-include", os.path.join(SHIM, "hlsl_cpp.h"), "-I", GEN, "-o", exe, "-"],
                         input=fix_hlsl(cpp.stdout), capture_output=True, text=True)
    if cxx.returncode != 0:
        raise RuntimeError("compiling the front-end probe failed:\n%s" % cxx.stderr[:4000])
    return exe


def _stamp():
    import hashlib
    h = hashlib.sha1()
    for f in sorted(os.listdir(SHIM)) + ["../hlsl.h", "../mathlib.h", "../oracle.h", "../build_refshaders.py", "../../tests/frontend_probe.cpp"]:
        path = os.path.join(SHIM, f)
        if os.path.isfile(path):
            h.update(open(path, "rb").read())
    return h.hexdigest()


def build_all(names=None, keep_source=False, force=False):
    """Builds the shaders whose .so is missing or older than the shim (a stamp file records the shim's hash)."""
    if not os.path.isdir(os.path.join(REF, "Shaders", "Source")):
        return []  # the GPU box: only the prebuilt oracle/_ref/shaders/*.so exist
    import concurrent.futures
    os.makedirs(OUT, exist_ok=True)
    stamp_path, stamp = os.path.join(OUT, "shim.stamp"), _stamp()
    fresh = os.path.exists(stamp_path) and open(stamp_path).read() == stamp
    names = names or pass_list()
    todo = [n for n in names if force or not fresh or not os.path.exists(os.path.join(OUT, n + ".so"))]
    if todo:
        build(todo[0], keep_source)  # generates the vector header once, before the parallel part
        with concurrent.futures.ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
            for fut in [ex.submit(build, n, keep_source) for n in todo[1:]]:
                fut.result()
    if todo or not os.path.exists(os.path.join(OUT, "frontend_probe_ref")):
        build_frontend_probe()
    if todo:
        with open(stamp_path, "w") as f:
            f.write(stamp)
    return [os.path.join(OUT, n + ".so") for n in names]


if __name__ == "__main__":
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    for so in build_all(args or None, "--keep" in sys.argv, "--force" in sys.argv or bool(args)):
        print(so)
