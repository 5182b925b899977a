// TEST INFRASTRUCTURE ONLY -- never linked into, imported by or called from the product library.
//
// A C++ environment in which the reference's OWN shader sources (/root/reference/Shaders/Source/*.cs.hlsl with everything they
// include) compile with g++ and run on the CPU, one thread-group at a time.  oracle/build_refshaders.py preprocesses a shader where
// it lies, patches the handful of HLSL constructs that are not C++ syntax (attributes, out / inout, semantics, float literals) on
// the fly and compiles the stream against this header into oracle/_ref/shaders/<pass>.so; no reference source is copied.
//
// What this header provides is HLSL *language* semantics only:
//   * vector types with real swizzle members (generated: oracle/refshader/gen_vec.py), matrices, scalar intrinsics;
//   * Texture2D / RWTexture2D / SamplerState on top of the oracle's hlsl::Tex (format decode / quantising stores, clamp samplers,
//     Gather order -- oracle/hlsl.h);
//   * thread groups with groupshared memory and GroupMemoryBarrierWithGroupSync (every thread of a group is a ucontext fiber);
//   * registration of the constants / inputs / outputs a shader declares through the NRD_CONSTANT / NRD_INPUT / NRD_OUTPUT macros
//     (NRD.hlsli's "custom engine" branch), so that one generic driver can bind any pass.
// The one NRD dependency that is absent from /root/reference -- MathLib's ml.hlsli -- is oracle/refshader/ml.hlsli: thin wrappers
// around the oracle's restatement (oracle/mathlib.h), so that a difference between a reference pass and the oracle's pass can only
// come from the pass body.
#pragma once
#include "../hlsl.h"
#include "../mathlib.h"

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ucontext.h>
#include <vector>

#include "../oracle.h"

// Everything below -- and the shader that follows this header in the translation unit -- lives in this namespace, so that the HLSL
// intrinsics hide the C library's global abs / floor / ... instead of overloading them (closed by the epilogue build_refshaders.py
// appends to the stream).
namespace refshader
{
typedef unsigned int uint;

// ---- scalar intrinsics (the float ones forward to the oracle's so that NaN rules etc. are the same) --------------------------
inline float saturate(float x) { return hlsl::saturate(x); }
inline float lerp(float a, float b, float t) { return hlsl::lerp(a, b, t); }
inline float step(float a, float x) { return hlsl::step(a, x); }
inline float rcp(float x) { return hlsl::rcp(x); }
inline float rsqrt(float x) { return hlsl::rsqrt(x); }
inline float frac(float x) { return hlsl::frac(x); }
inline float min(float a, float b) { return hlsl::min(a, b); }
inline float max(float a, float b) { return hlsl::max(a, b); }
inline float clamp(float x, float a, float b) { return hlsl::clamp(x, a, b); }
inline float abs(float a) { return hlsl::abs(a); }
inline float sqrt(float a) { return hlsl::sqrt(a); }
inline float floor(float a) { return hlsl::floor(a); }
inline float ceil(float a) { return std::ceil(a); }
inline float exp2(float a) { return hlsl::exp2(a); }
inline float exp(float a) { return hlsl::exp(a); }
inline float log(float a) { return hlsl::log(a); }
inline float log2(float a) { return std::log2(a); }
inline float pow(float a, float b) { return hlsl::pow(a, b); }
inline float atan(float a) { return hlsl::atan(a); }
inline float sign(float a) { return hlsl::sign(a); }
inline float sin(float a) { return std::sin(a); }
inline float cos(float a) { return std::cos(a); }
inline float tan(float a) { return std::tan(a); }
inline float acos(float a) { return std::acos(a); }
inline float asin(float a) { return std::asin(a); }
inline float atan2(float a, float b) { return std::atan2(a, b); }
inline float fmod(float a, float b) { return std::fmod(a, b); }
inline float round(float a) { return std::nearbyint(a); } // HLSL round: to nearest even
inline float trunc(float a) { return std::trunc(a); }
inline bool isnan(float a) { return a != a; }
inline bool isinf(float a) { return std::fabs(a) == INFINITY; }
inline float mad(float a, float b, float c) { return a * b + c; }
inline float smoothstep(float a, float b, float x) { float t = saturate((x - a) / (b - a)); return t * t * (3.0f - 2.0f * t); }
inline float dot(float a, float b) { return a * b; }
inline float length(float a) { return std::fabs(a); }
inline bool any(bool a) { return a; }
inline bool all(bool a) { return a; }
inline bool any(float a) { return a != 0.0f; }
inline int min(int a, int b) { return a < b ? a : b; }
inline int max(int a, int b) { return a > b ? a : b; }
inline uint min(uint a, uint b) { return a < b ? a : b; }
inline uint max(uint a, uint b) { return a > b ? a : b; }
inline int min(int a, uint b) { return a < (int)b ? a : (int)b; }
inline int max(int a, uint b) { return a > (int)b ? a : (int)b; }
inline int min(uint a, int b) { return (int)a < b ? (int)a : b; }
inline int max(uint a, int b) { return (int)a > b ? (int)a : b; }
inline float min(float a, int b) { return min(a, (float)b); }
inline float max(float a, int b) { return max(a, (float)b); }
inline float min(int a, float b) { return min((float)a, b); }
inline float max(int a, float b) { return max((float)a, b); }
inline float min(float a, uint b) { return min(a, (float)b); }
inline float max(float a, uint b) { return max(a, (float)b); }
inline int clamp(int x, int a, int b) { return min(max(x, a), b); }
inline uint clamp(uint x, uint a, uint b) { return min(max(x, a), b); }
inline int abs(int a) { return a < 0 ? -a : a; }
inline uint asuint(float f) { return hlsl::asuint(f); }
inline uint asuint(uint u) { return u; }
inline float asfloat(uint u) { return hlsl::asfloat(u); }
inline uint f32tof16(float f) { return hlsl::f32tof16(f); }
inline float f16tof32(uint h) { return hlsl::f16tof32((uint16_t)h); }
inline uint firstbithigh(uint v) { return v ? 31u - (uint)__builtin_clz(v) : 0xFFFFFFFFu; }
inline uint countbits(uint v) { return (uint)__builtin_popcount(v); }
inline uint reversebits(uint v) { uint r = 0; for (int i = 0; i < 32; i++) r |= ((v >> i) & 1u) << (31 - i); return r; }

#include "hlsl_vec_gen.h"

// scalar "swizzles" (x.xxx on a float is HLSL for float3(x)): build_refshaders.py rewrites NAME.xx / .xxx / .xxxx into these calls
#define REFSHADER_SPLAT(T) \
    inline T##2 _splat_xx(T a) { return T##2(a); } \
    inline T##3 _splat_xxx(T a) { return T##3(a); } \
    inline T##4 _splat_xxxx(T a) { return T##4(a); } \
    inline T##2 _splat_xx(const T##2& a) { return a.xx; } \
    inline T##3 _splat_xxx(const T##2& a) { return a.xxx; } \
    inline T##4 _splat_xxxx(const T##2& a) { return a.xxxx; } \
    inline T##2 _splat_xx(const T##3& a) { return a.xx; } \
    inline T##3 _splat_xxx(const T##3& a) { return a.xxx; } \
    inline T##4 _splat_xxxx(const T##3& a) { return a.xxxx; } \
    inline T##2 _splat_xx(const T##4& a) { return a.xx; } \
    inline T##3 _splat_xxx(const T##4& a) { return a.xxx; } \
    inline T##4 _splat_xxxx(const T##4& a) { return a.xxxx; }
REFSHADER_SPLAT(float) REFSHADER_SPLAT(int) REFSHADER_SPLAT(uint)
// NAME.x on a scalar variable (REBLUR_FAST_TYPE is float): build_refshaders.py rewrites NAME.x into _comp_x(NAME), an lvalue
template <class V> inline auto _comp_x(V& a) -> decltype((a.x)) { return a.x; }
template <class V> inline auto _comp_x(const V& a) -> decltype((a.x)) { return a.x; }
inline float& _comp_x(float& a) { return a; }
inline const float& _comp_x(const float& a) { return a; }
inline int& _comp_x(int& a) { return a; }
inline const int& _comp_x(const int& a) { return a; }
inline uint& _comp_x(uint& a) { return a; }
inline const uint& _comp_x(const uint& a) { return a; }
// mixed scalar arguments (clamp( x, 0, 65504.0 ) ...): everything is evaluated in float like HLSL does
template <class A, class B> inline float clamp(float x, A a, B b) { return clamp(x, (float)a, (float)b); }

// ---- conversions between these types and the oracle's (namespace hlsl) ----------------------------------------------------------
inline hlsl::float2 O(const float2& a) { return hlsl::float2(a.x, a.y); }
inline hlsl::float3 O(const float3& a) { return hlsl::float3(a.x, a.y, a.z); }
inline hlsl::float4 O(const float4& a) { return hlsl::float4(a.x, a.y, a.z, a.w); }
inline hlsl::int2 O(const int2& a) { return hlsl::int2(a.x, a.y); }
inline float2 S(const hlsl::float2& a) { return float2(a.x, a.y); }
inline float3 S(const hlsl::float3& a) { return float3(a.x, a.y, a.z); }
inline float4 S(const hlsl::float4& a) { return float4(a.x, a.y, a.z, a.w); }

// ---- matrices (column-major storage like the oracle's: c[k] is column k, mul(M, v) = sum c[k] * v[k]) ---------------------------
struct float4x4
{
    float4 c[4];
};
inline hlsl::float4x4 O(const float4x4& m)
{
    hlsl::float4x4 r;
    for (int i = 0; i < 4; i++) r.c[i] = O(m.c[i]);
    return r;
}
inline float4 mul(const float4x4& m, const float4& v) { return S(hlsl::mul(O(m), O(v))); }
struct float3x3 // rows, as float3x3( T, B, N ) builds them
{
    float3 r[3];
    float3x3() {}
    float3x3(const float3& a, const float3& b, const float3& c) { r[0] = a; r[1] = b; r[2] = c; }
    float3x3(float a, float b, float c, float d, float e, float f, float g, float h, float i) { r[0] = float3(a, b, c); r[1] = float3(d, e, f); r[2] = float3(g, h, i); }
    float3& operator[](int i) { return r[i]; }
    const float3& operator[](int i) const { return r[i]; }
};
inline float3 mul(const float3x3& m, const float3& v) { return float3(dot(m.r[0], v), dot(m.r[1], v), dot(m.r[2], v)); }
inline float3 mul(const float3& v, const float3x3& m) { return m.r[0] * v.x + m.r[1] * v.y + m.r[2] * v.z; }
inline float3x3 transpose(const float3x3& m)
{
    return float3x3(float3(m.r[0].x, m.r[1].x, m.r[2].x), float3(m.r[0].y, m.r[1].y, m.r[2].y), float3(m.r[0].z, m.r[1].z, m.r[2].z));
}
inline float3x3 S(const hlsl::float3x3& m) { return float3x3(S(m.r[0]), S(m.r[1]), S(m.r[2])); }
inline hlsl::float3x3 O(const float3x3& m)
{
    hlsl::float3x3 r;
    for (int i = 0; i < 3; i++) r.r[i] = O(m.r[i]);
    return r;
}
struct float2x3
{
    float3 r[2];
    float2x3() {}
    float2x3(const float3& a, const float3& b) { r[0] = a; r[1] = b; }
    float3& operator[](int i) { return r[i]; }
    const float3& operator[](int i) const { return r[i]; }
};
struct float2x2
{
    float2 r[2];
    float2x2() {}
    float2x2(const float2& a, const float2& b) { r[0] = a; r[1] = b; }
    float2x2(float a, float b, float c, float d) { r[0] = float2(a, b); r[1] = float2(c, d); }
    float2& operator[](int i) { return r[i]; }
    const float2& operator[](int i) const { return r[i]; }
};
inline float2 mul(const float2x2& m, const float2& v) { return float2(dot(m.r[0], v), dot(m.r[1], v)); }

// ---- resources ---------------------------------------------------------------------------------------------------------------------
struct SamplerState
{
    int linear; // register s0 = gNearestClamp, s1 = gLinearClamp (NRD.hlsli NRD_SAMPLERS)
};
// a one-channel texel: HLSL allows .x / .r on a scalar
struct float1
{
    union { float x; float r; };
    float1() : x(0.0f) {}
    explicit float1(float v) : x(v) {}
    operator float() const { return x; }
};
// floatN x = gIn_T[ p ]; build_refshaders.py rewrites the initialiser into _fetch_init<floatN>( gIn_T[ p ] ): a one-channel fetch
// (float1) is replicated like HLSL does, a vector fetch initialises the vector as it is
template <class V> inline V _fetch_init(const float1& a) { return V(float(a)); }
template <class V, class T> inline V _fetch_init(const T& a) { return V(a); }
template <class T> struct TexelOf;
struct TexelGatherFloat
{
    typedef float4 G;
    static float4 gather(const hlsl::Tex& t, const float2& uv, int ch, const int2& offset) { return S(t.gather(O(uv), ch, O(offset))); }
};
struct TexelGatherUint
{
    typedef uint4 G;
    static uint4 gather(const hlsl::Tex& t, const float2& uv, int, const int2& offset)
    {
        hlsl::uint4 v = t.gatheru(O(uv), O(offset));
        return uint4(v.x, v.y, v.z, v.w);
    }
};
template <> struct TexelOf<float> : TexelGatherFloat { typedef float1 R; static float from(const hlsl::Tex& t, int x, int y) { return t.load(x, y).x; } static void to(hlsl::Tex& t, int x, int y, float v) { t.store(x, y, hlsl::float4(v, 0, 0, 0)); } static float cv(const hlsl::float4& v) { return v.x; } };
template <> struct TexelOf<float2> : TexelGatherFloat { typedef float2 R; static float2 from(const hlsl::Tex& t, int x, int y) { hlsl::float4 v = t.load(x, y); return float2(v.x, v.y); } static void to(hlsl::Tex& t, int x, int y, const float2& v) { t.store(x, y, hlsl::float4(v.x, v.y, 0, 0)); } static float2 cv(const hlsl::float4& v) { return float2(v.x, v.y); } };
template <> struct TexelOf<float3> : TexelGatherFloat { typedef float3 R; static float3 from(const hlsl::Tex& t, int x, int y) { hlsl::float4 v = t.load(x, y); return float3(v.x, v.y, v.z); } static void to(hlsl::Tex& t, int x, int y, const float3& v) { t.store(x, y, hlsl::float4(v.x, v.y, v.z, 0)); } static float3 cv(const hlsl::float4& v) { return float3(v.x, v.y, v.z); } };
template <> struct TexelOf<float4> : TexelGatherFloat { typedef float4 R; static float4 from(const hlsl::Tex& t, int x, int y) { return S(t.load(x, y)); } static void to(hlsl::Tex& t, int x, int y, const float4& v) { t.store(x, y, O(v)); } static float4 cv(const hlsl::float4& v) { return S(v); } };
template <> struct TexelOf<uint> : TexelGatherUint { typedef uint R; static uint from(const hlsl::Tex& t, int x, int y) { return t.loadu(x, y); } static void to(hlsl::Tex& t, int x, int y, uint v) { t.storeu(x, y, v); } };

template <class T> struct Texture2D
{
    typedef typename TexelOf<T>::R R;
    hlsl::Tex* t = nullptr;
    R operator[](const int2& p) const { return R(TexelOf<T>::from(*t, p.x, p.y)); }
    R operator[](const uint2& p) const { return R(TexelOf<T>::from(*t, (int)p.x, (int)p.y)); }
    template <int... I> R operator[](const Swz<int, I...>& p) const { return (*this)[int2(p)]; }
    template <int... I> R operator[](const Swz<uint, I...>& p) const { return (*this)[uint2(p)]; }
    R Load(const int3& p) const { return R(TexelOf<T>::from(*t, p.x, p.y)); }
    R Load(const int3& p, const int2& offset) const { return R(TexelOf<T>::from(*t, p.x + offset.x, p.y + offset.y)); }
    R SampleLevel(SamplerState s, const float2& uv, float) const { return R(TexelOf<T>::cv(s.linear ? t->sampleLinear(O(uv)) : t->sampleNearest(O(uv)))); }
    // texel offsets of a nearest / linear sample = a uv shifted by whole texels
    R SampleLevel(SamplerState s, const float2& uv, float lod, const int2& offset) const { return SampleLevel(s, uv + float2(offset) / float2((float)t->w, (float)t->h), lod); }
    typedef typename TexelOf<T>::G G; // float4, or uint4 for a uint texture
    G GatherRed(SamplerState, const float2& uv) const { return TexelOf<T>::gather(*t, uv, 0, int2(0, 0)); }
    G GatherRed(SamplerState, const float2& uv, const int2& offset) const { return TexelOf<T>::gather(*t, uv, 0, offset); }
    G GatherRed(SamplerState, const float2& uv, const float2& offset) const { return TexelOf<T>::gather(*t, uv, 0, int2(offset)); }
    G GatherGreen(SamplerState, const float2& uv) const { return TexelOf<T>::gather(*t, uv, 1, int2(0, 0)); }
    G GatherBlue(SamplerState, const float2& uv) const { return TexelOf<T>::gather(*t, uv, 2, int2(0, 0)); }
    G GatherAlpha(SamplerState, const float2& uv) const { return TexelOf<T>::gather(*t, uv, 3, int2(0, 0)); }
    void GetDimensions(uint& w, uint& h) const { w = (uint)t->w; h = (uint)t->h; }
};
template <class T> struct RWTexture2D
{
    hlsl::Tex* t = nullptr;
    struct Ref
    {
        hlsl::Tex* t;
        int x, y;
        void operator=(const T& v) { TexelOf<T>::to(*t, x, y, v); }
        operator typename TexelOf<T>::R() const { return TexelOf<T>::from(*t, x, y); }
    };
    Ref operator[](const int2& p) { return Ref{t, p.x, p.y}; }
    Ref operator[](const uint2& p) { return Ref{t, (int)p.x, (int)p.y}; }
    template <int... I> Ref operator[](const Swz<int, I...>& p) { return (*this)[int2(p)]; }
    template <int... I> Ref operator[](const Swz<uint, I...>& p) { return (*this)[uint2(p)]; }
};

// ---- what a shader declares --------------------------------------------------------------------------------------------------------
struct RefShaderSlot
{
    void* ptr;
    int size;
    const char* name;
    int kind; // 0 constant, 1 input texture, 2 output texture
};
inline std::vector<RefShaderSlot>& RefShaderSlots()
{
    static std::vector<RefShaderSlot> slots;
    return slots;
}
struct RefShaderReg
{
    RefShaderReg(void* ptr, int size, const char* name, int kind) { RefShaderSlots().push_back(RefShaderSlot{ptr, size, name, kind}); }
};
template <class T> inline hlsl::Tex** RefShaderTexPtr(Texture2D<T>* t) { return &t->t; }
template <class T> inline hlsl::Tex** RefShaderTexPtr(RWTexture2D<T>* t) { return &t->t; }

// ---- thread groups -------------------------------------------------------------------------------------------------------------------
typedef void (*RefShaderMain)(int2 threadPos, uint2 groupPos, int2 pixelPos, uint threadIndex);  // NRD_CS_MAIN_ARGS (Common.hlsli)
typedef void (*RefShaderMain3)(uint2 threadPos, uint2 groupPos, uint threadIndex);                 // the tile classifiers
struct RefShaderGroup
{
    static const int kMaxThreads = 1024;
    static const size_t kStack = 512 * 1024;
    ucontext_t scheduler, fiber[kMaxThreads];
    bool done[kMaxThreads];
    char* stacks = nullptr;
    RefShaderMain entry = nullptr;
    RefShaderMain3 entry3 = nullptr;
    int gx = 0, gy = 0, groupX = 0, groupY = 0, current = -1;
};
inline RefShaderGroup& RefShaderCurrentGroup()
{
    static RefShaderGroup g;
    return g;
}
inline void RefShaderFiberBody(int index)
{
    RefShaderGroup& g = RefShaderCurrentGroup();
    const int tx = index % g.gx, ty = index / g.gx;
    if (g.entry) g.entry(int2(tx, ty), uint2((uint)g.groupX, (uint)g.groupY), int2(g.groupX * g.gx + tx, g.groupY * g.gy + ty), (uint)index);
    else g.entry3(uint2((uint)tx, (uint)ty), uint2((uint)g.groupX, (uint)g.groupY), (uint)index);
    g.done[index] = true;
    swapcontext(&g.fiber[index], &g.scheduler);
}
// every thread of the group arrives here (or has returned) before any continues: round-robin over the fibers
inline void GroupMemoryBarrierWithGroupSync()
{
    RefShaderGroup& g = RefShaderCurrentGroup();
    swapcontext(&g.fiber[g.current], &g.scheduler);
}
// The SIGMA tile classifier separates its phases with GroupMemoryBarrier() only: its 8x4 group is one warp, which executes in
// lockstep on the GPUs the shader was written for.  Fibers do not: the memory barrier is made an execution barrier as well.
inline void GroupMemoryBarrier() { GroupMemoryBarrierWithGroupSync(); }
// the fibers of a group run one at a time: atomics on groupshared memory are plain read-modify-writes
template <class A, class B> inline void InterlockedAdd(A& dst, B v) { dst += (A)v; }
template <class A, class B> inline void InterlockedAdd(A& dst, B v, A& original) { original = dst; dst += (A)v; }
inline void InterlockedOr(uint& dst, uint v) { dst |= v; }
inline void InterlockedAnd(uint& dst, uint v) { dst &= v; }
inline void InterlockedMax(uint& dst, uint v) { dst = dst > v ? dst : v; }
inline void InterlockedMin(uint& dst, uint v) { dst = dst < v ? dst : v; }
inline void RefShaderSetEntry(RefShaderMain e) { RefShaderCurrentGroup().entry = e; RefShaderCurrentGroup().entry3 = nullptr; }
inline void RefShaderSetEntry(RefShaderMain3 e) { RefShaderCurrentGroup().entry = nullptr; RefShaderCurrentGroup().entry3 = e; }
inline void RefShaderRunGroup(int gx, int gy, int groupX, int groupY)
{
    RefShaderGroup& g = RefShaderCurrentGroup();
    const int n = gx * gy;
    if (!g.stacks) g.stacks = (char*)malloc(RefShaderGroup::kStack * RefShaderGroup::kMaxThreads);
    g.gx = gx; g.gy = gy; g.groupX = groupX; g.groupY = groupY;
    for (int i = 0; i < n; i++)
    {
        g.done[i] = false;
        getcontext(&g.fiber[i]);
        g.fiber[i].uc_stack.ss_sp = g.stacks + RefShaderGroup::kStack * i;
        g.fiber[i].uc_stack.ss_size = RefShaderGroup::kStack;
        g.fiber[i].uc_link = &g.scheduler;
        makecontext(&g.fiber[i], (void (*)())RefShaderFiberBody, 1, i);
    }
    for (bool alive = true; alive;)
    {
        alive = false;
        for (int i = 0; i < n; i++)
            if (!g.done[i])
            {
                g.current = i;
                swapcontext(&g.scheduler, &g.fiber[i]);
                alive = alive || !g.done[i];
            }
    }
}

// One dispatch: constants are copied member by member in declaration order (the reference's host code fills a C++ struct generated
// from the same NRD_CONSTANT list, Source/InstanceImpl.h), textures are bound in declaration order (inputs, then outputs -- the
// order of DispatchDesc::resources).  Returns 0, or a negative number when the shader's declarations do not match the dispatch.
template <class Entry> inline int RefShaderDispatch(Entry entry, int gx, int gy, const void* constants, int constantsSize, hlsl::Tex* tex, int texNum, int gridW, int gridH)
{
    int offset = 0, texIndex = 0;
    for (const RefShaderSlot& s : RefShaderSlots())
        if (s.kind == 0)
        {
            if (offset + s.size > constantsSize) return -1;
            memcpy(s.ptr, (const char*)constants + offset, (size_t)s.size);
            offset += s.size;
        }
    if (offset != constantsSize) return -2;
    for (int kind = 1; kind <= 2; kind++)
        for (const RefShaderSlot& s : RefShaderSlots())
            if (s.kind == kind)
            {
                if (texIndex >= texNum) return -3;
                *(hlsl::Tex**)s.ptr = &tex[texIndex++];
            }
    if (texIndex != texNum) return -4;
    RefShaderSetEntry(entry);
    for (int y = 0; y < gridH; y++)
        for (int x = 0; x < gridW; x++) RefShaderRunGroup(gx, gy, x, y);
    return 0;
}

// C entry used by the generated refshader_dispatch of every pass: same texture descriptors as oracle_dispatch (oracle/oracle.h)
template <class Entry> inline int RefShaderDispatchC(Entry entry, int gx, int gy, const void* constants, int constantsSize, const OracleTexture* textures, int texturesNum, int gridW, int gridH)
{
    hlsl::Tex tex[32];
    if (texturesNum > 32) return -5;
    for (int i = 0; i < texturesNum; i++)
    {
        tex[i].data = (uint8_t*)textures[i].data;
        tex[i].w = textures[i].width;
        tex[i].h = textures[i].height;
        tex[i].pitch = textures[i].pitchBytes;
        tex[i].fmt = textures[i].format;
        tex[i].yoff = textures[i].firstRow;
        tex[i].ox = textures[i].originX;
        tex[i].oy = textures[i].originY;
    }
    return RefShaderDispatch(entry, gx, gy, constants, constantsSize, tex, texturesNum, gridW, gridH);
}
