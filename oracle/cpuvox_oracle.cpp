/*
 * cpuvox_oracle.cpp — TEST INFRASTRUCTURE ONLY (see cpuvox_oracle.h).
 *
 * CPU restatement of pipliz/cpuvox's raybuffer renderer. Every function cites the reference
 * file:line it follows (paths relative to /root/reference/Assets/). IEEE fp32 throughout, built with
 * -O2 -ffp-contract=off -fno-fast-math so no FMA contraction and no reassociation happens.
 *
 * PARITY UNPINNED: the reference has no tests/golden vectors and cannot be built here (C# on
 * UnityEngine + Burst, no dotnet/mono). This is a port of the source, not the shipping Burst
 * FloatMode.Fast binary. Unity.Mathematics / UnityEngine calls are restated from their documented
 * behaviour (SURVEY.md Appendix A).
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may load
 * this. The product library shares no code with it.
 */
#include "cpuvox_oracle.h"

#include <atomic>
#include <climits>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <thread>
#include <vector>

namespace {

// ---------------------------------------------------------------------------------------------
// Unity.Mathematics scalar semantics (Appendix A1)
// ---------------------------------------------------------------------------------------------
struct f2 { float x, y; };
struct f3 { float x, y, z; };
struct f4 { float x, y, z, w; };
struct i2 { int x, y; };

inline float m_lerp(float a, float b, float t) { return a + t * (b - a); }
inline float m_unlerp(float a, float b, float x) { return (x - a) / (b - a); }
inline f3 m_lerp3(f3 a, f3 b, float t) { return {m_lerp(a.x, b.x, t), m_lerp(a.y, b.y, t), m_lerp(a.z, b.z, t)}; }
inline float m_sign(float x) { return (float)((x > 0.0f ? 1 : 0) - (x < 0.0f ? 1 : 0)); }
// math.min / math.max as the reference build pins them (unity_shim.hpp: isnan(y) || x < y ? x : y): a NaN second operand gives the
// first, a tie (±0) gives the second
inline float m_min(float a, float b) { return (std::isnan(b) || a < b) ? a : b; }
inline float m_max(float a, float b) { return (std::isnan(b) || a > b) ? a : b; }
inline int i_min(int a, int b) { return a < b ? a : b; }
inline int i_max(int a, int b) { return a > b ? a : b; }
inline int i_clamp(int x, int a, int b) { return i_max(a, i_min(b, x)); }
// (int)float on x64 .NET/Burst is cvttss2si: out-of-range and NaN give 0x80000000.
inline int f2i(float f) {
    if (!(f >= -2147483648.0f && f < 2147483648.0f)) return INT_MIN;
    return (int)f;
}
// math.round / Mathf.RoundToInt: half-to-even (Appendix A1, A7).
inline float m_round(float x) { return rintf(x); }

const float FLOAT_EPSILON = 1.401298464324817e-45f; // C# float.Epsilon, the smallest denormal
const uint32_t SKYBOX = 0x191919FFu;                // ColorARGB32(25,25,25) bytes a,r,g,b (DrawSegmentRayJob.cs:702)

// column-major float4x4, mul(M, v) = c0*v.x + c1*v.y + c2*v.z + c3*v.w
struct m4 {
    float c[4][4]; // c[col][row]
};
inline f4 mul(const m4& m, f4 v) {
    f4 r;
    r.x = m.c[0][0] * v.x + m.c[1][0] * v.y + m.c[2][0] * v.z + m.c[3][0] * v.w;
    r.y = m.c[0][1] * v.x + m.c[1][1] * v.y + m.c[2][1] * v.z + m.c[3][1] * v.w;
    r.z = m.c[0][2] * v.x + m.c[1][2] * v.y + m.c[2][2] * v.z + m.c[3][2] * v.w;
    r.w = m.c[0][3] * v.x + m.c[1][3] * v.y + m.c[2][3] * v.z + m.c[3][3] * v.w;
    return r;
}
inline m4 mul(const m4& a, const m4& b) {
    m4 r;
    for (int j = 0; j < 4; j++) {
        f4 col = mul(a, f4{b.c[j][0], b.c[j][1], b.c[j][2], b.c[j][3]});
        r.c[j][0] = col.x; r.c[j][1] = col.y; r.c[j][2] = col.z; r.c[j][3] = col.w;
    }
    return r;
}
inline m4 m4_identity() {
    m4 r; memset(&r, 0, sizeof r);
    r.c[0][0] = r.c[1][1] = r.c[2][2] = r.c[3][3] = 1.0f;
    return r;
}
inline m4 m4_scale(float x, float y, float z) { m4 r = m4_identity(); r.c[0][0] = x; r.c[1][1] = y; r.c[2][2] = z; return r; }
inline m4 m4_translate(float x, float y, float z) { m4 r = m4_identity(); r.c[3][0] = x; r.c[3][1] = y; r.c[3][2] = z; return r; }
// General inverse by cofactors in fp32. Unity.Mathematics.inverse uses a different evaluation order;
// host-side only, stated as an assumption (not bit-identical to the package).
m4 m4_inverse(const m4& mm) {
    float m[16], inv[16];
    for (int j = 0; j < 4; j++) for (int i = 0; i < 4; i++) m[j * 4 + i] = mm.c[j][i];
    inv[0] = m[5] * m[10] * m[15] - m[5] * m[11] * m[14] - m[9] * m[6] * m[15] + m[9] * m[7] * m[14] + m[13] * m[6] * m[11] - m[13] * m[7] * m[10];
    inv[4] = -m[4] * m[10] * m[15] + m[4] * m[11] * m[14] + m[8] * m[6] * m[15] - m[8] * m[7] * m[14] - m[12] * m[6] * m[11] + m[12] * m[7] * m[10];
    inv[8] = m[4] * m[9] * m[15] - m[4] * m[11] * m[13] - m[8] * m[5] * m[15] + m[8] * m[7] * m[13] + m[12] * m[5] * m[11] - m[12] * m[7] * m[9];
    inv[12] = -m[4] * m[9] * m[14] + m[4] * m[10] * m[13] + m[8] * m[5] * m[14] - m[8] * m[6] * m[13] - m[12] * m[5] * m[10] + m[12] * m[6] * m[9];
    inv[1] = -m[1] * m[10] * m[15] + m[1] * m[11] * m[14] + m[9] * m[2] * m[15] - m[9] * m[3] * m[14] - m[13] * m[2] * m[11] + m[13] * m[3] * m[10];
    inv[5] = m[0] * m[10] * m[15] - m[0] * m[11] * m[14] - m[8] * m[2] * m[15] + m[8] * m[3] * m[14] + m[12] * m[2] * m[11] - m[12] * m[3] * m[10];
    inv[9] = -m[0] * m[9] * m[15] + m[0] * m[11] * m[13] + m[8] * m[1] * m[15] - m[8] * m[3] * m[13] - m[12] * m[1] * m[11] + m[12] * m[3] * m[9];
    inv[13] = m[0] * m[9] * m[14] - m[0] * m[10] * m[13] - m[8] * m[1] * m[14] + m[8] * m[2] * m[13] + m[12] * m[1] * m[10] - m[12] * m[2] * m[9];
    inv[2] = m[1] * m[6] * m[15] - m[1] * m[7] * m[14] - m[5] * m[2] * m[15] + m[5] * m[3] * m[14] + m[13] * m[2] * m[7] - m[13] * m[3] * m[6];
    inv[6] = -m[0] * m[6] * m[15] + m[0] * m[7] * m[14] + m[4] * m[2] * m[15] - m[4] * m[3] * m[14] - m[12] * m[2] * m[7] + m[12] * m[3] * m[6];
    inv[10] = m[0] * m[5] * m[15] - m[0] * m[7] * m[13] - m[4] * m[1] * m[15] + m[4] * m[3] * m[13] + m[12] * m[1] * m[7] - m[12] * m[3] * m[5];
    inv[14] = -m[0] * m[5] * m[14] + m[0] * m[6] * m[13] + m[4] * m[1] * m[14] - m[4] * m[2] * m[13] - m[12] * m[1] * m[6] + m[12] * m[2] * m[5];
    inv[3] = -m[1] * m[6] * m[11] + m[1] * m[7] * m[10] + m[5] * m[2] * m[11] - m[5] * m[3] * m[10] - m[9] * m[2] * m[7] + m[9] * m[3] * m[6];
    inv[7] = m[0] * m[6] * m[11] - m[0] * m[7] * m[10] - m[4] * m[2] * m[11] + m[4] * m[3] * m[10] + m[8] * m[2] * m[7] - m[8] * m[3] * m[6];
    inv[11] = -m[0] * m[5] * m[11] + m[0] * m[7] * m[9] + m[4] * m[1] * m[11] - m[4] * m[3] * m[9] - m[8] * m[1] * m[7] + m[8] * m[3] * m[5];
    inv[15] = m[0] * m[5] * m[10] - m[0] * m[6] * m[9] - m[4] * m[1] * m[10] + m[4] * m[2] * m[9] + m[8] * m[1] * m[6] - m[8] * m[2] * m[5];
    float det = m[0] * inv[0] + m[1] * inv[4] + m[2] * inv[8] + m[3] * inv[12];
    float rdet = 1.0f / det;
    m4 r;
    for (int j = 0; j < 4; j++) for (int i = 0; i < 4; i++) r.c[j][i] = inv[j * 4 + i] * rdet;
    return r;
}

// ---------------------------------------------------------------------------------------------
// UnityEngine restatements (Appendix A2-A9)
// ---------------------------------------------------------------------------------------------
const float DEG2RAD = 0.017453292f; // Mathf.Deg2Rad as a float constant

struct quat { float x, y, z, w; };
inline quat q_mul(quat a, quat b) {
    return {a.w * b.x + a.x * b.w + a.y * b.z - a.z * b.y,
            a.w * b.y + a.y * b.w + a.z * b.x - a.x * b.z,
            a.w * b.z + a.z * b.w + a.x * b.y - a.y * b.x,
            a.w * b.w - a.x * b.x - a.y * b.y - a.z * b.z};
}
// Quaternion * Vector3
inline f3 q_rot(quat q, f3 p) {
    float x2 = q.x * 2.0f, y2 = q.y * 2.0f, z2 = q.z * 2.0f;
    float xx = q.x * x2, yy = q.y * y2, zz = q.z * z2;
    float xy = q.x * y2, xz = q.x * z2, yz = q.y * z2;
    float wx = q.w * x2, wy = q.w * y2, wz = q.w * z2;
    f3 r;
    r.x = (1.0f - (yy + zz)) * p.x + (xy - wz) * p.y + (xz + wy) * p.z;
    r.y = (xy + wz) * p.x + (1.0f - (xx + zz)) * p.y + (yz - wx) * p.z;
    r.z = (xz - wy) * p.x + (yz + wx) * p.y + (1.0f - (xx + yy)) * p.z;
    return r;
}
// Quaternion.Euler(x,y,z): rotate z, then x, then y  =>  qY * qX * qZ (A9)
quat q_euler(float xd, float yd, float zd) {
    float hx = xd * DEG2RAD * 0.5f, hy = yd * DEG2RAD * 0.5f, hz = zd * DEG2RAD * 0.5f;
    quat qx = {(float)sin((double)hx), 0, 0, (float)cos((double)hx)};
    quat qy = {0, (float)sin((double)hy), 0, (float)cos((double)hy)};
    quat qz = {0, 0, (float)sin((double)hz), (float)cos((double)hz)};
    return q_mul(q_mul(qy, qx), qz);
}
inline f3 v_cross(f3 a, f3 b) { return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }
inline float v_dot(f3 a, f3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
inline f3 v_normalize(f3 a) {
    float l = sqrtf(v_dot(a, a));
    if (l > 1e-5f) return {a.x / l, a.y / l, a.z / l}; // Vector3.Normalize
    return {0, 0, 0};
}
// Matrix4x4.LookAt(from, to, up) rotation columns (A4); from is always the origin at our call sites.
void look_basis(f3 forward_in, f3 up_in, f3& right, f3& up, f3& fwd) {
    fwd = v_normalize(forward_in);
    right = v_normalize(v_cross(up_in, fwd));
    up = v_cross(fwd, right);
}
m4 look_at_origin(f3 forward_in, f3 up_in) {
    f3 r, u, f;
    look_basis(forward_in, up_in, r, u, f);
    m4 m = m4_identity();
    m.c[0][0] = r.x; m.c[0][1] = r.y; m.c[0][2] = r.z;
    m.c[1][0] = u.x; m.c[1][1] = u.y; m.c[1][2] = u.z;
    m.c[2][0] = f.x; m.c[2][1] = f.y; m.c[2][2] = f.z;
    return m;
}
// Quaternion.LookRotation(forward, Vector3.up): basis -> quaternion
quat q_look_rotation(f3 forward_in) {
    f3 r, u, f;
    look_basis(forward_in, f3{0, 1, 0}, r, u, f);
    float m00 = r.x, m01 = u.x, m02 = f.x;
    float m10 = r.y, m11 = u.y, m12 = f.y;
    float m20 = r.z, m21 = u.z, m22 = f.z;
    float tr = m00 + m11 + m22;
    quat q;
    if (tr > 0.0f) {
        float s = sqrtf(tr + 1.0f);
        q.w = s * 0.5f; s = 0.5f / s;
        q.x = (m21 - m12) * s; q.y = (m02 - m20) * s; q.z = (m10 - m01) * s;
    } else if (m00 >= m11 && m00 >= m22) {
        float s = sqrtf(1.0f + m00 - m11 - m22), t = 0.5f / s;
        q.x = 0.5f * s; q.y = (m10 + m01) * t; q.z = (m20 + m02) * t; q.w = (m21 - m12) * t;
    } else if (m11 > m22) {
        float s = sqrtf(1.0f + m11 - m00 - m22), t = 0.5f / s;
        q.x = (m01 + m10) * t; q.y = 0.5f * s; q.z = (m12 + m21) * t; q.w = (m02 - m20) * t;
    } else {
        float s = sqrtf(1.0f + m22 - m00 - m11), t = 0.5f / s;
        q.x = (m02 + m20) * t; q.y = (m12 + m21) * t; q.z = 0.5f * s; q.w = (m10 - m01) * t;
    }
    return q;
}
// Camera.nonJitteredProjectionMatrix = GL-convention perspective (A2)
m4 perspective(float fov_deg, float aspect, float zn, float zf) {
    float t = (float)tan((double)(fov_deg * DEG2RAD * 0.5f));
    float cot = 1.0f / t;
    m4 m; memset(&m, 0, sizeof m);
    m.c[0][0] = cot / aspect;
    m.c[1][1] = cot;
    m.c[2][2] = -(zf + zn) / (zf - zn);
    m.c[3][2] = -(2.0f * zf * zn) / (zf - zn);
    m.c[2][3] = -1.0f;
    return m;
}
// Camera.worldToCameraMatrix = Scale(1,1,-1) * inverse(TRS(pos, rot, 1)) (A3), written out for a rigid transform.
m4 world_to_camera(f3 pos, quat rot) {
    f3 r = q_rot(rot, f3{1, 0, 0}), u = q_rot(rot, f3{0, 1, 0}), f = q_rot(rot, f3{0, 0, 1});
    m4 m = m4_identity();
    m.c[0][0] = r.x; m.c[1][0] = r.y; m.c[2][0] = r.z; m.c[3][0] = -v_dot(r, pos);
    m.c[0][1] = u.x; m.c[1][1] = u.y; m.c[2][1] = u.z; m.c[3][1] = -v_dot(u, pos);
    m.c[0][2] = -f.x; m.c[1][2] = -f.y; m.c[2][2] = -f.z; m.c[3][2] = v_dot(f, pos);
    return m;
}
// Vector2.SignedAngle (A5)
float signed_angle(f2 a, f2 b) {
    float denom = sqrtf((a.x * a.x + a.y * a.y) * (b.x * b.x + b.y * b.y));
    float ang;
    if (denom < 1e-15f) ang = 0.0f;
    else {
        float d = (a.x * b.x + a.y * b.y) / denom;
        d = d < -1.0f ? -1.0f : (d > 1.0f ? 1.0f : d);
        ang = (float)acos((double)d) * 57.29578f;
    }
    float s = (a.x * b.y - a.y * b.x) >= 0.0f ? 1.0f : -1.0f; // Mathf.Sign
    return ang * s;
}

// ---------------------------------------------------------------------------------------------
// World read side: Code/World.cs:130-149,161-188,245-259,285-293
// ---------------------------------------------------------------------------------------------
struct RLEColumn {            // World.cs:161-169, 12 bytes
    int32_t elementOffset;
    uint16_t runCount, worldMin, worldMax;
    uint16_t _pad;
};
struct RLEElement { int16_t ColorsIndex, Length; }; // World.cs:245-259
static_assert(sizeof(RLEColumn) == 12, "RLEColumn layout");

struct WorldLod {
    const uint8_t* blob = nullptr;
    int64_t bytes = 0;
    int columnCount = 0;
    const RLEColumn* columns = nullptr;
    const RLEElement* elements = nullptr; // elementsStart = columns + columnCount (World.cs:310)
    int lod = 0;
    int indexingMulX = 0;                 // dimensions.z >> lod (World.cs:31)
};

} // namespace

struct orc_world {
    int dimX, dimY, dimZ;
    WorldLod lods[ORC_LOD_LEVELS];
    int lastLod = 0; // last LOD of the contiguous run set from LOD 0: rays never switch past it
};

namespace {

// World.GetVoxelColumn (World.cs:130-142) + GetIndexKnownInBounds (:145-149)
inline int get_voxel_column(const orc_world* w, const WorldLod& l, i2 pos, RLEColumn& column) {
    int mx = w->dimX - 1, mz = w->dimZ - 1;
    if ((pos.x & mx) != pos.x || (pos.y & mz) != pos.y) return -1;
    int idx = (pos.x >> l.lod) * l.indexingMulX + (pos.y >> l.lod);
    column = l.columns[idx];
    return column.runCount;
}

// ---------------------------------------------------------------------------------------------
// SegmentDDAData: Code/Utils/SegmentDDAData.cs
// ---------------------------------------------------------------------------------------------
struct DDA {
    i2 position, step;
    f2 start, dir, tDelta, tMax;
    f2 dist; // intersectionDistances: x = last, y = next

    // ctor :17-28
    void init(f2 s, f2 d) {
        start = s; dir = d;
        position = {f2i(floorf(s.x)), f2i(floorf(s.y))};
        tDelta = {1.0f / m_max(0.0000001f, fabsf(d.x)), 1.0f / m_max(0.0000001f, fabsf(d.y))};
        f2 sg = {m_sign(d.x), m_sign(d.y)};
        step = {f2i(sg.x), f2i(sg.y)};
        float fx = s.x - floorf(s.x), fy = s.y - floorf(s.y);
        tMax.x = (sg.x * -fx + (sg.x * 0.5f) + 0.5f) * tDelta.x;
        tMax.y = (sg.y * -fy + (sg.y * 0.5f) + 0.5f) * tDelta.y;
        dist = {m_max(tMax.x - tDelta.x, tMax.y - tDelta.y), m_min(tMax.x, tMax.y)};
    }
    // NextLOD :31-73
    void next_lod(int currentVoxelSize) {
        int rx = position.x & (currentVoxelSize * 2 - 1);
        int ry = position.y & (currentVoxelSize * 2 - 1);
        // a still axis entered from outside has tMax = +inf (step_to_world_intersection): its last crossing stays -inf
        f2 prev = {tMax.x != INFINITY ? tMax.x - tDelta.x : -INFINITY, tMax.y != INFINITY ? tMax.y - tDelta.y : -INFINITY};
        if (dir.x >= 0.0f) { if (rx < currentVoxelSize) tMax.x += tDelta.x; else prev.x -= tDelta.x; }
        else               { if (rx < currentVoxelSize) prev.x -= tDelta.x; else tMax.x += tDelta.x; }
        if (dir.y >= 0.0f) { if (ry < currentVoxelSize) tMax.y += tDelta.y; else prev.y -= tDelta.y; }
        else               { if (ry < currentVoxelSize) prev.y -= tDelta.y; else tMax.y += tDelta.y; }
        dist = {m_max(prev.x, prev.y), m_min(tMax.x, tMax.y)};
        position.x -= rx; position.y -= ry;
        tDelta.x *= 2.0f; tDelta.y *= 2.0f;
        step.x *= 2; step.y *= 2;
    }
    // StepToWorldIntersection :75-130
    bool step_to_world_intersection(f2 dims) {
        f2 inv = {1.0f / dir.x, 1.0f / dir.y};
        f2 tmin = {-INFINITY, -INFINITY}, tmax = {INFINITY, INFINITY};
        if (dir.x != 0.0f) {
            float t1 = -start.x * inv.x, t2 = (dims.x - start.x) * inv.x;
            tmin.x = m_min(t1, t2); tmax.x = m_max(t1, t2);
        }
        if (dir.y != 0.0f) {
            float t1 = -start.y * inv.y, t2 = (dims.y - start.y) * inv.y;
            tmin.y = m_min(t1, t2); tmax.y = m_max(t1, t2);
        }
        float tmint = m_max(tmin.x, tmin.y), tmaxt = m_min(tmax.x, tmax.y);
        if (tmaxt < tmint || tmint <= 0.0f) return false;
        f2 tLast;
        if (tmin.x < tmin.y && tmin.x != -INFINITY) {
            tLast.y = tmin.y;
            float off = tmint * dir.x;
            float hit = start.x + off;
            hit = dir.x > 0.0f ? floorf(hit) : ceilf(hit);
            off = hit - start.x;
            tLast.x = off / dir.x;
        } else if (dir.y != 0.0f) {
            tLast.x = tmin.x;
            float off = tmint * dir.y;
            float hit = start.y + off;
            hit = dir.y > 0.0f ? floorf(hit) : ceilf(hit);
            off = hit - start.y;
            tLast.y = off / dir.y;
        } else {
            tLast = {tmin.x, -INFINITY};
        }
        // still-axis rule (DESIGN.md §5): an axis with dir == 0 never bounds the entry and is never crossed (tLast -inf, tMax +inf)
        tMax = {dir.x != 0.0f ? tLast.x + tDelta.x : INFINITY, dir.y != 0.0f ? tLast.y + tDelta.y : INFINITY};
        dist = {m_max(tLast.x, tLast.y), m_min(tMax.x, tMax.y)};
        float mid = m_lerp(dist.x, dist.y, 0.5f);
        position = {f2i(floorf(start.x + mid * dir.x)), f2i(floorf(start.y + mid * dir.y))};
        return true;
    }
    // Step :135-150
    bool do_step(float farclip) {
        float crossed;
        if (tMax.x < tMax.y) { crossed = tMax.x; tMax.x += tDelta.x; position.x += step.x; }
        else                 { crossed = tMax.y; tMax.y += tDelta.y; position.y += step.y; }
        dist = {crossed, m_min(tMax.x, tMax.y)};
        return crossed >= farclip;
    }
    bool beyond_far_clip(float farClip) const { return m_min(tMax.x, tMax.y) >= farClip; } // :152-155
};

// ---------------------------------------------------------------------------------------------
// CameraData helpers: Code/Utils/CameraData.cs:38-163
// ---------------------------------------------------------------------------------------------
inline float cross2(float ax, float ay, float bx, float by) { return ax * by - ay * bx; } // :117-120
inline void clip_min(f3 pMin, f3 pMax, float frustum, float& out) { // :101-107
    float fi = 1.0f / frustum;
    float c0 = cross2(1.0f, fi, pMax.x, pMax.z);
    float c1 = cross2(1.0f, fi, pMin.x, pMin.z);
    out = 1.0f - (c0 / (c0 - c1));
}
inline void clip_max(f3 pMin, f3 pMax, float frustum, float& out) { // :109-115
    float fi = 1.0f / frustum;
    float c0 = cross2(1.0f, fi, pMax.x, pMax.z);
    float c1 = cross2(1.0f, fi, pMin.x, pMin.z);
    out = c1 / (c1 - c0);
}
// GetWorldBoundsClippingCamSpace :50-99. f3 = (screen axis coord, z', w): .x = coord, .y = z', .z = w
bool world_bounds_clipping(f3 pMin, f3 pMax, float bMin, float bMax, float& minLerp, float& maxLerp) {
    if (pMin.x > pMin.z * bMax) {
        if (pMax.x > pMax.z * bMax) { minLerp = 0.0f; maxLerp = 1.0f; return true; }
        clip_min(pMin, pMax, bMax, minLerp);
        if (pMax.x < pMax.z * bMin) clip_max(pMin, pMax, bMin, maxLerp); else maxLerp = 1.0f;
    } else if (pMax.x > pMax.z * bMax) {
        clip_max(pMin, pMax, bMax, maxLerp);
        if (pMin.x < pMin.z * bMin) clip_min(pMin, pMax, bMin, minLerp); else minLerp = 0.0f;
    } else {
        if (pMin.x < pMin.z * bMin) {
            if (pMax.x < pMax.z * bMin) { minLerp = 0.0f; maxLerp = 1.0f; return true; }
            clip_min(pMin, pMax, bMin, minLerp);
            maxLerp = 1.0f;
        } else if (pMax.x < pMax.z * bMin) {
            clip_max(pMin, pMax, bMin, maxLerp);
            minLerp = 0.0f;
        } else { minLerp = 0.0f; maxLerp = 1.0f; }
    }
    return false;
}
// ClipHomogeneousCameraSpaceLine :123-137 (near plane at z' <= 0; f3.y = z')
bool clip_near(f3& a, f3& b) {
    if (a.y <= 0.0f) {
        if (b.y <= 0.0f) return false;
        float v = b.y / (b.y - a.y);
        a = m_lerp3(b, a, v);
    } else if (b.y <= 0.0f) {
        float v = a.y / (a.y - b.y);
        b = m_lerp3(a, b, v);
    }
    return true;
}
// :140-157 with the u coordinate carried along
bool clip_near_u(f3& a, f3& b, float& uA, float& uB) {
    if (a.y <= 0.0f) {
        if (b.y <= 0.0f) return false;
        float v = b.y / (b.y - a.y);
        a = m_lerp3(b, a, v);
        uA = m_lerp(uB, uA, v);
    } else if (b.y <= 0.0f) {
        float v = a.y / (a.y - b.y);
        b = m_lerp3(a, b, v);
        uB = m_lerp(uA, uB, v);
    }
    return true;
}

// ---------------------------------------------------------------------------------------------
// Segment contexts: RenderManager.DrawSegments context fill, Code/RenderManager.cs:281-318
// ---------------------------------------------------------------------------------------------
struct SegCtx {
    int rayCount;
    int axisMappedToY;
    int rayIndexOffset;
    int pixMin, pixMax;
    int seenLen;
    int buffer; // 0 = TD, 1 = LR
};
void fill_segment_contexts(const orc_frame_setup* s, int W, int H, SegCtx ctx[4], int& totalRays) {
    totalRays = 0;
    float vx = s->vanishing_point_screen[0], vy = s->vanishing_point_screen[1];
    for (int k = 0; k < 4; k++) {
        SegCtx& c = ctx[k];
        memset(&c, 0, sizeof c);
        c.rayCount = s->segments[k].ray_count;
        totalRays += c.rayCount;
        if (c.rayCount <= 0) continue;
        c.axisMappedToY = (k > 1) ? 0 : 1;
        c.rayIndexOffset = 0;
        if (k == 1) c.rayIndexOffset = s->segments[0].ray_count;
        if (k == 3) c.rayIndexOffset = s->segments[2].ray_count;
        if (k < 2) {
            c.buffer = 0;
            int v = i_clamp(f2i(m_round(vy)), 0, H - 1);
            if (k == 0) { c.pixMin = v; c.pixMax = H - 1; } else { c.pixMin = 0; c.pixMax = v; }
        } else {
            c.buffer = 1;
            int v = i_clamp(f2i(m_round(vx)), 0, W - 1);
            if (k == 3) { c.pixMin = 0; c.pixMax = v; } else { c.pixMin = v; c.pixMax = W - 1; }
        }
        c.seenLen = c.axisMappedToY ? H : W; // (int)ceil(screen[axisMappedToY]) :317
    }
}

struct Counters {
    uint64_t dda_steps = 0, columns_nonempty = 0, runs_visited = 0, px_voxel = 0, px_sky = 0, rays = 0;
    // diagnostics only (orc_ray_stats): work distribution along one ray
    uint64_t columns_entered = 0, renarrows = 0, spans_tested = 0, spans_committed = 0, spans_wrote = 0;
};

struct RayCont { // RayContinuation, DrawSegmentRayJob.cs:146-153
    int segment;
    int planeRayIndex;
    uint32_t* rayColumn;
    DDA dda;
    int lod;
};

// WriteSkybox :699-708 / WriteSkyboxFull :710-716
void write_skybox(int mn, int mx, uint32_t* col, const uint8_t* seen, Counters& cn) {
    for (int y = mn; y <= mx; y++) if (seen[y] == 0) { col[y] = SKYBOX; cn.px_sky++; }
}
void write_skybox_full(int mn, int mx, uint32_t* col, Counters& cn) {
    for (int y = mn; y <= mx; y++) { col[y] = SKYBOX; cn.px_sky++; }
}

// ReducePixelHorizon :660-697
void reduce_pixel_horizon(int origMin, int origMax, int& bMin, int& bMax, int& nfMin, int& nfMax,
                          const uint8_t* seen, float& fbMin, float& fbMax) {
    if (bMin <= nfMin) {
        bMin = nfMin;
        if (bMax >= nfMin) {
            nfMin = bMax + 1;
            while (nfMin <= origMax && seen[nfMin] > 0) nfMin += 1;
            fbMin = nfMin - 0.501f;
        }
    }
    if (bMax >= nfMax) {
        bMax = nfMax;
        if (bMin <= nfMax) {
            nfMax = bMin - 1;
            while (nfMax >= origMin && seen[nfMax] > 0) nfMax -= 1;
            fbMax = nfMax + 0.501f;
        }
    }
}

struct Cam {
    m4 worldToScreen;
    f2 posXZ;
    float posY;
    bool inverse;
    float farClip;
    float lodDist[ORC_LOD_LEVELS];
};

// RaySetupJob :12-40, DDASetupJob :49-77, TraceToFirstColumnJob :87-144.
// Returns true when the ray continues into RenderJob (cont filled); false when it was skybox-filled or invalid.
bool setup_ray(const orc_world* w, const orc_frame_setup* s, const SegCtx ctx[4], const Cam& cam,
               uint32_t* td, uint32_t* lr, int W, int H, int flatIndex, RayCont& cont, Counters& cn,
               bool write_pixels, int* out_status) {
    // RaySetupJob
    int planeIndex = flatIndex, seg = -1;
    for (int j = 0; j < 4; j++) {
        int segmentRays = ctx[j].rayCount;
        if (segmentRays <= 0) continue;
        if (planeIndex >= segmentRays) { planeIndex -= segmentRays; continue; }
        seg = j;
        break;
    }
    if (seg < 0) { if (out_status) *out_status = -1; return false; }
    const orc_segment& sd = s->segments[seg];
    // DDASetupJob
    float endRayLerp = planeIndex / (float)sd.ray_count;
    f2 d = {m_lerp(sd.cam_local_plane_ray_min[0], sd.cam_local_plane_ray_max[0], endRayLerp),
            m_lerp(sd.cam_local_plane_ray_min[1], sd.cam_local_plane_ray_max[1], endRayLerp)};
    float rs = 1.0f / sqrtf(d.x * d.x + d.y * d.y); // normalize = x * rsqrt(dot), rsqrt = 1/sqrt
    d = {d.x * rs, d.y * rs};
    cont.segment = seg;
    cont.planeRayIndex = planeIndex;
    cont.dda.init(cam.posXZ, d);
    cont.lod = 0;
    // RayBuffer.Native.GetRayColumn (RayBuffer.cs:121-128) on the flattened buffer
    int row = planeIndex + ctx[seg].rayIndexOffset;
    cont.rayColumn = ctx[seg].buffer == 0 ? td + (int64_t)row * H : lr + (int64_t)row * W;
    cn.rays++;
    // TraceToFirstColumnJob
    float farClip = cam.farClip;
    float lodMax = cam.lodDist[0];
    i2 sp = cont.dda.position;
    if (sp.x < 0 || sp.y < 0 || sp.x >= w->dimX || sp.y >= w->dimZ) {
        if (cont.dda.step_to_world_intersection(f2{(float)w->dimX, (float)w->dimZ})) {
            while (cont.lod < w->lastLod && cont.dda.dist.x >= lodMax) { // never past the last uploaded LOD
                cont.dda.next_lod(1 << cont.lod);
                cont.lod++;
                cn.dda_steps++;
                lodMax = cam.lodDist[cont.lod];
            }
            if (cont.dda.beyond_far_clip(farClip)) {
                if (write_pixels) write_skybox_full(ctx[seg].pixMin, ctx[seg].pixMax, cont.rayColumn, cn);
                if (out_status) *out_status = 1;
                return false;
            }
            if (out_status) *out_status = 0;
            return true;
        }
        if (write_pixels) write_skybox_full(ctx[seg].pixMin, ctx[seg].pixMax, cont.rayColumn, cn);
        if (out_status) *out_status = 1;
        return false;
    }
    if (out_status) *out_status = 0;
    return true;
}

// ExecuteRay, DrawSegmentRayJob.cs:195-620
void execute_ray(const orc_world* w, const SegCtx& sc, const Cam& cam, const RayCont& rc, int ITER,
                 std::vector<uint8_t>& seenStorage, Counters& cn) {
    DDA ray = rc.dda;
    uint32_t* rayColumn = rc.rayColumn;
    int lod = rc.lod;
    int voxelScale = 1 << lod;
    const WorldLod* world = &w->lods[lod];
    float farClip = cam.farClip;
    RLEColumn worldColumn; memset(&worldColumn, 0, sizeof worldColumn);
    float lodMax = cam.lodDist[lod];

    seenStorage.assign((size_t)sc.seenLen, 0);   // stackalloc, zero-initialised :208
    uint8_t* seen = seenStorage.data();

    const int origMin = sc.pixMin, origMax = sc.pixMax;
    int nextFreePixelMin = origMin, nextFreePixelMax = origMax;

    float worldMaxY = (float)w->dimY;
    float cameraPosYNormalized = cam.posY / worldMaxY;

    float frustumBoundsMin = nextFreePixelMin - 0.501f;
    float frustumBoundsMax = nextFreePixelMax + 0.501f;
    float frustumDirMaxWorld = FLOAT_EPSILON;
    float frustumDirMinWorld = FLOAT_EPSILON;

    // SetupProjectedPlaneParams :622-651
    f3 planeStartBottomProjected, planeStartTopProjected, planeRayDirectionProjected;
    {
        f4 top = mul(cam.worldToScreen, f4{ray.start.x, worldMaxY, ray.start.y, 1.0f});
        f4 bot = mul(cam.worldToScreen, f4{ray.start.x, 0.0f, ray.start.y, 1.0f});
        f4 dir = mul(cam.worldToScreen, f4{ray.dir.x, 0.0f, ray.dir.y, 0.0f});
        if (sc.axisMappedToY == 0) {
            planeStartBottomProjected = {bot.x, bot.z, bot.w};
            planeStartTopProjected = {top.x, top.z, top.w};
            planeRayDirectionProjected = {dir.x, dir.z, dir.w};
        } else {
            planeStartBottomProjected = {bot.y, bot.z, bot.w};
            planeStartTopProjected = {top.y, top.z, top.w};
            planeRayDirectionProjected = {dir.y, dir.z, dir.w};
        }
    }
    auto madd3 = [](f3 a, f3 d, float t) { return f3{a.x + d.x * t, a.y + d.y * t, a.z + d.z * t}; };

    while (true) {
        if (lod < w->lastLod && ray.dist.x >= lodMax) { // :237-243, never past the last uploaded LOD
            ray.next_lod(voxelScale);
            lod++;
            voxelScale *= 2;
            world++;
            lodMax = cam.lodDist[lod];
        }

        cn.dda_steps++;
        int columnRuns = get_voxel_column(w, *world, ray.position, worldColumn);
        if (columnRuns == -1) { write_skybox(origMin, origMax, rayColumn, seen, cn); return; }
        if (columnRuns == 0) {
            if (ray.do_step(farClip)) break;
            continue;
        }
        cn.columns_nonempty++;

        float worldBoundsMin = 0.0f;
        float worldBoundsMax = worldMaxY;

        if (frustumDirMaxWorld != FLOAT_EPSILON) { // :261-281
            float distTop = frustumDirMaxWorld > 0.0f ? ray.dist.y : ray.dist.x;
            float distBot = frustumDirMinWorld < 0.0f ? ray.dist.y : ray.dist.x;
            float newMax = cam.posY + frustumDirMaxWorld * distTop;
            float newMin = cam.posY + frustumDirMinWorld * distBot;
            if (newMin > worldBoundsMax || newMax < worldBoundsMin) { write_skybox(origMin, origMax, rayColumn, seen, cn); return; }
            if ((float)worldColumn.worldMin > newMax || (float)worldColumn.worldMax < newMin) {
                if (ray.do_step(farClip)) break;
                continue;
            }
            worldBoundsMin = newMin;
            worldBoundsMax = newMax;
        }

        f3 camSpaceMinLast = madd3(planeStartBottomProjected, planeRayDirectionProjected, ray.dist.x); // :289-293
        f3 camSpaceMinNext = madd3(planeStartBottomProjected, planeRayDirectionProjected, ray.dist.y);
        f3 camSpaceMaxLast = madd3(planeStartTopProjected, planeRayDirectionProjected, ray.dist.x);
        f3 camSpaceMaxNext = madd3(planeStartTopProjected, planeRayDirectionProjected, ray.dist.y);

        if (ray.dist.x > 2.0f && frustumDirMaxWorld == FLOAT_EPSILON) { // :295-422
            cn.renarrows++;
            float clipLastMinLerp, clipLastMaxLerp, clipNextMinLerp, clipNextMaxLerp;
            bool clippedLast = world_bounds_clipping(camSpaceMinLast, camSpaceMaxLast, frustumBoundsMin, frustumBoundsMax, clipLastMinLerp, clipLastMaxLerp);
            bool clippedNext = world_bounds_clipping(camSpaceMinNext, camSpaceMaxNext, frustumBoundsMin, frustumBoundsMax, clipNextMinLerp, clipNextMaxLerp);
            float camSpaceClippedMin, camSpaceClippedMax;
            if (clippedLast) {
                if (clippedNext) { write_skybox(origMin, origMax, rayColumn, seen, cn); return; }
                worldBoundsMin = m_lerp(0.0f, worldMaxY, clipNextMinLerp);
                worldBoundsMax = m_lerp(0.0f, worldMaxY, clipNextMaxLerp);
                frustumDirMaxWorld = (worldBoundsMax - cam.posY) / ray.dist.y;
                frustumDirMinWorld = (worldBoundsMin - cam.posY) / ray.dist.y;
                f3 minClip = m_lerp3(camSpaceMinNext, camSpaceMaxNext, clipNextMinLerp);
                f3 maxClip = m_lerp3(camSpaceMinNext, camSpaceMaxNext, clipNextMaxLerp);
                camSpaceClippedMin = minClip.x / minClip.z;
                camSpaceClippedMax = maxClip.x / maxClip.z;
                if (camSpaceClippedMax < camSpaceClippedMin) std::swap(camSpaceClippedMin, camSpaceClippedMax);
            } else if (clippedNext) {
                worldBoundsMin = m_lerp(0.0f, worldMaxY, clipLastMinLerp);
                worldBoundsMax = m_lerp(0.0f, worldMaxY, clipLastMaxLerp);
                f3 minClip = m_lerp3(camSpaceMinLast, camSpaceMaxLast, clipLastMinLerp);
                f3 maxClip = m_lerp3(camSpaceMinLast, camSpaceMaxLast, clipLastMaxLerp);
                frustumDirMaxWorld = (worldBoundsMax - cam.posY) / ray.dist.x;
                frustumDirMinWorld = (worldBoundsMin - cam.posY) / ray.dist.x;
                camSpaceClippedMin = minClip.x / minClip.z;
                camSpaceClippedMax = maxClip.x / maxClip.z;
                if (camSpaceClippedMax < camSpaceClippedMin) std::swap(camSpaceClippedMin, camSpaceClippedMax);
            } else {
                if (clipLastMinLerp < clipNextMinLerp) {
                    worldBoundsMin = m_lerp(0.0f, worldMaxY, clipLastMinLerp);
                    frustumDirMinWorld = (worldBoundsMin - cam.posY) / ray.dist.x;
                } else {
                    worldBoundsMin = m_lerp(0.0f, worldMaxY, clipNextMinLerp);
                    frustumDirMinWorld = (worldBoundsMin - cam.posY) / ray.dist.y;
                }
                if (clipLastMaxLerp > clipNextMaxLerp) {
                    worldBoundsMax = m_lerp(0.0f, worldMaxY, clipLastMaxLerp);
                    frustumDirMaxWorld = (worldBoundsMax - cam.posY) / ray.dist.x;
                } else {
                    worldBoundsMax = m_lerp(0.0f, worldMaxY, clipNextMaxLerp);
                    frustumDirMaxWorld = (worldBoundsMax - cam.posY) / ray.dist.y;
                }
                f3 minClipA = m_lerp3(camSpaceMinLast, camSpaceMaxLast, clipLastMinLerp);
                f3 maxClipA = m_lerp3(camSpaceMinLast, camSpaceMaxLast, clipLastMaxLerp);
                f3 minClipB = m_lerp3(camSpaceMinNext, camSpaceMaxNext, clipNextMinLerp);
                f3 maxClipB = m_lerp3(camSpaceMinNext, camSpaceMaxNext, clipNextMaxLerp);
                float minNext = minClipB.x / minClipB.z;
                float minLast = minClipA.x / minClipA.z;
                float maxNext = maxClipB.x / maxClipB.z;
                float maxLast = maxClipA.x / maxClipA.z;
                if (maxNext < minNext) std::swap(maxNext, minNext);
                if (maxLast < minLast) std::swap(maxLast, minLast);
                camSpaceClippedMin = m_min(minLast, minNext);
                camSpaceClippedMax = m_max(maxLast, maxNext);
            }

            worldBoundsMin = floorf(worldBoundsMin);
            worldBoundsMax = ceilf(worldBoundsMax);

            int writableMinPixel = f2i(floorf(camSpaceClippedMin));
            int writableMaxPixel = f2i(ceilf(camSpaceClippedMax));

            if (writableMaxPixel < nextFreePixelMin || writableMinPixel > nextFreePixelMax) { write_skybox(origMin, origMax, rayColumn, seen, cn); return; }
            if (writableMinPixel > nextFreePixelMin) {
                nextFreePixelMin = writableMinPixel;
                while (nextFreePixelMin <= origMax && seen[nextFreePixelMin] > 0) nextFreePixelMin += 1;
            }
            if (writableMaxPixel < nextFreePixelMax) {
                nextFreePixelMax = writableMaxPixel;
                while (nextFreePixelMax >= origMin && seen[nextFreePixelMax] > 0) nextFreePixelMax -= 1;
            }
            if (nextFreePixelMin > nextFreePixelMax) { write_skybox(origMin, origMax, rayColumn, seen, cn); return; }
        }

        cn.columns_entered++;
        float elementBoundsMin, elementBoundsMax;
        const RLEElement* elementPointer;
        const RLEElement* guardStart = world->elements + worldColumn.elementOffset; // ElementGuardStart World.cs:175-178
        if (ITER > 0) {
            elementBoundsMin = worldMaxY; elementBoundsMax = worldMaxY;
            elementPointer = guardStart;
        } else {
            elementBoundsMin = 0.0f; elementBoundsMax = 0.0f;
            elementPointer = guardStart + worldColumn.runCount + 1; // ElementGuardEnd :180-183
        }
        const uint32_t* worldColumnColors = (const uint32_t*)guardStart + worldColumn.runCount + 2; // ColorPointer :185-188

        while (true) { // :441-611
            elementPointer += ITER;
            RLEElement element = *elementPointer;
            if (element.Length == 0) break; // !IsValid
            cn.runs_visited++;

            if (ITER > 0) {
                elementBoundsMax = elementBoundsMin;
                elementBoundsMin = elementBoundsMin - (float)(element.Length * voxelScale);
            } else {
                elementBoundsMin = elementBoundsMax;
                elementBoundsMax = elementBoundsMin + (float)(element.Length * voxelScale);
            }
            if (element.ColorsIndex < 0) continue; // IsAir

            if (elementBoundsMin > worldBoundsMax) { if (ITER < 0) break; else continue; }
            if (elementBoundsMax < worldBoundsMin) { if (ITER > 0) break; else continue; }

            float portionBottom = m_unlerp(0.0f, worldMaxY, elementBoundsMin);
            float portionTop = m_unlerp(0.0f, worldMaxY, elementBoundsMax);
            f3 camSpaceFrontBottom = m_lerp3(camSpaceMinLast, camSpaceMaxLast, portionBottom);
            f3 camSpaceFrontTop = m_lerp3(camSpaceMinLast, camSpaceMaxLast, portionTop);

            { // side of the run :484-542
                float uA = (float)element.Length;
                float uB = 0.0f;
                // the clip modifies camSpaceFrontBottom/Top in place (ref args); the cap below reuses the clipped values
                bool ok = clip_near_u(camSpaceFrontBottom, camSpaceFrontTop, uA, uB);
                if (ok) {
                    f2 uvA = {1.0f / camSpaceFrontBottom.z, uA / camSpaceFrontBottom.z};
                    f2 uvB = {1.0f / camSpaceFrontTop.z, uB / camSpaceFrontTop.z};
                    f2 bf = {camSpaceFrontBottom.x / camSpaceFrontBottom.z, camSpaceFrontTop.x / camSpaceFrontTop.z}; // ProjectClippedToScreen
                    if (bf.x > bf.y) { std::swap(bf.x, bf.y); std::swap(uvA, uvB); }
                    int bMin = f2i(m_round(bf.x));
                    int bMax = f2i(m_round(bf.y));
                    cn.spans_tested++;
                    if (bMax >= nextFreePixelMin && bMin <= nextFreePixelMax) {
                        cn.spans_committed++;
                        const uint64_t pxBefore = cn.px_voxel;
                        reduce_pixel_horizon(origMin, origMax, bMin, bMax, nextFreePixelMin, nextFreePixelMax, seen, frustumBoundsMin, frustumBoundsMax);
                        for (int y = bMin; y <= bMax; y++) {
                            if (seen[y] == 0) {
                                frustumDirMaxWorld = FLOAT_EPSILON;
                                seen[y] = 1;
                                float l = m_unlerp(bf.x, bf.y, (float)y);
                                float wx = m_lerp(uvA.x, uvB.x, l), wy = m_lerp(uvA.y, uvB.y, l);
                                float u = wy / wx;
                                int colorIdx = i_clamp(f2i(floorf(u)), 0, element.Length - 1) + element.ColorsIndex;
                                rayColumn[y] = worldColumnColors[colorIdx];
                                cn.px_voxel++;
                            }
                        }
                        if (cn.px_voxel != pxBefore) cn.spans_wrote++;
                        if (nextFreePixelMin > nextFreePixelMax) { write_skybox(origMin, origMax, rayColumn, seen, cn); return; }
                    }
                }
            }

            // top/bottom cap :544-610. NOTE: camSpaceFrontTop/Bottom may have been near-clipped above (refs).
            f3 secA, secB;
            uint32_t secondaryColor;
            if (portionTop < cameraPosYNormalized) {
                if (elementBoundsMax > worldBoundsMax) continue;
                secondaryColor = worldColumnColors[element.ColorsIndex + 0];
                secA = m_lerp3(camSpaceMinNext, camSpaceMaxNext, portionTop);
                secB = camSpaceFrontTop;
            } else if (portionBottom > cameraPosYNormalized) {
                if (elementBoundsMin < worldBoundsMin) continue;
                secondaryColor = worldColumnColors[element.ColorsIndex + element.Length - 1];
                secA = m_lerp3(camSpaceMinNext, camSpaceMaxNext, portionBottom);
                secB = camSpaceFrontBottom;
            } else continue;

            if (clip_near(secA, secB)) {
                float fx = m_round(secA.x / secA.z), fy = m_round(secB.x / secB.z);
                int bMin = f2i(fx), bMax = f2i(fy);
                if (bMin > bMax) std::swap(bMin, bMax);
                cn.spans_tested++;
                if (bMax >= nextFreePixelMin && bMin <= nextFreePixelMax) {
                    cn.spans_committed++;
                    const uint64_t pxBefore = cn.px_voxel;
                    reduce_pixel_horizon(origMin, origMax, bMin, bMax, nextFreePixelMin, nextFreePixelMax, seen, frustumBoundsMin, frustumBoundsMax);
                    for (int y = bMin; y <= bMax; y++) {
                        if (seen[y] == 0) {
                            frustumDirMaxWorld = FLOAT_EPSILON;
                            seen[y] = 1;
                            rayColumn[y] = secondaryColor;
                            cn.px_voxel++;
                        }
                    }
                    if (cn.px_voxel != pxBefore) cn.spans_wrote++;
                    if (nextFreePixelMin > nextFreePixelMax) { write_skybox(origMin, origMax, rayColumn, seen, cn); return; }
                }
            }
        }

        if (ray.do_step(farClip)) break;
    }
    write_skybox(origMin, origMax, rayColumn, seen, cn); // :619
}

Cam make_cam(const orc_camera& c) {
    Cam cam;
    for (int j = 0; j < 4; j++) for (int i = 0; i < 4; i++) cam.worldToScreen.c[j][i] = c.world_to_screen[j * 4 + i];
    cam.posXZ = {c.position_xz[0], c.position_xz[1]};
    cam.posY = c.position_y;
    cam.inverse = c.inverse_element_iteration_direction != 0;
    cam.farClip = c.far_clip;
    for (int i = 0; i < ORC_LOD_LEVELS; i++) cam.lodDist[i] = c.lod_distances[i];
    return cam;
}

template <class F>
void parallel_for(int n, int n_threads, F fn) {
    if (n_threads <= 0) n_threads = (int)std::thread::hardware_concurrency();
    if (n_threads < 1) n_threads = 1;
    if (n_threads == 1 || n <= 1) { for (int i = 0; i < n; i++) fn(i, 0); return; }
    std::atomic<int> next(0);
    std::vector<std::thread> th;
    for (int t = 0; t < n_threads; t++)
        th.emplace_back([&, t]() { for (;;) { int i = next.fetch_add(1); if (i >= n) break; fn(i, t); } });
    for (auto& x : th) x.join();
}

} // namespace

extern "C" {

orc_world* orc_world_create(int32_t dim_x, int32_t dim_y, int32_t dim_z) {
    orc_world* w = new orc_world();
    w->dimX = dim_x; w->dimY = dim_y; w->dimZ = dim_z;
    return w;
}

int orc_world_set_lod(orc_world* w, int32_t lod, const void* blob, int64_t bytes, int32_t column_count) {
    if (!w || lod < 0 || lod >= ORC_LOD_LEVELS || !blob) return -1;
    WorldLod& l = w->lods[lod];
    l.blob = (const uint8_t*)blob; l.bytes = bytes; l.columnCount = column_count;
    l.columns = (const RLEColumn*)blob;
    l.elements = (const RLEElement*)(l.columns + column_count);
    l.lod = lod;
    l.indexingMulX = w->dimZ >> lod;
    w->lastLod = 0;
    while (w->lastLod + 1 < ORC_LOD_LEVELS && w->lods[w->lastLod + 1].blob) w->lastLod++;
    return 0;
}

void orc_world_free(orc_world* w) { delete w; }

void orc_min_max(const float* a, const float* b, int32_t n, float* out_min, float* out_max) {
    for (int32_t i = 0; i < n; i++) { out_min[i] = m_min(a[i], b[i]); out_max[i] = m_max(a[i], b[i]); }
}

int orc_hardware_threads(void) { int n = (int)std::thread::hardware_concurrency(); return n > 0 ? n : 1; }

void orc_quat_euler(float x, float y, float z, float out[4]) {
    quat q = q_euler(x, y, z);
    out[0] = q.x; out[1] = q.y; out[2] = q.z; out[3] = q.w;
}

// UnityManager.LimitRotationHorizon, Code/UnityManager.cs:193-201
void orc_limit_rotation_horizon(orc_pose* p) {
    quat q = {p->rotation[0], p->rotation[1], p->rotation[2], p->rotation[3]};
    f3 forward = q_rot(q, f3{0, 0, 1});
    if (fabsf(forward.y) < 0.001f) {
        forward.y = (forward.y >= 0.0f ? 1.0f : -1.0f) * 0.001f; // Mathf.Sign(0) = +1
        quat r = q_look_rotation(forward);                          // transform.forward = v => LookRotation(v)
        p->rotation[0] = r.x; p->rotation[1] = r.y; p->rotation[2] = r.z; p->rotation[3] = r.w;
    }
}

// UnityManager.SetupLods, Code/UnityManager.cs:417-458 (window == render resolution => pixelW = pixelH = 1, A8)
void orc_setup_lods(int32_t worldMaxDimension, int32_t resX, int32_t resY, float fov, float lodError, float out[ORC_LOD_LEVELS]) {
    float clipMax = (float)(worldMaxDimension * 2);
    float pixelW = (1.0f / resX) * resX, pixelH = (1.0f / resY) * resY;
    int midW = resX / 2, midH = resY / 2;
    float t = (float)tan((double)(fov * DEG2RAD * 0.5f));
    float aspect = (float)resX / (float)resY;
    auto dir = [&](float px, float py) {
        f3 d = {(2.0f * px / resX - 1.0f) * aspect * t, (2.0f * py / resY - 1.0f) * t, 1.0f};
        return v_normalize(d);
    };
    f3 a = dir((float)midW, (float)midH), b = dir(midW + pixelW, midH + pixelH);
    bool has[ORC_LOD_LEVELS] = {false};
    float lods[ORC_LOD_LEVELS] = {0};
    float pixelWidth = 1.41f / lodError;
    for (float p = 0.0f; p < 1.0f; p += 0.0001f) {
        float rayDist = p * clipMax;
        f3 pA = {a.x * rayDist, a.y * rayDist, a.z * rayDist}, pB = {b.x * rayDist, b.y * rayDist, b.z * rayDist};
        f3 dd = {pA.x - pB.x, pA.y - pB.y, pA.z - pB.z};
        float pAB = sqrtf(v_dot(dd, dd));
        for (int j = 0; j < ORC_LOD_LEVELS; j++)
            if (!has[j] && pAB > pixelWidth * (float)(2 << j)) { has[j] = true; lods[j] = p; }
    }
    has[ORC_LOD_LEVELS - 1] = true; lods[ORC_LOD_LEVELS - 1] = 2.0f;
    for (int i = 0; i < ORC_LOD_LEVELS; i++) out[i] = ceilf((has[i] ? lods[i] : 2.0f) * clipMax);
}

// RenderManager.DrawWorld up to DrawSegments: Code/RenderManager.cs:119-152,374-501; CameraData ctor CameraData.cs:18-36
int orc_frame_setup_from_pose(const orc_pose* pose, const float lodDist[ORC_LOD_LEVELS], int32_t worldDimY, orc_frame_setup* out) {
    (void)worldDimY;
    if (!pose || !out) return -1;
    memset(out, 0, sizeof *out);
    const int W = pose->pixel_width, H = pose->pixel_height;
    quat rot = {pose->rotation[0], pose->rotation[1], pose->rotation[2], pose->rotation[3]};
    f3 pos = {pose->position[0], pose->position[1], pose->position[2]};
    f3 forward = q_rot(rot, f3{0, 0, 1}), up = q_rot(rot, f3{0, 1, 0});
    float aspect = (float)W / (float)H;
    m4 proj = perspective(pose->fov_y_degrees, aspect, pose->near_clip, pose->far_clip);
    f2 screen = {(float)W, (float)H};

    // CalculateVanishingPointWorld :374-378 (A6: -near / sin(euler.x) == near / forward.y)
    float vpOff = pose->near_clip / forward.y;
    f3 vpLocal = {0.0f, vpOff, 0.0f}; // worldPos - position, position + up*off - position
    {   // subtract in world space exactly as the reference does
        f3 vpWorld = {pos.x + 0.0f * vpOff, pos.y + 1.0f * vpOff, pos.z + 0.0f * vpOff};
        vpLocal = {vpWorld.x - pos.x, vpWorld.y - pos.y, vpWorld.z - pos.z};
    }
    // ProjectVanishingPointScreenToWorld :380-394
    m4 look = look_at_origin(forward, up);
    m4 view = mul(m4_scale(1, 1, -1), m4_inverse(look));
    m4 localToScreen = mul(proj, view);
    f4 camPos = mul(localToScreen, f4{vpLocal.x, vpLocal.y, vpLocal.z, 1.0f});
    f2 vp = {((camPos.x / camPos.w) * 0.5f + 0.5f) * (float)W, ((camPos.y / camPos.w) * 0.5f + 0.5f) * (float)H};
    out->vanishing_point_screen[0] = vp.x; out->vanishing_point_screen[1] = vp.y;

    // TransformPixel :487-500
    m4 unproj = m4_inverse(proj);
    unproj = mul(m4_inverse(m4_scale(1, 1, -1)), unproj);
    unproj = mul(look, unproj);
    auto transform_pixel = [&](f2 pixel, float o[2]) {
        f4 v = mul(unproj, f4{((pixel.x / (float)W) - 0.5f) * 2.0f, ((pixel.y / (float)H) - 0.5f) * 2.0f, 1.0f, 1.0f});
        o[0] = v.x / v.w; o[1] = v.z / v.w;
    };

    // GetGenericSegmentParameters :402-485
    auto segment = [&](float distToOtherEnd, f2 neutral, int primaryAxis, orc_segment& seg) {
        memset(&seg, 0, sizeof seg);
        int secondaryAxis = 1 - primaryAxis;
        float vpa[2] = {vp.x, vp.y}, scr[2] = {screen.x, screen.y}, neu[2] = {neutral.x, neutral.y};
        float sMin[2], sMax[2];
        sMin[0] = sMin[1] = vpa[secondaryAxis] - distToOtherEnd;
        sMax[0] = sMax[1] = vpa[secondaryAxis] + distToOtherEnd;
        float a = vpa[primaryAxis] + distToOtherEnd * m_sign(neu[primaryAxis]);
        sMin[primaryAxis] = a; sMax[primaryAxis] = a;
        if (sMax[secondaryAxis] <= 0.0f || sMin[secondaryAxis] >= scr[secondaryAxis]) return;
        float mn[2], mx[2];
        if (vp.x >= 0.0f && vp.y >= 0.0f && vp.x <= screen.x && vp.y <= screen.y) {
            mn[0] = sMin[0]; mn[1] = sMin[1]; mx[0] = sMax[0]; mx[1] = sMax[1];
        } else {
            f2 dirSimpleMiddle = {m_lerp(sMin[0], sMax[0], 0.5f) - vp.x, m_lerp(sMin[1], sMax[1], 0.5f) - vp.y};
            float angleLeft = 90.0f, angleRight = -90.0f;
            f2 dirRight = {0, 0}, dirLeft = {0, 0};
            f2 vectors[4] = {{0.0f, 0.0f}, {0.0f, screen.y}, {screen.x, 0.0f}, {screen.x, screen.y}};
            for (int i = 0; i < 4; i++) {
                f2 dir = {vectors[i].x - vp.x, vectors[i].y - vp.y};
                float dp = primaryAxis == 0 ? dir.x : dir.y;
                float sc = distToOtherEnd / fabsf(dp);
                f2 scaledEnd = {dir.x * sc, dir.y * sc};
                float angle = signed_angle(neutral, dir);
                if (angle < angleLeft) { angleLeft = angle; dirLeft = scaledEnd; }
                if (angle > angleRight) { angleRight = angle; dirRight = scaledEnd; }
            }
            f2 cornerLeft = {dirLeft.x + vp.x, dirLeft.y + vp.y};
            f2 cornerRight = {dirRight.x + vp.x, dirRight.y + vp.y};
            f2 simpleMax = {sMax[0], sMax[1]}, simpleMin = {sMin[0], sMin[1]};
            if (angleLeft < -45.0f) cornerLeft = signed_angle(dirSimpleMiddle, simpleMax) > 0.0f ? simpleMin : simpleMax;   // :466 (point used as a direction, as is)
            if (angleRight > 45.0f) cornerRight = signed_angle(dirSimpleMiddle, simpleMax) < 0.0f ? simpleMin : simpleMax; // :469
            float cl[2] = {cornerLeft.x, cornerLeft.y}, cr[2] = {cornerRight.x, cornerRight.y};
            bool swap = cl[secondaryAxis] > cr[secondaryAxis];
            mn[0] = swap ? cr[0] : cl[0]; mn[1] = swap ? cr[1] : cl[1];
            mx[0] = swap ? cl[0] : cr[0]; mx[1] = swap ? cl[1] : cr[1];
        }
        seg.min_screen[0] = mn[0]; seg.min_screen[1] = mn[1];
        seg.max_screen[0] = mx[0]; seg.max_screen[1] = mx[1];
        transform_pixel(f2{mn[0], mn[1]}, seg.cam_local_plane_ray_min);
        transform_pixel(f2{mx[0], mx[1]}, seg.cam_local_plane_ray_max);
        int rc = f2i(m_round(mx[secondaryAxis] - mn[secondaryAxis]));
        seg.ray_count = rc > 0 ? rc : 0;
    };
    // DrawWorld :128-142
    if (vp.y < screen.y) segment(screen.y - vp.y, f2{0, 1}, 1, out->segments[0]);
    if (vp.y > 0.0f) segment(vp.y, f2{0, -1}, 1, out->segments[1]);
    if (vp.x < screen.x) segment(screen.x - vp.x, f2{1, 0}, 0, out->segments[2]);
    if (vp.x > 0.0f) segment(vp.x, f2{-1, 0}, 0, out->segments[3]);

    // CameraData ctor, CameraData.cs:18-36
    m4 wts = mul(proj, world_to_camera(pos, rot));
    wts = mul(m4_scale(0.5f, 0.5f, 1.0f), wts);
    wts = mul(m4_translate(0.5f, 0.5f, 1.0f), wts);
    wts = mul(m4_scale(screen.x, screen.y, 1.0f), wts);
    for (int j = 0; j < 4; j++) for (int i = 0; i < 4; i++) out->camera.world_to_screen[j * 4 + i] = wts.c[j][i];
    out->camera.position_xz[0] = pos.x; out->camera.position_xz[1] = pos.z;
    out->camera.position_y = pos.y;
    out->camera.inverse_element_iteration_direction = forward.y >= 0.0f ? 1 : 0;
    out->camera.far_clip = pose->far_clip;
    for (int i = 0; i < ORC_LOD_LEVELS; i++) out->camera.lod_distances[i] = lodDist[i];
    return 0;
}

// BenchmarkPath.anim sampled with cubic Hermite (A9); UnityManager.cs:86-87 scales the position by the world dimensions.
void orc_benchmark_pose(float t, const int32_t dims[3], orc_pose* p) {
    struct Key { float time, v[3], in[3], out[3]; };
    static const Key euler[] = { // Code/BenchmarkPath.anim:16-82
        {0.0f, {0, 45, 0}, {0, 0, 0}, {0, 0, 0}},
        {0.25f, {0, -45, 0}, {0, -360, 0}, {0, -360, 0}},
        {0.5f, {-16.2f, -135, 0}, {0, 0, 0}, {0, 0, 0}},
        {0.75f, {59.12f, -135, 0}, {0, 0, 0}, {0, 0, 0}},
        {0.875f, {59.12f, -135, 180}, {0, 0, 1440}, {0, 0, 1440}},
        {1.0f, {59.12f, -135, 360}, {0, 0, 0}, {0, 0, 0}},
        {1.15f, {85, -225.5f, 360}, {0, 0, 0}, {0, 0, 0}},
    };
    static const Key posk[] = { // :89-146
        {0.0f, {-0.1f, 0.5f, -0.1f}, {0, 0, 0}, {0, 0, 0}},
        {0.25f, {1.1f, 0.5f, -0.1f}, {0, 0, 0}, {0, 0, 0}},
        {0.5f, {0.9f, 0.3f, 0.9f}, {0, 0, 0}, {0, 0, 0}},
        {0.75f, {0.9f, 0.95f, 0.9f}, {0, 0, 0}, {0, 0, 0}},
        {1.0f, {0.9f, 0.95f, 0.9f}, {0, 0, 0}, {0, 0, 0}},
        {1.15f, {0.427f, 0.95f, 0.52f}, {0, 0, 0}, {0, 0, 0}},
    };
    auto sample = [](const Key* k, int n, float t, float o[3]) {
        if (t <= k[0].time) { for (int c = 0; c < 3; c++) o[c] = k[0].v[c]; return; }
        if (t >= k[n - 1].time) { for (int c = 0; c < 3; c++) o[c] = k[n - 1].v[c]; return; }
        int i = 0;
        while (i + 1 < n && t > k[i + 1].time) i++;
        float dt = k[i + 1].time - k[i].time;
        float s = (t - k[i].time) / dt;
        float s2 = s * s, s3 = s2 * s;
        float h00 = 2 * s3 - 3 * s2 + 1, h10 = s3 - 2 * s2 + s, h01 = -2 * s3 + 3 * s2, h11 = s3 - s2;
        for (int c = 0; c < 3; c++)
            o[c] = h00 * k[i].v[c] + h10 * k[i].out[c] * dt + h01 * k[i + 1].v[c] + h11 * k[i + 1].in[c] * dt;
    };
    float e[3], q[3];
    sample(euler, 7, t, e);
    sample(posk, 6, t, q);
    p->position[0] = q[0] * (float)dims[0]; p->position[1] = q[1] * (float)dims[1]; p->position[2] = q[2] * (float)dims[2];
    orc_quat_euler(e[0], e[1], e[2], p->rotation);
}

int orc_ray_setup(const orc_world* w, const orc_frame_setup* s, int32_t W, int32_t H, orc_ray_state* out, int32_t max_rays) {
    SegCtx ctx[4]; int total;
    fill_segment_contexts(s, W, H, ctx, total);
    Cam cam = make_cam(s->camera);
    int n = total < max_rays ? total : max_rays;
    for (int i = 0; i < n; i++) {
        RayCont rc; Counters cn; int status = 0;
        memset(&rc, 0, sizeof rc);
        setup_ray(w, s, ctx, cam, nullptr, nullptr, W, H, i, rc, cn, false, &status);
        orc_ray_state& o = out[i];
        o.segment = rc.segment; o.plane_ray_index = rc.planeRayIndex; o.status = status; o.lod = rc.lod;
        o.position[0] = rc.dda.position.x; o.position[1] = rc.dda.position.y;
        o.step[0] = rc.dda.step.x; o.step[1] = rc.dda.step.y;
        o.start[0] = rc.dda.start.x; o.start[1] = rc.dda.start.y;
        o.dir[0] = rc.dda.dir.x; o.dir[1] = rc.dda.dir.y;
        o.t_delta[0] = rc.dda.tDelta.x; o.t_delta[1] = rc.dda.tDelta.y;
        o.t_max[0] = rc.dda.tMax.x; o.t_max[1] = rc.dda.tMax.y;
        o.intersection_distances[0] = rc.dda.dist.x; o.intersection_distances[1] = rc.dda.dist.y;
    }
    return total;
}

int orc_render_raybuffers(const orc_world* w, const orc_frame_setup* s, int32_t W, int32_t H, uint32_t* td, uint32_t* lr,
                          int32_t ray_begin, int32_t ray_end, int32_t n_threads, orc_counters* counters) {
    if (!w || !s || !td || !lr) return -1;
    SegCtx ctx[4]; int total;
    fill_segment_contexts(s, W, H, ctx, total);
    if (ray_end < 0 || ray_end > total) ray_end = total;
    if (ray_begin < 0) ray_begin = 0;
    Cam cam = make_cam(s->camera);
    int nt = n_threads <= 0 ? orc_hardware_threads() : n_threads;
    std::vector<Counters> cns((size_t)nt);
    std::vector<std::vector<uint8_t>> seen((size_t)nt);
    int n = ray_end - ray_begin;
    parallel_for(n > 0 ? n : 0, nt, [&](int i, int t) {
        RayCont rc;
        if (!setup_ray(w, s, ctx, cam, td, lr, W, H, ray_begin + i, rc, cns[t], true, nullptr)) return;
        execute_ray(w, ctx[rc.segment], cam, rc, cam.inverse ? -1 : 1, seen[t], cns[t]); // RenderJob.Execute :164-179
    });
    if (counters) {
        memset(counters, 0, sizeof *counters);
        for (auto& c : cns) {
            counters->dda_steps += c.dda_steps; counters->columns_nonempty += c.columns_nonempty;
            counters->runs_visited += c.runs_visited; counters->px_voxel += c.px_voxel;
            counters->px_sky += c.px_sky; counters->rays += c.rays;
        }
    }
    return 0;
}

/* Test hook: the DDA cell sequence of one ray exactly as ExecuteRay walks it (LOD switch at the top of every iteration,
 * DrawSegmentRayJob.cs:237-243, then Step :613). Per step: cell x, cell z, lod, and the (last, next) distances. */
int orc_dda_walk(const float start[2], const float dir[2], const float lod_distances[ORC_LOD_LEVELS], float far_clip,
                 int32_t max_steps, int32_t* out_cells, float* out_dists) {
    DDA d;
    d.init(f2{start[0], start[1]}, f2{dir[0], dir[1]});
    int lod = 0, voxelScale = 1, n = 0;
    float lodMax = lod_distances[0];
    while (n < max_steps) {
        if (d.dist.x >= lodMax) { d.next_lod(voxelScale); lod++; voxelScale *= 2; lodMax = lod_distances[lod]; }
        out_cells[3 * n] = d.position.x; out_cells[3 * n + 1] = d.position.y; out_cells[3 * n + 2] = lod;
        out_dists[2 * n] = d.dist.x; out_dists[2 * n + 1] = d.dist.y;
        n++;
        if (d.do_step(far_clip)) break;
    }
    return n;
}

/* Diagnostics: per-ray work distribution, ORC_RAY_STAT_FIELDS uint64 per flat ray index:
 * dda_steps, columns_nonempty, columns_entered, renarrows, runs_visited, spans_tested, spans_committed, spans_wrote,
 * px_voxel, px_sky. Pixels go to scratch rows. */
int orc_ray_stats(const orc_world* w, const orc_frame_setup* s, int32_t W, int32_t H, uint64_t* out, int32_t max_rays) {
    if (!w || !s || !out) return -1;
    SegCtx ctx[4]; int total;
    fill_segment_contexts(s, W, H, ctx, total);
    Cam cam = make_cam(s->camera);
    int n = total < max_rays ? total : max_rays;
    int nt = orc_hardware_threads();
    std::vector<std::vector<uint8_t>> seen((size_t)nt);
    std::vector<std::vector<uint32_t>> scratch((size_t)nt);
    parallel_for(n, nt, [&](int i, int t) {
        Counters cn;
        RayCont rc;
        scratch[t].resize((size_t)(W > H ? W : H));
        if (setup_ray(w, s, ctx, cam, nullptr, nullptr, W, H, i, rc, cn, false, nullptr)) {
            rc.rayColumn = scratch[t].data();
            execute_ray(w, ctx[rc.segment], cam, rc, cam.inverse ? -1 : 1, seen[t], cn);
        }
        uint64_t* o = out + (size_t)i * ORC_RAY_STAT_FIELDS;
        o[0] = cn.dda_steps; o[1] = cn.columns_nonempty; o[2] = cn.columns_entered; o[3] = cn.renarrows; o[4] = cn.runs_visited;
        o[5] = cn.spans_tested; o[6] = cn.spans_committed; o[7] = cn.spans_wrote; o[8] = cn.px_voxel; o[9] = cn.px_sky;
    });
    return total;
}

/*
 * Phase 2: BlitSegments (RenderManager.cs:199-256) + RayBufferBlit.shader frag (Shaders/RayBufferBlit.shader:55-62),
 * restated per pixel centre (x+0.5, y+0.5), bottom-left origin. Triangle k = (VP, MaxScreen_k, MinScreen_k) with
 * attributes uv=(0,0),(1,0),(0,1): uv.x/uv.y are the affine barycentric weights of Max/Min. The GPU rasteriser's
 * coverage and interpolation bits are not reproducible; this formula is the parity target (SURVEY.md §8 a18):
 *   pixel belongs to the first segment k (RayCount > 0) whose weights are both >= 0, else to the one with the
 *   largest min(weight); t = b/(b+c); row = clamp(floor((offset_k + t*scale_k) * bufferRows), segment rows);
 *   column = y (top/down buffer) or x (left/right buffer); point sampling.
 */
int orc_blit(const orc_frame_setup* s, int32_t W, int32_t H, const uint32_t* td, const uint32_t* lr, uint32_t* frame,
             int32_t row_begin, int32_t row_end, int32_t n_threads) {
    if (!s || !td || !lr || !frame) return -1;
    if (row_begin < 0) row_begin = 0;
    if (row_end < 0 || row_end > H) row_end = H;
    const float vx = s->vanishing_point_screen[0], vy = s->vanishing_point_screen[1];
    const int tdRows = W + 2 * H, lrRows = 2 * W + H;
    float scale[4], offset[4];
    for (int k = 0; k < 4; k++) scale[k] = (float)s->segments[k].ray_count / (float)(k < 2 ? tdRows : lrRows);
    offset[0] = 0.0f; offset[1] = scale[0]; offset[2] = 0.0f; offset[3] = scale[2];
    int rowOff[4] = {0, s->segments[0].ray_count, 0, s->segments[2].ray_count};
    parallel_for(row_end - row_begin, n_threads, [&](int yi, int) {
        int y = row_begin + yi;
        float py = (float)y + 0.5f;
        for (int x = 0; x < W; x++) {
            float px = (float)x + 0.5f;
            int best = -1; float bestB = 0, bestC = 0, bestScore = -INFINITY;
            for (int k = 0; k < 4; k++) {
                const orc_segment& sg = s->segments[k];
                if (sg.ray_count <= 0) continue;
                float e1x = sg.max_screen[0] - vx, e1y = sg.max_screen[1] - vy; // VP -> Max (weight b)
                float e2x = sg.min_screen[0] - vx, e2y = sg.min_screen[1] - vy; // VP -> Min (weight c)
                float dx = px - vx, dy = py - vy;
                float det = e1x * e2y - e1y * e2x;
                // The interpolated uv.x, uv.y of the shader are the affine weights nb/det, nc/det; x = uv.x / (uv.x + uv.y) (shader :55)
                // does not depend on the common factor 1/det, so the weights are kept unnormalised (signs as for det > 0).
                float nb = dx * e2y - dy * e2x, nc = e1x * dy - e1y * dx;
                if (det < 0.0f) { nb = -nb; nc = -nc; }
                if (nb >= 0.0f && nc >= 0.0f) { best = k; bestB = nb; bestC = nc; break; }
                float score = m_min(nb, nc) / fabsf(det);  // outside every triangle (rounding on an outer edge): the nearest one
                if (score > bestScore) { bestScore = score; best = k; bestB = nb; bestC = nc; }
            }
            uint32_t color = 0;
            if (best >= 0) {
                float t = bestB / (bestB + bestC);
                float v = offset[best] + t * scale[best];
                int rows = best < 2 ? tdRows : lrRows;
                int row = f2i(floorf(v * (float)rows));
                int rc = s->segments[best].ray_count;
                row = i_clamp(row, rowOff[best], rowOff[best] + rc - 1);
                color = best < 2 ? td[(int64_t)row * H + y] : lr[(int64_t)row * W + x];
            }
            frame[(int64_t)y * W + x] = color;
        }
    });
    return 0;
}

/*
 * Debug views: RayBufferBlit.shader frag, COPY_MAIN1 / COPY_MAIN2 variants (Shaders/RayBufferBlit.shader:48-53):
 *   uv = SV_POSITION.xy / _ScreenParams.xy  (pixel centre, y from the TOP: D3D, SURVEY.md A12)
 *   return tex2D(buffer, float2(1 - uv.y, uv.x))   point filtered (RayBuffer.cs:32), clamp addressing
 * Texture x runs along one ray row (row_len texels), texture y over the ray rows. Frame rows are bottom-up like orc_blit's.
 */
int orc_blit_raybuffer(const uint32_t* buf, int32_t rows, int32_t row_len, int32_t W, int32_t H, uint32_t* frame) {
    if (!buf || !frame || rows < 1 || row_len < 1 || W < 1 || H < 1) return -1;
    for (int y = 0; y < H; y++) {
        for (int x = 0; x < W; x++) {
            float vx = (float)x + 0.5f, vy = (float)H - ((float)y + 0.5f);
            float uvx = vx / (float)W, uvy = vy / (float)H;
            float tu = 1.0f - uvy, tv = uvx;
            int col = i_clamp(f2i(floorf(tu * (float)row_len)), 0, row_len - 1);
            int row = i_clamp(f2i(floorf(tv * (float)rows)), 0, rows - 1);
            frame[(int64_t)y * W + x] = buf[(int64_t)row * row_len + col];
        }
    }
    return 0;
}

} // extern "C"
