/*
 * host_setup.cpp — host-side (CPU) mirror of the managed code around the hot path, for hosts without
 * UnityEngine (tests, bench, headless servers). A Unity host keeps RenderManager's own C# for these and
 * only calls the device entry points.
 *
 * Mirrors: RenderManager.CalculateVanishingPointWorld / ProjectVanishingPointScreenToWorld /
 * GetGenericSegmentParameters (Assets/Code/RenderManager.cs:374-501), the DrawWorld segment selection
 * (:128-142), CameraData ctor (Assets/Code/Utils/CameraData.cs:18-36), UnityManager.SetupLods /
 * LimitRotationHorizon (Assets/Code/UnityManager.cs:193-201,417-458) and the BenchmarkPath.anim sampler
 * (Assets/Code/BenchmarkPath.anim:16-152, UnityManager.cs:86-87).
 *
 * UnityEngine/Unity.Mathematics behaviour is restated from documentation (SURVEY.md Appendix A): GL-convention
 * projection, worldToCamera = Scale(1,1,-1)*inverse(TRS), LookAt basis, SignedAngle, half-to-even rounding.
 * All arithmetic is fp32 with a fixed evaluation order (built with -ffp-contract=off) so that the values
 * handed to the device are reproducible bit for bit.
 */
#include "nvtx_ranges.h"
#include "../../include/cpuvox_b200.h"

#include <climits>
#include <cmath>
#include <cstring>

namespace {

struct Vec2 { float v[2]; float& operator[](int i) { return v[i]; } float operator[](int i) const { return v[i]; } };
struct Vec3 { float x, y, z; };
struct Vec4 { float x, y, z, w; };
struct Quat { float x, y, z, w; };

// 4x4 stored as columns (float4x4 c0..c3); at(r,c) addresses row r of column c.
struct Mat4 {
    float col[4][4];
    float& at(int r, int c) { return col[c][r]; }
    float at(int r, int c) const { return col[c][r]; }
    static Mat4 zero() { Mat4 m; memset(&m, 0, sizeof m); return m; }
    static Mat4 identity() { Mat4 m = zero(); for (int i = 0; i < 4; i++) m.at(i, i) = 1.0f; return m; }
    static Mat4 scale(float x, float y, float z) { Mat4 m = identity(); m.at(0, 0) = x; m.at(1, 1) = y; m.at(2, 2) = z; return m; }
    static Mat4 translate(float x, float y, float z) { Mat4 m = identity(); m.at(0, 3) = x; m.at(1, 3) = y; m.at(2, 3) = z; return m; }
};

// mul(M, v) = c0*v.x + c1*v.y + c2*v.z + c3*v.w, summed left to right
Vec4 transform(const Mat4& m, Vec4 v) {
    float out[4];
    for (int r = 0; r < 4; r++) out[r] = m.at(r, 0) * v.x + m.at(r, 1) * v.y + m.at(r, 2) * v.z + m.at(r, 3) * v.w;
    return {out[0], out[1], out[2], out[3]};
}
Mat4 concat(const Mat4& a, const Mat4& b) { // mul(a, b): column j of the result is a * (column j of b)
    Mat4 m;
    for (int j = 0; j < 4; j++) {
        Vec4 c = transform(a, Vec4{b.col[j][0], b.col[j][1], b.col[j][2], b.col[j][3]});
        m.col[j][0] = c.x; m.col[j][1] = c.y; m.col[j][2] = c.z; m.col[j][3] = c.w;
    }
    return m;
}
// General 4x4 inverse, classical adjugate over the flattened column-major array, fp32.
Mat4 invert(const Mat4& src) {
    const float* m = &src.col[0][0];
    float a[16];
    a[0]  =  m[5]*m[10]*m[15] - m[5]*m[11]*m[14] - m[9]*m[6]*m[15] + m[9]*m[7]*m[14] + m[13]*m[6]*m[11] - m[13]*m[7]*m[10];
    a[4]  = -m[4]*m[10]*m[15] + m[4]*m[11]*m[14] + m[8]*m[6]*m[15] - m[8]*m[7]*m[14] - m[12]*m[6]*m[11] + m[12]*m[7]*m[10];
    a[8]  =  m[4]*m[9]*m[15]  - m[4]*m[11]*m[13] - m[8]*m[5]*m[15] + m[8]*m[7]*m[13] + m[12]*m[5]*m[11] - m[12]*m[7]*m[9];
    a[12] = -m[4]*m[9]*m[14]  + m[4]*m[10]*m[13] + m[8]*m[5]*m[14] - m[8]*m[6]*m[13] - m[12]*m[5]*m[10] + m[12]*m[6]*m[9];
    a[1]  = -m[1]*m[10]*m[15] + m[1]*m[11]*m[14] + m[9]*m[2]*m[15] - m[9]*m[3]*m[14] - m[13]*m[2]*m[11] + m[13]*m[3]*m[10];
    a[5]  =  m[0]*m[10]*m[15] - m[0]*m[11]*m[14] - m[8]*m[2]*m[15] + m[8]*m[3]*m[14] + m[12]*m[2]*m[11] - m[12]*m[3]*m[10];
    a[9]  = -m[0]*m[9]*m[15]  + m[0]*m[11]*m[13] + m[8]*m[1]*m[15] - m[8]*m[3]*m[13] - m[12]*m[1]*m[11] + m[12]*m[3]*m[9];
    a[13] =  m[0]*m[9]*m[14]  - m[0]*m[10]*m[13] - m[8]*m[1]*m[14] + m[8]*m[2]*m[13] + m[12]*m[1]*m[10] - m[12]*m[2]*m[9];
    a[2]  =  m[1]*m[6]*m[15]  - m[1]*m[7]*m[14]  - m[5]*m[2]*m[15] + m[5]*m[3]*m[14] + m[13]*m[2]*m[7]  - m[13]*m[3]*m[6];
    a[6]  = -m[0]*m[6]*m[15]  + m[0]*m[7]*m[14]  + m[4]*m[2]*m[15] - m[4]*m[3]*m[14] - m[12]*m[2]*m[7]  + m[12]*m[3]*m[6];
    a[10] =  m[0]*m[5]*m[15]  - m[0]*m[7]*m[13]  - m[4]*m[1]*m[15] + m[4]*m[3]*m[13] + m[12]*m[1]*m[7]  - m[12]*m[3]*m[5];
    a[14] = -m[0]*m[5]*m[14]  + m[0]*m[6]*m[13]  + m[4]*m[1]*m[14] - m[4]*m[2]*m[13] - m[12]*m[1]*m[6]  + m[12]*m[2]*m[5];
    a[3]  = -m[1]*m[6]*m[11]  + m[1]*m[7]*m[10]  + m[5]*m[2]*m[11] - m[5]*m[3]*m[10] - m[9]*m[2]*m[7]   + m[9]*m[3]*m[6];
    a[7]  =  m[0]*m[6]*m[11]  - m[0]*m[7]*m[10]  - m[4]*m[2]*m[11] + m[4]*m[3]*m[10] + m[8]*m[2]*m[7]   - m[8]*m[3]*m[6];
    a[11] = -m[0]*m[5]*m[11]  + m[0]*m[7]*m[9]   + m[4]*m[1]*m[11] - m[4]*m[3]*m[9]  - m[8]*m[1]*m[7]   + m[8]*m[3]*m[5];
    a[15] =  m[0]*m[5]*m[10]  - m[0]*m[6]*m[9]   - m[4]*m[1]*m[10] + m[4]*m[2]*m[9]  + m[8]*m[1]*m[6]   - m[8]*m[2]*m[5];
    float det = m[0]*a[0] + m[1]*a[4] + m[2]*a[8] + m[3]*a[12];
    float inv_det = 1.0f / det;
    Mat4 out;
    float* o = &out.col[0][0];
    for (int i = 0; i < 16; i++) o[i] = a[i] * inv_det;
    return out;
}

const float kDeg2Rad = 0.017453292f;
const float kRad2Deg = 57.29578f;

inline float mix(float a, float b, float t) { return a + t * (b - a); }
inline float sgn(float x) { return (float)((x > 0.0f) - (x < 0.0f)); }            // math.sign: sign(0) = 0
inline float mathf_sign(float x) { return x >= 0.0f ? 1.0f : -1.0f; }            // Mathf.Sign: sign(0) = +1
inline int to_int(float f) { return (f >= -2147483648.0f && f < 2147483648.0f) ? (int)f : INT_MIN; }
inline int round_to_int(float f) { return to_int(rintf(f)); }                     // Mathf.RoundToInt: half-to-even

inline float dot3(Vec3 a, Vec3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
inline Vec3 cross3(Vec3 a, Vec3 b) { return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }
inline Vec3 unit(Vec3 a) { // Vector3.Normalize
    float len = sqrtf(dot3(a, a));
    if (len > 1e-5f) return {a.x / len, a.y / len, a.z / len};
    return {0, 0, 0};
}

Quat qmul(Quat a, Quat b) {
    return {a.w * b.x + a.x * b.w + a.y * b.z - a.z * b.y,
            a.w * b.y + a.y * b.w + a.z * b.x - a.x * b.z,
            a.w * b.z + a.z * b.w + a.x * b.y - a.y * b.x,
            a.w * b.w - a.x * b.x - a.y * b.y - a.z * b.z};
}
Vec3 rotate(Quat q, Vec3 p) { // Quaternion * Vector3
    float x2 = q.x * 2.0f, y2 = q.y * 2.0f, z2 = q.z * 2.0f;
    float xx = q.x * x2, yy = q.y * y2, zz = q.z * z2, xy = q.x * y2, xz = q.x * z2, yz = q.y * z2;
    float wx = q.w * x2, wy = q.w * y2, wz = q.w * z2;
    return {(1.0f - (yy + zz)) * p.x + (xy - wz) * p.y + (xz + wy) * p.z,
            (xy + wz) * p.x + (1.0f - (xx + zz)) * p.y + (yz - wx) * p.z,
            (xz - wy) * p.x + (yz + wx) * p.y + (1.0f - (xx + yy)) * p.z};
}

struct Basis { Vec3 right, up, forward; };
Basis look_basis(Vec3 fwd, Vec3 upHint) { // Matrix4x4.LookAt / Quaternion.LookRotation basis
    Basis b;
    b.forward = unit(fwd);
    b.right = unit(cross3(upHint, b.forward));
    b.up = cross3(b.forward, b.right);
    return b;
}
Mat4 basis_matrix(const Basis& b) {
    Mat4 m = Mat4::identity();
    m.at(0, 0) = b.right.x;   m.at(1, 0) = b.right.y;   m.at(2, 0) = b.right.z;
    m.at(0, 1) = b.up.x;      m.at(1, 1) = b.up.y;      m.at(2, 1) = b.up.z;
    m.at(0, 2) = b.forward.x; m.at(1, 2) = b.forward.y; m.at(2, 2) = b.forward.z;
    return m;
}
Quat basis_quat(const Basis& b) {
    float m00 = b.right.x, m01 = b.up.x, m02 = b.forward.x;
    float m10 = b.right.y, m11 = b.up.y, m12 = b.forward.y;
    float m20 = b.right.z, m21 = b.up.z, m22 = b.forward.z;
    float trace = m00 + m11 + m22;
    Quat q;
    if (trace > 0.0f) {
        float s = sqrtf(trace + 1.0f);
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

Mat4 gl_perspective(float fovY, float aspect, float zn, float zf) { // Camera.nonJitteredProjectionMatrix (A2)
    float cot = 1.0f / (float)tan((double)(fovY * kDeg2Rad * 0.5f));
    Mat4 m = Mat4::zero();
    m.at(0, 0) = cot / aspect;
    m.at(1, 1) = cot;
    m.at(2, 2) = -(zf + zn) / (zf - zn);
    m.at(2, 3) = -(2.0f * zf * zn) / (zf - zn);
    m.at(3, 2) = -1.0f;
    return m;
}
Mat4 view_matrix(Vec3 pos, Quat rot) { // Camera.worldToCameraMatrix (A3), rigid inverse written out
    Vec3 r = rotate(rot, Vec3{1, 0, 0}), u = rotate(rot, Vec3{0, 1, 0}), f = rotate(rot, Vec3{0, 0, 1});
    Mat4 m = Mat4::identity();
    m.at(0, 0) = r.x;  m.at(0, 1) = r.y;  m.at(0, 2) = r.z;  m.at(0, 3) = -dot3(r, pos);
    m.at(1, 0) = u.x;  m.at(1, 1) = u.y;  m.at(1, 2) = u.z;  m.at(1, 3) = -dot3(u, pos);
    m.at(2, 0) = -f.x; m.at(2, 1) = -f.y; m.at(2, 2) = -f.z; m.at(2, 3) = dot3(f, pos);
    return m;
}
float signed_angle(Vec2 a, Vec2 b) { // Vector2.SignedAngle (A5)
    float denom = sqrtf((a[0] * a[0] + a[1] * a[1]) * (b[0] * b[0] + b[1] * b[1]));
    float unsignedAngle = 0.0f;
    if (!(denom < 1e-15f)) {
        float c = (a[0] * b[0] + a[1] * b[1]) / denom;
        if (c < -1.0f) c = -1.0f; else if (c > 1.0f) c = 1.0f;
        unsignedAngle = (float)acos((double)c) * kRad2Deg;
    }
    return unsignedAngle * mathf_sign(a[0] * b[1] - a[1] * b[0]);
}

struct SegmentSolver {
    Vec2 vp, screen;
    Mat4 screenToLocal;
    int W, H;

    void unproject(Vec2 pixel, float out[2]) const { // TransformPixel, RenderManager.cs:487-500
        Vec4 v = transform(screenToLocal, Vec4{((pixel[0] / (float)W) - 0.5f) * 2.0f, ((pixel[1] / (float)H) - 0.5f) * 2.0f, 1.0f, 1.0f});
        out[0] = v.x / v.w; out[1] = v.z / v.w;
    }

    // GetGenericSegmentParameters, RenderManager.cs:402-485
    void solve(float distToOtherEnd, Vec2 neutral, int primary, cvx_segment* seg) const {
        memset(seg, 0, sizeof *seg);
        const int secondary = 1 - primary;
        Vec2 simpleMin, simpleMax;
        simpleMin[0] = simpleMin[1] = vp[secondary] - distToOtherEnd;
        simpleMax[0] = simpleMax[1] = vp[secondary] + distToOtherEnd;
        float far_edge = vp[primary] + distToOtherEnd * sgn(neutral[primary]);
        simpleMin[primary] = far_edge; simpleMax[primary] = far_edge;
        if (simpleMax[secondary] <= 0.0f || simpleMin[secondary] >= screen[secondary]) return; // 45-degree rays miss the screen

        Vec2 lo, hi;
        bool vpOnScreen = vp[0] >= 0.0f && vp[1] >= 0.0f && vp[0] <= screen[0] && vp[1] <= screen[1];
        if (vpOnScreen) { lo = simpleMin; hi = simpleMax; }
        else {
            Vec2 middleDir = {{mix(simpleMin[0], simpleMax[0], 0.5f) - vp[0], mix(simpleMin[1], simpleMax[1], 0.5f) - vp[1]}};
            float angleLeft = 90.0f, angleRight = -90.0f;
            Vec2 dirLeft = {{0, 0}}, dirRight = {{0, 0}};
            const Vec2 corners[4] = {{{0.0f, 0.0f}}, {{0.0f, screen[1]}}, {{screen[0], 0.0f}}, {{screen[0], screen[1]}}};
            for (int i = 0; i < 4; i++) {
                Vec2 dir = {{corners[i][0] - vp[0], corners[i][1] - vp[1]}};
                float k = distToOtherEnd / fabsf(dir[primary]);
                Vec2 scaledEnd = {{dir[0] * k, dir[1] * k}};
                float angle = signed_angle(neutral, dir);
                if (angle < angleLeft) { angleLeft = angle; dirLeft = scaledEnd; }
                if (angle > angleRight) { angleRight = angle; dirRight = scaledEnd; }
            }
            Vec2 cornerLeft = {{dirLeft[0] + vp[0], dirLeft[1] + vp[1]}};
            Vec2 cornerRight = {{dirRight[0] + vp[0], dirRight[1] + vp[1]}};
            // the reference passes the *point* simpleCaseMax as a direction here (:466,:469); kept as is
            if (angleLeft < -45.0f) cornerLeft = signed_angle(middleDir, simpleMax) > 0.0f ? simpleMin : simpleMax;
            if (angleRight > 45.0f) cornerRight = signed_angle(middleDir, simpleMax) < 0.0f ? simpleMin : simpleMax;
            bool swapped = cornerLeft[secondary] > cornerRight[secondary];
            lo = swapped ? cornerRight : cornerLeft;
            hi = swapped ? cornerLeft : cornerRight;
        }
        seg->min_screen[0] = lo[0]; seg->min_screen[1] = lo[1];
        seg->max_screen[0] = hi[0]; seg->max_screen[1] = hi[1];
        unproject(lo, seg->cam_local_plane_ray_min);
        unproject(hi, seg->cam_local_plane_ray_max);
        int rays = round_to_int(hi[secondary] - lo[secondary]);
        seg->ray_count = rays > 0 ? rays : 0;
    }
};

// ScreenPointToRay in camera space (A8): the point of pixel (px, py) on the plane z = 1, i.e. the unnormalised direction
Vec3 camera_ray(float px, float py, int W, int H, float aspect, float tanHalf) {
    return Vec3{(2.0f * px / W - 1.0f) * aspect * tanHalf, (2.0f * py / H - 1.0f) * tanHalf, 1.0f};
}

struct CurveKey { float time; float value[3]; float inSlope[3]; float outSlope[3]; };

// Non-weighted AnimationCurve segment: cubic Hermite (A9)
void sample_curve(const CurveKey* keys, int n, float t, float out[3]) {
    if (t <= keys[0].time) { memcpy(out, keys[0].value, sizeof(float) * 3); return; }
    if (t >= keys[n - 1].time) { memcpy(out, keys[n - 1].value, sizeof(float) * 3); return; }
    int i = 0;
    while (i + 1 < n && t > keys[i + 1].time) i++;
    const CurveKey& k0 = keys[i];
    const CurveKey& k1 = keys[i + 1];
    float dt = k1.time - k0.time;
    float s = (t - k0.time) / dt;
    float s2 = s * s, s3 = s2 * s;
    float h00 = 2 * s3 - 3 * s2 + 1, h10 = s3 - 2 * s2 + s, h01 = -2 * s3 + 3 * s2, h11 = s3 - s2;
    for (int c = 0; c < 3; c++)
        out[c] = h00 * k0.value[c] + h10 * k0.outSlope[c] * dt + h01 * k1.value[c] + h11 * k1.inSlope[c] * dt;
}

// Assets/Code/BenchmarkPath.anim m_EulerCurves (:16-82) and m_PositionCurves (:89-146)
const CurveKey kEulerKeys[7] = {
    {0.0f,   {0.0f, 45.0f, 0.0f},       {0, 0, 0},    {0, 0, 0}},
    {0.25f,  {0.0f, -45.0f, 0.0f},      {0, -360, 0}, {0, -360, 0}},
    {0.5f,   {-16.2f, -135.0f, 0.0f},   {0, 0, 0},    {0, 0, 0}},
    {0.75f,  {59.12f, -135.0f, 0.0f},   {0, 0, 0},    {0, 0, 0}},
    {0.875f, {59.12f, -135.0f, 180.0f}, {0, 0, 1440}, {0, 0, 1440}},
    {1.0f,   {59.12f, -135.0f, 360.0f}, {0, 0, 0},    {0, 0, 0}},
    {1.15f,  {85.0f, -225.5f, 360.0f},  {0, 0, 0},    {0, 0, 0}},
};
const CurveKey kPositionKeys[6] = {
    {0.0f,  {-0.1f, 0.5f, -0.1f},   {0, 0, 0}, {0, 0, 0}},
    {0.25f, {1.1f, 0.5f, -0.1f},    {0, 0, 0}, {0, 0, 0}},
    {0.5f,  {0.9f, 0.3f, 0.9f},     {0, 0, 0}, {0, 0, 0}},
    {0.75f, {0.9f, 0.95f, 0.9f},    {0, 0, 0}, {0, 0, 0}},
    {1.0f,  {0.9f, 0.95f, 0.9f},    {0, 0, 0}, {0, 0, 0}},
    {1.15f, {0.427f, 0.95f, 0.52f}, {0, 0, 0}, {0, 0, 0}},
};

} // namespace

extern "C" {

// Quaternion.Euler(x,y,z): Z, then X, then Y => qY*qX*qZ
void cvx_host_quat_euler(float x_deg, float y_deg, float z_deg, float out_quat[4]) {
    float hx = x_deg * kDeg2Rad * 0.5f, hy = y_deg * kDeg2Rad * 0.5f, hz = z_deg * kDeg2Rad * 0.5f;
    Quat qx = {(float)sin((double)hx), 0, 0, (float)cos((double)hx)};
    Quat qy = {0, (float)sin((double)hy), 0, (float)cos((double)hy)};
    Quat qz = {0, 0, (float)sin((double)hz), (float)cos((double)hz)};
    Quat q = qmul(qmul(qy, qx), qz);
    out_quat[0] = q.x; out_quat[1] = q.y; out_quat[2] = q.z; out_quat[3] = q.w;
}

void cvx_host_limit_rotation_horizon(cvx_pose* pose) {
    Quat q = {pose->rotation[0], pose->rotation[1], pose->rotation[2], pose->rotation[3]};
    Vec3 forward = rotate(q, Vec3{0, 0, 1});
    if (fabsf(forward.y) < 0.001f) {
        forward.y = mathf_sign(forward.y) * 0.001f;
        Quat r = basis_quat(look_basis(forward, Vec3{0, 1, 0})); // transform.forward = v  =>  LookRotation(v, up)
        pose->rotation[0] = r.x; pose->rotation[1] = r.y; pose->rotation[2] = r.z; pose->rotation[3] = r.w;
    }
}

void cvx_host_setup_lods(int32_t world_max_dimension, int32_t res_x, int32_t res_y, float fov_y_degrees, float lod_error,
                         float out_lod_distances[CVX_LOD_LEVELS]) {
    const float clipMax = (float)(world_max_dimension * 2); // REPEAT_WORLD == false => multiplier 2
    const float pixelW = (1.0f / res_x) * res_x, pixelH = (1.0f / res_y) * res_y;
    const int midW = res_x / 2, midH = res_y / 2;
    const float tanHalf = (float)tan((double)(fov_y_degrees * kDeg2Rad * 0.5f));
    const float aspect = (float)res_x / (float)res_y;
    auto ray_dir = [&](float px, float py) { return unit(camera_ray(px, py, res_x, res_y, aspect, tanHalf)); };
    const Vec3 a = ray_dir((float)midW, (float)midH), b = ray_dir(midW + pixelW, midH + pixelH);
    bool found[CVX_LOD_LEVELS] = {false};
    float at[CVX_LOD_LEVELS] = {0};
    const float pixelWidth = 1.41f / lod_error;
    for (float p = 0.0f; p < 1.0f; p += 0.0001f) {
        float rayDist = p * clipMax;
        Vec3 pa = {a.x * rayDist, a.y * rayDist, a.z * rayDist}, pb = {b.x * rayDist, b.y * rayDist, b.z * rayDist};
        Vec3 d = {pa.x - pb.x, pa.y - pb.y, pa.z - pb.z};
        float gap = sqrtf(dot3(d, d));
        for (int j = 0; j < CVX_LOD_LEVELS; j++)
            if (!found[j] && gap > pixelWidth * (float)(2 << j)) { found[j] = true; at[j] = p; }
    }
    found[CVX_LOD_LEVELS - 1] = true; at[CVX_LOD_LEVELS - 1] = 2.0f; // last LOD never ends
    for (int i = 0; i < CVX_LOD_LEVELS; i++) out_lod_distances[i] = ceilf((found[i] ? at[i] : 2.0f) * clipMax);
}

void cvx_host_screen_ray(const cvx_pose* pose, float px, float py, float out_origin[3], float out_direction[3]) {
    const float tanHalf = (float)tan((double)(pose->fov_y_degrees * kDeg2Rad * 0.5f));
    const float aspect = (float)pose->pixel_width / (float)pose->pixel_height;
    const Quat rot = {pose->rotation[0], pose->rotation[1], pose->rotation[2], pose->rotation[3]};
    const Vec3 cam = camera_ray(px, py, pose->pixel_width, pose->pixel_height, aspect, tanHalf);
    const Vec3 onNear = rotate(rot, Vec3{cam.x * pose->near_clip, cam.y * pose->near_clip, pose->near_clip});
    const Vec3 dir = rotate(rot, unit(cam));
    out_origin[0] = pose->position[0] + onNear.x; out_origin[1] = pose->position[1] + onNear.y; out_origin[2] = pose->position[2] + onNear.z;
    out_direction[0] = dir.x; out_direction[1] = dir.y; out_direction[2] = dir.z;
}

int cvx_host_frame_setup(const cvx_pose* pose, const float lod_distances[CVX_LOD_LEVELS], int32_t world_dim_y, cvx_frame_setup* out) {
    (void)world_dim_y;
    if (!pose || !lod_distances || !out || pose->pixel_width < 1 || pose->pixel_height < 1) return CVX_ERR_INVALID_ARGUMENT;
    CVX_RANGE("Setup VP + segment params");  // RenderManager.cs:119,127
    memset(out, 0, sizeof *out);
    const int W = pose->pixel_width, H = pose->pixel_height;
    const Quat rot = {pose->rotation[0], pose->rotation[1], pose->rotation[2], pose->rotation[3]};
    const Vec3 pos = {pose->position[0], pose->position[1], pose->position[2]};
    const Vec3 forward = rotate(rot, Vec3{0, 0, 1}), up = rotate(rot, Vec3{0, 1, 0});
    const Mat4 proj = gl_perspective(pose->fov_y_degrees, (float)W / (float)H, pose->near_clip, pose->far_clip);

    // vanishing point: the world point straight below/above the camera on the near plane (RenderManager.cs:374-378),
    // projected through a camera-local view matrix (:380-394)
    const float vpOffset = pose->near_clip / forward.y; // -near / sin(eulerAngles.x), sin(pitch) = -forward.y (A6)
    const Vec3 vpWorld = {pos.x + 0.0f * vpOffset, pos.y + 1.0f * vpOffset, pos.z + 0.0f * vpOffset};
    const Vec3 vpLocal = {vpWorld.x - pos.x, vpWorld.y - pos.y, vpWorld.z - pos.z};
    const Mat4 look = basis_matrix(look_basis(forward, up));
    const Mat4 localView = concat(Mat4::scale(1, 1, -1), invert(look));
    const Mat4 localToScreen = concat(proj, localView);
    const Vec4 clip = transform(localToScreen, Vec4{vpLocal.x, vpLocal.y, vpLocal.z, 1.0f});

    SegmentSolver solver;
    solver.W = W; solver.H = H;
    solver.screen = {{(float)W, (float)H}};
    solver.vp = {{((clip.x / clip.w) * 0.5f + 0.5f) * (float)W, ((clip.y / clip.w) * 0.5f + 0.5f) * (float)H}};
    Mat4 s2l = invert(proj);
    s2l = concat(invert(Mat4::scale(1, 1, -1)), s2l);
    solver.screenToLocal = concat(look, s2l);
    out->vanishing_point_screen[0] = solver.vp[0];
    out->vanishing_point_screen[1] = solver.vp[1];

    // DrawWorld's four quadrant calls, RenderManager.cs:128-142
    if (solver.vp[1] < solver.screen[1]) solver.solve(solver.screen[1] - solver.vp[1], Vec2{{0, 1}}, 1, &out->segments[0]);
    if (solver.vp[1] > 0.0f)             solver.solve(solver.vp[1], Vec2{{0, -1}}, 1, &out->segments[1]);
    if (solver.vp[0] < solver.screen[0]) solver.solve(solver.screen[0] - solver.vp[0], Vec2{{1, 0}}, 0, &out->segments[2]);
    if (solver.vp[0] > 0.0f)             solver.solve(solver.vp[0], Vec2{{-1, 0}}, 0, &out->segments[3]);

    // CameraData ctor, CameraData.cs:18-36
    Mat4 wts = concat(proj, view_matrix(pos, rot));
    wts = concat(Mat4::scale(0.5f, 0.5f, 1.0f), wts);
    wts = concat(Mat4::translate(0.5f, 0.5f, 1.0f), wts);
    wts = concat(Mat4::scale((float)W, (float)H, 1.0f), wts);
    memcpy(out->camera.world_to_screen, &wts.col[0][0], sizeof(float) * 16);
    out->camera.position_xz[0] = pos.x;
    out->camera.position_xz[1] = pos.z;
    out->camera.position_y = pos.y;
    out->camera.inverse_element_iteration_direction = forward.y >= 0.0f ? 1 : 0;
    out->camera.far_clip = pose->far_clip;
    memcpy(out->camera.lod_distances, lod_distances, sizeof(float) * CVX_LOD_LEVELS);
    return CVX_OK;
}

float cvx_host_benchmark_length(void) { return 1.15f; }

void cvx_host_benchmark_pose(float clip_time, const int32_t world_dims[3], cvx_pose* inout_pose) {
    float euler[3], position[3];
    sample_curve(kEulerKeys, 7, clip_time, euler);
    sample_curve(kPositionKeys, 6, clip_time, position);
    for (int i = 0; i < 3; i++) inout_pose->position[i] = position[i] * (float)world_dims[i]; // UnityManager.cs:87
    cvx_host_quat_euler(euler[0], euler[1], euler[2], inout_pose->rotation);
}

} // extern "C"
