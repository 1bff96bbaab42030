"""TEST INFRASTRUCTURE — second, independent restatement of the reference's Phase 1 in pure Python (numpy float32 scalars).

Written by reading the C# only (not the C++ oracle), statement by statement, so that a transcription slip in
oracle/cpuvox_oracle.cpp shows up as a disagreement between two restatements (tests/test_oracle.py::test_python_restatement_agrees).
It is slow (seconds per small frame) and is used on small worlds and resolutions only. Nothing in the product imports it.

Follows, with the reference line numbers under /root/reference/Assets/Code:
  RenderManager.DrawSegments context fill          RenderManager.cs:281-318
  RaySetupJob / DDASetupJob / TraceToFirstColumn   Rendering/DrawSegmentRayJob.cs:12-144
  ExecuteRay                                       Rendering/DrawSegmentRayJob.cs:195-620
  SetupProjectedPlaneParams, ReducePixelHorizon,
  WriteSkybox(Full)                                Rendering/DrawSegmentRayJob.cs:622-716
  SegmentDDAData                                   Utils/SegmentDDAData.cs:17-155
  CameraData clip/projection helpers               Utils/CameraData.cs:38-163
  World.GetVoxelColumn, RLEColumn, RLEElement      World.cs:130-149,161-188,245-259
Unity.Mathematics semantics as listed in SURVEY.md Appendix A1 (lerp = a + t*(b-a), unlerp = (x-a)/(b-a), round = half to even,
sign(0) = 0, normalize = v * (1/sqrt(dot)), mul(M, v) = c0*x + c1*y + c2*z + c3*w, (int)float truncates)."""
from __future__ import annotations

import numpy as np

F = np.float32
EPSILON = np.array([1], dtype=np.uint32).view(np.float32)[0]   # float.Epsilon: the smallest denormal
NEG_INF, POS_INF = F(-np.inf), F(np.inf)
SKYBOX = np.uint32(0x191919FF)   # ColorARGB32(25, 25, 25): bytes a=255, r, g, b
INT_MIN = -2147483648


def to_int(f) -> int:
    """(int)float on x64 (cvttss2si): truncation, INT_MIN for NaN / out of range."""
    f = F(f)
    if not (f > F(-2147483904.0) and f < F(2147483648.0)):
        return INT_MIN
    return int(np.trunc(f))


def lerp(a, b, t):
    return a + t * (b - a)


def unlerp(a, b, x):
    return (x - a) / (b - a)


def umin(x, y):
    """math.min as the reference build pins it (Unity.Mathematics): isnan(y) || x < y ? x : y. A NaN y gives x, a tie (±0) gives y."""
    return x if (np.isnan(y) or x < y) else y


def umax(x, y):
    """math.max: isnan(y) || x > y ? x : y."""
    return x if (np.isnan(y) or x > y) else y


def sign(x):
    return F(1.0) if x > F(0) else (F(-1.0) if x < F(0) else F(0.0))


def lerp3(a, b, t):
    return (lerp(a[0], b[0], t), lerp(a[1], b[1], t), lerp(a[2], b[2], t))


# ---- World (read side) -------------------------------------------------------------------------------------------------------
class PyWorldLod:
    def __init__(self, dims, lod, blob, column_count):
        self.dims, self.lod = dims, lod
        words = np.frombuffer(np.ascontiguousarray(blob).tobytes(), dtype=np.uint32)
        self.headers = words[:3 * column_count].reshape(column_count, 3)
        self.cells = words[3 * column_count:]
        self.indexing_mul_x = dims[2] >> lod                      # World.cs:31
        self.mask = (dims[0] - 1, dims[2] - 1)                     # dimensionMaskXZ, World.cs:32

    def get_voxel_column(self, px, pz):                            # World.cs:130-142
        if (px & self.mask[0]) != px or (pz & self.mask[1]) != pz:
            return -1, None
        idx = (px >> self.lod) * self.indexing_mul_x + (pz >> self.lod)   # GetIndexKnownInBounds :145-149
        off, w1, w2 = (int(v) for v in self.headers[idx])
        return w1 & 0xFFFF, (off, w1 & 0xFFFF, w1 >> 16, w2 & 0xFFFF)    # runCount, (storage offset, runCount, worldMin, worldMax)

    def element(self, cell_index):                                 # RLEElement {short ColorsIndex; short Length} World.cs:245-259
        e = int(self.cells[cell_index])
        ci, ln = e & 0xFFFF, (e >> 16) & 0xFFFF
        return (ci - 0x10000 if ci >= 0x8000 else ci), (ln - 0x10000 if ln >= 0x8000 else ln)


# ---- SegmentDDAData ----------------------------------------------------------------------------------------------------------
class DDA:
    def __init__(self, start, direction):                          # SegmentDDAData.cs:17-28
        self.start, self.dir = (F(start[0]), F(start[1])), (F(direction[0]), F(direction[1]))
        fl = (np.floor(self.start[0]), np.floor(self.start[1]))
        self.position = [to_int(fl[0]), to_int(fl[1])]
        self.t_delta = [F(1.0) / umax(F(0.0000001), abs(self.dir[0])), F(1.0) / umax(F(0.0000001), abs(self.dir[1]))]
        sd = (sign(self.dir[0]), sign(self.dir[1]))
        self.step = [to_int(sd[0]), to_int(sd[1])]
        frac = (self.start[0] - fl[0], self.start[1] - fl[1])
        self.t_max = [(sd[k] * -frac[k] + (sd[k] * F(0.5)) + F(0.5)) * self.t_delta[k] for k in range(2)]
        self.dist = [umax(self.t_max[0] - self.t_delta[0], self.t_max[1] - self.t_delta[1]), umin(self.t_max[0], self.t_max[1])]

    def next_lod(self, size):                                      # :31-73
        rem = [self.position[0] & (size * 2 - 1), self.position[1] & (size * 2 - 1)]
        # a still axis entered from outside has t_max = +inf (step_to_world_intersection): its last crossing stays -inf
        prev = [self.t_max[k] - self.t_delta[k] if self.t_max[k] != POS_INF else NEG_INF for k in range(2)]
        for k in range(2):
            if self.dir[k] >= F(0):
                if rem[k] < size:
                    self.t_max[k] = self.t_max[k] + self.t_delta[k]
                else:
                    prev[k] = prev[k] - self.t_delta[k]
            else:
                if rem[k] < size:
                    prev[k] = prev[k] - self.t_delta[k]
                else:
                    self.t_max[k] = self.t_max[k] + self.t_delta[k]
        self.dist = [umax(prev[0], prev[1]), umin(self.t_max[0], self.t_max[1])]
        self.position = [self.position[0] - rem[0], self.position[1] - rem[1]]
        self.t_delta = [self.t_delta[0] * F(2.0), self.t_delta[1] * F(2.0)]
        self.step = [self.step[0] * 2, self.step[1] * 2]

    def step_to_world_intersection(self, dim_x, dim_z):            # :75-130
        dims = (F(dim_x), F(dim_z))
        with np.errstate(all="ignore"):
            inv = (F(1.0) / self.dir[0], F(1.0) / self.dir[1])
        tmin, tmax = [NEG_INF, NEG_INF], [POS_INF, POS_INF]
        for k in range(2):
            if self.dir[k] != F(0):
                t1 = -self.start[k] * inv[k]
                t2 = (dims[k] - self.start[k]) * inv[k]
                tmin[k], tmax[k] = umin(t1, t2), umax(t1, t2)
        tmint, tmaxt = umax(tmin[0], tmin[1]), umin(tmax[0], tmax[1])
        if tmaxt < tmint or tmint <= F(0):
            return False
        t_last = [F(0), F(0)]
        if tmin[0] < tmin[1] and tmin[0] != NEG_INF:
            a, o = 0, 1
        else:
            a, o = 1, 0
        t_last[o] = tmin[o]
        if self.dir[a] != F(0):
            offset = tmint * self.dir[a]
            hit = self.start[a] + offset
            hit = np.floor(hit) if self.dir[a] > F(0) else np.ceil(hit)
            offset = hit - self.start[a]
            t_last[a] = offset / self.dir[a]
        else:
            t_last[a] = NEG_INF
        # still-axis rule (DESIGN.md §5): an axis with dir == 0 never bounds the entry and is never crossed (t_last -inf, t_max +inf)
        self.t_max = [t_last[k] + self.t_delta[k] if self.dir[k] != F(0) else POS_INF for k in range(2)]
        self.dist = [umax(t_last[0], t_last[1]), umin(self.t_max[0], self.t_max[1])]
        mid = lerp(self.dist[0], self.dist[1], F(0.5))
        self.position = [to_int(np.floor(self.start[0] + mid * self.dir[0])), to_int(np.floor(self.start[1] + mid * self.dir[1]))]
        return True

    def do_step(self, farclip):                                    # :135-150
        if self.t_max[0] < self.t_max[1]:
            crossed = self.t_max[0]
            self.t_max[0] = self.t_max[0] + self.t_delta[0]
            self.position[0] += self.step[0]
        else:
            crossed = self.t_max[1]
            self.t_max[1] = self.t_max[1] + self.t_delta[1]
            self.position[1] += self.step[1]
        self.dist = [crossed, umin(self.t_max[0], self.t_max[1])]
        return crossed >= farclip

    def is_beyond_far_clip(self, farclip):                         # :152-155
        return umin(self.t_max[0], self.t_max[1]) >= farclip


# ---- CameraData helpers ------------------------------------------------------------------------------------------------------
def mul_m_v(m, x, y, z, w):
    """mul(float4x4, float4): c0*x + c1*y + c2*z + c3*w, column-major m (16 float32)."""
    return tuple(m[r] * x + m[4 + r] * y + m[8 + r] * z + m[12 + r] * w for r in range(4))


def _cross(ax, ay, bx, by):
    return ax * by - ay * bx


def _clip_min(p_min, p_max, frustum):                              # CameraData.cs:101-107
    inv = F(1.0) / frustum
    c0 = _cross(F(1.0), inv, p_max[0], p_max[2])
    c1 = _cross(F(1.0), inv, p_min[0], p_min[2])
    return F(1.0) - (c0 / (c0 - c1))


def _clip_max(p_min, p_max, frustum):                              # :109-115
    inv = F(1.0) / frustum
    c0 = _cross(F(1.0), inv, p_max[0], p_max[2])
    c1 = _cross(F(1.0), inv, p_min[0], p_min[2])
    return c1 / (c1 - c0)


def world_bounds_clipping(p_min, p_max, b_min, b_max):             # GetWorldBoundsClippingCamSpace :50-99 -> (clipped, minLerp, maxLerp)
    if p_min[0] > p_min[2] * b_max:
        if p_max[0] > p_max[2] * b_max:
            return True, F(0), F(1)
        mn = _clip_min(p_min, p_max, b_max)
        mx = _clip_max(p_min, p_max, b_min) if p_max[0] < p_max[2] * b_min else F(1)
        return False, mn, mx
    if p_max[0] > p_max[2] * b_max:
        mx = _clip_max(p_min, p_max, b_max)
        mn = _clip_min(p_min, p_max, b_min) if p_min[0] < p_min[2] * b_min else F(0)
        return False, mn, mx
    if p_min[0] < p_min[2] * b_min:
        if p_max[0] < p_max[2] * b_min:
            return True, F(0), F(1)
        return False, _clip_min(p_min, p_max, b_min), F(1)
    if p_max[0] < p_max[2] * b_min:
        return False, F(0), _clip_max(p_min, p_max, b_min)
    return False, F(0), F(1)


def clip_line(a, b, u_a=None, u_b=None):                           # ClipHomogeneousCameraSpaceLine :123-157 -> (ok, a, b, uA, uB)
    if a[1] <= F(0):
        if b[1] <= F(0):
            return False, a, b, u_a, u_b
        v = b[1] / (b[1] - a[1])
        a = lerp3(b, a, v)
        if u_a is not None:
            u_a = lerp(u_b, u_a, v)
    elif b[1] <= F(0):
        v = a[1] / (a[1] - b[1])
        b = lerp3(a, b, v)
        if u_a is not None:
            u_b = lerp(u_a, u_b, v)
    return True, a, b, u_a, u_b


# ---- the frame ---------------------------------------------------------------------------------------------------------------
def round_to_int(f):                                               # Mathf.RoundToInt: half to even
    return int(np.rint(F(f)))


def segment_contexts(setup, W, H):                                 # RenderManager.cs:281-318
    vp = (F(setup.vanishing_point_screen[0]), F(setup.vanishing_point_screen[1]))
    out = []
    for k in range(4):
        seg = setup.segments[k]
        c = {"ray_count": seg.ray_count, "seg": seg}
        if seg.ray_count > 0:
            c["axis"] = 0 if k > 1 else 1
            c["offset"] = setup.segments[0].ray_count if k == 1 else (setup.segments[2].ray_count if k == 3 else 0)
            cl = lambda v, hi: max(0, min(hi, v))   # noqa: E731
            if k == 0:
                mn, mx = cl(round_to_int(vp[1]), H - 1), H - 1
            elif k == 1:
                mn, mx = 0, cl(round_to_int(vp[1]), H - 1)
            elif k == 3:
                mn, mx = 0, cl(round_to_int(vp[0]), W - 1)
            else:
                mn, mx = cl(round_to_int(vp[0]), W - 1), W - 1
            c["pix_min"], c["pix_max"] = mn, mx
            c["buffer"] = 0 if k < 2 else 1
        out.append(c)
    return out


def render_raybuffers(worlds, setup, W, H, ray_indices=None):
    """worlds: list of PyWorldLod (LOD 0..). Returns (td, lr) uint32 arrays like the oracle's; rays not in ray_indices stay 0."""
    td = np.zeros((W + 2 * H, H), dtype=np.uint32)
    lr = np.zeros((2 * W + H, W), dtype=np.uint32)
    ctx = segment_contexts(setup, W, H)
    cam = setup.camera
    m = [F(v) for v in cam.world_to_screen]
    pos_xz, pos_y = (F(cam.position_xz[0]), F(cam.position_xz[1])), F(cam.position_y)
    far_clip = F(cam.far_clip)
    # a ray never switches past the last LOD given: its distance and the ones after it are +inf
    lod_dist = [F(v) if k < len(worlds) - 1 else POS_INF for k, v in enumerate(cam.lod_distances)]
    last_lod = len(worlds) - 1
    inverse = bool(cam.inverse_element_iteration_direction)
    total = sum(max(0, c["ray_count"]) for c in ctx)
    with np.errstate(all="ignore"):
        for flat in (range(total) if ray_indices is None else ray_indices):
            # RaySetupJob :20-39
            plane, seg = flat, None
            for j in range(4):
                n = ctx[j]["ray_count"]
                if n <= 0:
                    continue
                if plane >= n:
                    plane -= n
                    continue
                seg = ctx[j]
                break
            if seg is None:
                continue
            # DDASetupJob :59-76
            s = seg["seg"]
            end_lerp = F(plane) / F(s.ray_count)
            dx = lerp(F(s.cam_local_plane_ray_min[0]), F(s.cam_local_plane_ray_max[0]), end_lerp)
            dz = lerp(F(s.cam_local_plane_ray_min[1]), F(s.cam_local_plane_ray_max[1]), end_lerp)
            rs = F(1.0) / np.sqrt(dx * dx + dz * dz)
            ray = DDA(pos_xz, (dx * rs, dz * rs))
            row = (td if seg["buffer"] == 0 else lr)[plane + seg["offset"]]
            # TraceToFirstColumnJob :94-143
            lod = 0
            w0 = worlds[0]
            if ray.position[0] < 0 or ray.position[1] < 0 or ray.position[0] >= w0.dims[0] or ray.position[1] >= w0.dims[2]:
                if ray.step_to_world_intersection(w0.dims[0], w0.dims[2]):
                    lod_max = lod_dist[0]
                    while lod < last_lod and ray.dist[0] >= lod_max:
                        ray.next_lod(1 << lod)
                        lod += 1
                        lod_max = lod_dist[lod]
                    if ray.is_beyond_far_clip(far_clip):
                        row[seg["pix_min"]:seg["pix_max"] + 1] = SKYBOX      # WriteSkyboxFull
                        continue
                else:
                    row[seg["pix_min"]:seg["pix_max"] + 1] = SKYBOX
                    continue
            execute_ray(worlds, seg, ray, lod, row, m, pos_y, far_clip, lod_dist, -1 if inverse else 1, max(W, H))
    return td, lr


def execute_ray(worlds, seg, ray, lod, row, m, pos_y, far_clip, lod_dist, ITER, seen_len):   # DrawSegmentRayJob.cs:195-620
    voxel_scale = 1 << lod
    lod_max = lod_dist[lod]
    seen = np.zeros(seen_len + 2, dtype=np.uint8)
    orig_min, orig_max = seg["pix_min"], seg["pix_max"]
    nf_min, nf_max = orig_min, orig_max
    world_max_y = F(worlds[lod].dims[1])                      # read once from the starting LOD's world (:213)
    cam_y_norm = pos_y / world_max_y
    fb_min, fb_max = F(nf_min) - F(0.501), F(nf_max) + F(0.501)
    fdir_max = fdir_min = EPSILON

    # SetupProjectedPlaneParams :622-651
    top = mul_m_v(m, ray.start[0], world_max_y, ray.start[1], F(1))
    bot = mul_m_v(m, ray.start[0], F(0), ray.start[1], F(1))
    dr = mul_m_v(m, ray.dir[0], F(0), ray.dir[1], F(0))
    a = 0 if seg["axis"] == 0 else 1
    p_bot, p_top, p_dir = (bot[a], bot[2], bot[3]), (top[a], top[2], top[3]), (dr[a], dr[2], dr[3])

    def sky():
        for y in range(orig_min, orig_max + 1):
            if seen[y] == 0:
                row[y] = SKYBOX

    def along(p, d):
        return (p[0] + p_dir[0] * d, p[1] + p_dir[1] * d, p[2] + p_dir[2] * d)

    def reduce_horizon(b_min, b_max):                         # ReducePixelHorizon :660-697
        nonlocal nf_min, nf_max, fb_min, fb_max
        if b_min <= nf_min:
            b_min = nf_min
            if b_max >= nf_min:
                nf_min = b_max + 1
                while nf_min <= orig_max and seen[nf_min] > 0:
                    nf_min += 1
                fb_min = F(nf_min) - F(0.501)
        if b_max >= nf_max:
            b_max = nf_max
            if b_min <= nf_max:
                nf_max = b_min - 1
                while nf_max >= orig_min and seen[nf_max] > 0:
                    nf_max -= 1
                fb_max = F(nf_max) + F(0.501)
        return b_min, b_max

    while True:
        if lod < len(worlds) - 1 and ray.dist[0] >= lod_max:  # :237-243, never past the last LOD given
            ray.next_lod(voxel_scale)
            lod += 1
            voxel_scale *= 2
            lod_max = lod_dist[lod]
        world = worlds[lod]
        runs, col = world.get_voxel_column(ray.position[0], ray.position[1])
        if runs == -1:
            sky()
            return
        if runs == 0:
            if ray.do_step(far_clip):
                break
            continue
        wb_min, wb_max = F(0), world_max_y
        if fdir_max != EPSILON:                               # :261-281
            dist_top = ray.dist[1] if fdir_max > F(0) else ray.dist[0]
            dist_bot = ray.dist[1] if fdir_min < F(0) else ray.dist[0]
            new_max = pos_y + fdir_max * dist_top
            new_min = pos_y + fdir_min * dist_bot
            if new_min > wb_max or new_max < wb_min:
                sky()
                return
            if F(col[2]) > new_max or F(col[3]) < new_min:
                if ray.do_step(far_clip):
                    break
                continue
            wb_min, wb_max = new_min, new_max
        min_last, min_next = along(p_bot, ray.dist[0]), along(p_bot, ray.dist[1])      # :289-293
        max_last, max_next = along(p_top, ray.dist[0]), along(p_top, ray.dist[1])

        if ray.dist[0] > F(2.0) and fdir_max == EPSILON:      # :295-422
            c_last, l_min, l_max = world_bounds_clipping(min_last, max_last, fb_min, fb_max)
            c_next, n_min, n_max = world_bounds_clipping(min_next, max_next, fb_min, fb_max)
            if c_last:
                if c_next:
                    sky()
                    return
                wb_min, wb_max = lerp(F(0), world_max_y, n_min), lerp(F(0), world_max_y, n_max)
                fdir_max = (wb_max - pos_y) / ray.dist[1]
                fdir_min = (wb_min - pos_y) / ray.dist[1]
                mnc, mxc = lerp3(min_next, max_next, n_min), lerp3(min_next, max_next, n_max)
                c_min, c_max = mnc[0] / mnc[2], mxc[0] / mxc[2]
                if c_max < c_min:
                    c_min, c_max = c_max, c_min
            elif c_next:
                wb_min, wb_max = lerp(F(0), world_max_y, l_min), lerp(F(0), world_max_y, l_max)
                mnc, mxc = lerp3(min_last, max_last, l_min), lerp3(min_last, max_last, l_max)
                fdir_max = (wb_max - pos_y) / ray.dist[0]
                fdir_min = (wb_min - pos_y) / ray.dist[0]
                c_min, c_max = mnc[0] / mnc[2], mxc[0] / mxc[2]
                if c_max < c_min:
                    c_min, c_max = c_max, c_min
            else:
                if l_min < n_min:
                    wb_min = lerp(F(0), world_max_y, l_min)
                    fdir_min = (wb_min - pos_y) / ray.dist[0]
                else:
                    wb_min = lerp(F(0), world_max_y, n_min)
                    fdir_min = (wb_min - pos_y) / ray.dist[1]
                if l_max > n_max:
                    wb_max = lerp(F(0), world_max_y, l_max)
                    fdir_max = (wb_max - pos_y) / ray.dist[0]
                else:
                    wb_max = lerp(F(0), world_max_y, n_max)
                    fdir_max = (wb_max - pos_y) / ray.dist[1]
                mn_a, mx_a = lerp3(min_last, max_last, l_min), lerp3(min_last, max_last, l_max)
                mn_b, mx_b = lerp3(min_next, max_next, n_min), lerp3(min_next, max_next, n_max)
                min_n, min_l = mn_b[0] / mn_b[2], mn_a[0] / mn_a[2]
                max_n, max_l = mx_b[0] / mx_b[2], mx_a[0] / mx_a[2]
                if max_n < min_n:
                    max_n, min_n = min_n, max_n
                if max_l < min_l:
                    max_l, min_l = min_l, max_l
                c_min, c_max = umin(min_l, min_n), umax(max_l, max_n)
            wb_min, wb_max = np.floor(wb_min), np.ceil(wb_max)
            wr_min, wr_max = to_int(np.floor(c_min)), to_int(np.ceil(c_max))
            if wr_max < nf_min or wr_min > nf_max:
                sky()
                return
            if wr_min > nf_min:
                nf_min = wr_min
                while nf_min <= orig_max and seen[nf_min] > 0:
                    nf_min += 1
            if wr_max < nf_max:
                nf_max = wr_max
                while nf_max >= orig_min and seen[nf_max] > 0:
                    nf_max -= 1
            if nf_min > nf_max:
                sky()
                return

        off, run_count = col[0], col[1]
        if ITER > 0:                                          # :428-438
            e_min = e_max = world_max_y
            ptr = off                                         # ElementGuardStart
        else:
            e_min = e_max = F(0)
            ptr = off + run_count + 1                         # ElementGuardEnd
        colors = off + run_count + 2                          # ColorPointer

        while True:                                           # :441-611
            ptr += ITER
            ci, length = world.element(ptr)
            if length == 0:                                   # !IsValid
                break
            if ITER > 0:
                e_max = e_min
                e_min = e_min - F(length * voxel_scale)
            else:
                e_min = e_max
                e_max = e_min + F(length * voxel_scale)
            if ci < 0:                                        # IsAir
                continue
            if e_min > wb_max:
                if ITER < 0:
                    break
                continue
            if e_max < wb_min:
                if ITER > 0:
                    break
                continue
            portion_bottom = unlerp(F(0), world_max_y, e_min)
            portion_top = unlerp(F(0), world_max_y, e_max)
            front_bottom = lerp3(min_last, max_last, portion_bottom)
            front_top = lerp3(min_last, max_last, portion_top)
            # side of the run :484-542
            ok, front_bottom, front_top, u_a, u_b = clip_line(front_bottom, front_top, F(length), F(0))
            if ok:
                uv_a = (F(1.0) / front_bottom[2], u_a / front_bottom[2])
                uv_b = (F(1.0) / front_top[2], u_b / front_top[2])
                bf = [front_bottom[0] / front_bottom[2], front_top[0] / front_top[2]]      # ProjectClippedToScreen :159-163
                if bf[0] > bf[1]:
                    bf = [bf[1], bf[0]]
                    uv_a, uv_b = uv_b, uv_a
                b_min, b_max = to_int(np.rint(bf[0])), to_int(np.rint(bf[1]))
                if b_max >= nf_min and b_min <= nf_max:
                    b_min, b_max = reduce_horizon(b_min, b_max)
                    for y in range(b_min, b_max + 1):
                        if seen[y] == 0:
                            fdir_max = EPSILON
                            seen[y] = 1
                            l = unlerp(bf[0], bf[1], F(y))
                            wu = (lerp(uv_a[0], uv_b[0], l), lerp(uv_a[1], uv_b[1], l))
                            u = wu[1] / wu[0]
                            idx = max(0, min(length - 1, to_int(np.floor(u)))) + ci
                            row[y] = world.cells[colors + idx]
                    if nf_min > nf_max:
                        sky()
                        return
            # top / bottom of the run :544-610
            if portion_top < cam_y_norm:
                if e_max > wb_max:
                    continue
                color = world.cells[colors + ci]
                sec_a, sec_b = lerp3(min_next, max_next, portion_top), front_top
            elif portion_bottom > cam_y_norm:
                if e_min < wb_min:
                    continue
                color = world.cells[colors + ci + length - 1]
                sec_a, sec_b = lerp3(min_next, max_next, portion_bottom), front_bottom
            else:
                continue
            ok, sec_a, sec_b, _, _ = clip_line(sec_a, sec_b)
            if ok:
                b_min = to_int(np.rint(sec_a[0] / sec_a[2]))
                b_max = to_int(np.rint(sec_b[0] / sec_b[2]))
                if b_min > b_max:
                    b_min, b_max = b_max, b_min
                if b_max >= nf_min and b_min <= nf_max:
                    b_min, b_max = reduce_horizon(b_min, b_max)
                    for y in range(b_min, b_max + 1):
                        if seen[y] == 0:
                            fdir_max = EPSILON
                            seen[y] = 1
                            row[y] = color
                    if nf_min > nf_max:
                        sky()
                        return
        if ray.do_step(far_clip):
            break
    sky()


# ---- Phase 2 -----------------------------------------------------------------------------------------------------------------
def blit(setup, W, H, td, lr):
    """BlitSegments + RayBufferBlit.shader frag (RenderManager.cs:199-256, Shaders/RayBufferBlit.shader:55-62), vectorised over the
    screen: pixel centres (x + 0.5, y + 0.5), bottom-left origin; triangle k = (VP, MaxScreen_k, MinScreen_k) carries uv (0,0), (1,0),
    (0,1), so uv.x / uv.y are the affine weights b, c of Max / Min (kept unnormalised: times |det|); x = b / (b + c); row = floor((offset_k + x * scale_k) * rows)
    clamped to the segment's rows; column = y (top/down) or x (left/right). A pixel takes the first segment with b, c >= 0, else the
    one with the largest min(b, c) (the GPU rasteriser's coverage rule at shared edges is not reproducible; DESIGN.md §3.2)."""
    vx, vy = F(setup.vanishing_point_screen[0]), F(setup.vanishing_point_screen[1])
    td_rows, lr_rows = W + 2 * H, 2 * W + H
    px = (np.arange(W, dtype=np.float32) + F(0.5))[None, :].repeat(H, 0)
    py = (np.arange(H, dtype=np.float32) + F(0.5))[:, None].repeat(W, 1)
    dx, dy = px - vx, py - vy
    best = np.full((H, W), -1, dtype=np.int32)
    best_b = np.zeros((H, W), dtype=np.float32)
    best_c = np.zeros((H, W), dtype=np.float32)
    score = np.full((H, W), -np.inf, dtype=np.float32)
    done = np.zeros((H, W), dtype=bool)
    with np.errstate(all="ignore"):
        for k in range(4):
            sg = setup.segments[k]
            if sg.ray_count <= 0:
                continue
            e1x, e1y = F(sg.max_screen[0]) - vx, F(sg.max_screen[1]) - vy
            e2x, e2y = F(sg.min_screen[0]) - vx, F(sg.min_screen[1]) - vy
            det = e1x * e2y - e1y * e2x
            # unnormalised affine weights (x = uv.x / (uv.x + uv.y) does not depend on the common factor 1/det)
            b = dx * e2y - dy * e2x
            c = e1x * dy - e1y * dx
            if det < 0:
                b, c = -b, -c
            inside = (b >= 0) & (c >= 0) & ~done
            sc = np.where(np.isnan(c) | (b < c), b, c) / np.abs(det)   # math.min
            better = ~done & ~inside & (sc > score)
            take = inside | better
            best[take] = k
            best_b[take] = b[take]
            best_c[take] = c[take]
            score[better] = sc[better]
            done |= inside
        frame = np.zeros((H, W), dtype=np.uint32)
        ys, xs = np.mgrid[0:H, 0:W]
        for k in range(4):
            sel = best == k
            if not sel.any():
                continue
            rows = td_rows if k < 2 else lr_rows
            rc = setup.segments[k].ray_count
            off = setup.segments[0].ray_count if k == 1 else (setup.segments[2].ray_count if k == 3 else 0)
            scale = F(rc) / F(rows)
            offset = F(off) / F(rows) if k in (1, 3) else F(0)
            t = best_b[sel] / (best_b[sel] + best_c[sel])
            v = offset + t * scale
            r = np.floor(v * F(rows))
            r = np.where((r >= F(-2147483648.0)) & (r < F(2147483648.0)), r, F(-2147483648.0)).astype(np.int64)   # (int) cast; NaN -> INT_MIN
            r = np.clip(r, off, off + rc - 1)
            frame[sel] = td[r, ys[sel]] if k < 2 else lr[r, xs[sel]]
    return frame


# ---- host setup (logic cross-check in float64; the float32 restatements are the library's host_setup.cpp and the C++ oracle) ------
def _quat_rotate(q, v):
    x, y, z, w = q
    u = np.array([x, y, z], dtype=np.float64)
    v = np.asarray(v, dtype=np.float64)
    return v + 2.0 * np.cross(u, np.cross(u, v) + w * v)


def _signed_angle(a, b):                                           # Vector2.SignedAngle (SURVEY.md A5)
    den = np.sqrt(float(a[0] * a[0] + a[1] * a[1]) * float(b[0] * b[0] + b[1] * b[1]))
    if den < 1e-15:
        return 0.0
    ang = np.degrees(np.arccos(np.clip((a[0] * b[0] + a[1] * b[1]) / den, -1.0, 1.0)))
    return ang * (1.0 if a[0] * b[1] - a[1] * b[0] >= 0.0 else -1.0)


def host_frame_setup(position, rotation, fov_y_degrees, near, far, W, H):
    """RenderManager.DrawWorld up to DrawSegments (RenderManager.cs:119-152,374-501) + the CameraData ctor (CameraData.cs:18-36) in
    float64. Returns dict(vp, segments=[(min_screen, max_screen, ray_min, ray_max, ray_count) or None], world_to_screen 4x4, inverse)."""
    pos = np.asarray(position, dtype=np.float64)
    fwd, up = _quat_rotate(rotation, (0, 0, 1)), _quat_rotate(rotation, (0, 1, 0))
    t = np.tan(np.radians(fov_y_degrees) / 2.0)
    aspect = W / H
    proj = np.array([[1.0 / (aspect * t), 0, 0, 0], [0, 1.0 / t, 0, 0], [0, 0, -(far + near) / (far - near), -2.0 * far * near / (far - near)], [0, 0, -1, 0]])
    right = np.cross(up, fwd)
    right /= np.linalg.norm(right)                                 # Matrix4x4.LookAt(0, forward, up): columns right, up', forward (A4)
    up2 = np.cross(fwd, right)
    look = np.eye(4)
    look[:3, 0], look[:3, 1], look[:3, 2] = right, up2, fwd / np.linalg.norm(fwd)
    zflip = np.diag([1.0, 1.0, -1.0, 1.0])
    # CalculateVanishingPointWorld :374-378: sin(eulerAngles.x) = -forward.y (A6)
    vp_world = pos + np.array([0.0, 1.0, 0.0]) * (near / fwd[1])
    local_to_screen = proj @ (zflip @ np.linalg.inv(look))         # :386-388
    cam = local_to_screen @ np.append(vp_world - pos, 1.0)
    vp = (cam[:2] / cam[3] * 0.5 + 0.5) * np.array([W, H], dtype=np.float64)
    screen = np.array([W, H], dtype=np.float64)
    to_local = look @ (np.linalg.inv(zflip) @ np.linalg.inv(proj))  # TransformPixel :487-500

    def transform_pixel(px):
        v = to_local @ np.array([(px[0] / W - 0.5) * 2.0, (px[1] / H - 0.5) * 2.0, 1.0, 1.0])
        return np.array([v[0], v[2]]) / v[3]

    def segment(dist, neutral, primary):                           # GetGenericSegmentParameters :402-501
        sec = 1 - primary
        smin = np.array([vp[sec] - dist] * 2)
        smax = np.array([vp[sec] + dist] * 2)
        a = vp[primary] + dist * np.sign(neutral[primary])
        smin[primary] = smax[primary] = a
        if smax[sec] <= 0.0 or smin[sec] >= screen[sec]:
            return None
        if (vp >= 0.0).all() and (vp <= screen).all():
            mn, mx = smin, smax
        else:
            mid = (smin + 0.5 * (smax - smin)) - vp
            ang_l, ang_r, dir_l, dir_r = 90.0, -90.0, np.zeros(2), np.zeros(2)
            for corner in ((0.0, 0.0), (0.0, screen[1]), (screen[0], 0.0), (screen[0], screen[1])):
                d = np.array(corner) - vp
                scaled = d * (dist / abs(d[primary]))
                ang = _signed_angle(neutral, d)
                if ang < ang_l:
                    ang_l, dir_l = ang, scaled
                if ang > ang_r:
                    ang_r, dir_r = ang, scaled
            c_l, c_r = dir_l + vp, dir_r + vp
            if ang_l < -45.0:
                c_l = smin if _signed_angle(mid, smax) > 0.0 else smax      # (:466: a point passed as a direction, as in the reference)
            if ang_r > 45.0:
                c_r = smin if _signed_angle(mid, smax) < 0.0 else smax
            swap = c_l[sec] > c_r[sec]
            mn, mx = (c_r, c_l) if swap else (c_l, c_r)
        count = max(0, int(np.rint(mx[sec] - mn[sec])))
        return mn, mx, transform_pixel(mn), transform_pixel(mx), count

    segs = [None] * 4
    if vp[1] < H:
        segs[0] = segment(H - vp[1], (0.0, 1.0), 1)
    if vp[1] > 0.0:
        segs[1] = segment(vp[1], (0.0, -1.0), 1)
    if vp[0] < W:
        segs[2] = segment(W - vp[0], (1.0, 0.0), 0)
    if vp[0] > 0.0:
        segs[3] = segment(vp[0], (-1.0, 0.0), 0)
    # CameraData ctor: worldToCamera = Scale(1,1,-1) * inverse(TRS(pos, rot, 1)) (A3)
    rot = np.eye(4)
    rot[:3, 0], rot[:3, 1], rot[:3, 2] = _quat_rotate(rotation, (1, 0, 0)), up, fwd
    trs = rot.copy()
    trs[:3, 3] = pos
    w2c = zflip @ np.linalg.inv(trs)
    scale_half = np.diag([0.5, 0.5, 1.0, 1.0])
    trans = np.eye(4)
    trans[:3, 3] = (0.5, 0.5, 1.0)
    w2s = np.diag([W, H, 1.0, 1.0]) @ (trans @ (scale_half @ (proj @ w2c)))
    return {"vp": vp, "segments": segs, "world_to_screen": w2s, "inverse": bool(fwd[1] >= 0.0)}
