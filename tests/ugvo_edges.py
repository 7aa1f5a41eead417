"""UGV-FOA (K-UGVO, csrc/ugvo.cu) lanes beyond the pose-level edges of env_edges.py: a float64 restatement of the fake
laser with its perturbation set, laser edge blocks, centre-distance ties of the obstacle list, reset parameters that put
the map generator on its fallbacks, and reset legality tests on equality.

Fake laser.  `fake_laser` evaluates get_fake_laser the way oracle/c/ugvo.c does (tan, pow, acos and fma of the C library,
IEEE divisions) over lanes x rays; it equals the oracle bit for bit.  The kernel departs from it by documented error
sources only: its slope is fm64::sincos's quotient (K_SLOPE / K_STEEP ulps from tan), its ray angle comes from a
Divisor (1 ulp), its corner bearings from libdevice's acos (1 ulp).  `laser_variants` evaluates the restatement over that
perturbation set P; a ray is stable where every value over P agrees within the one-step bound.  `laser_blocks` are
parked lanes on each laser decision (L1 tangency, L2 centre on a ray's normal, L3 in-range boundary / crossing at the
segment end, L5 first accepted not nearest, L7 corner bearings, L8 near-vertical rays and the 1e8 guard, L9 ray-angle
wrap, L10 vehicle on the border, L11 ray length at laser_dis); L4 is `tie_rows`.

Ties.  The step kernel orders the in-range circles by an insertion sort per thread, the reset / observe path by a
warp-vote rank; both must keep np.argsort's order, lower index first on equal distances, because a ray stops at the
FIRST circle it accepts (note N8).  `tie_rows` places two circles at bit-equal distance from a parked vehicle, mirrored
about the x axis through it (dyadic coordinates: dx and +-dy are exact), with different radii, both crossed by the rays
near bearing 0; each geometry comes twice, with the radii swapped between the slots.

Map fallbacks (`MAP_EDGES`).  reset_map draws the target from blocks 1..64 and keeps block 64's draw when none is
safety_dis_st from the start; it tries 2048 candidates per obstacle and stops placing when none is legal.
`equality_cases` restate the Philox draws of an instance and set safety_dis_st so that fl(r + safety_dis_st) lands on
the distance from the start to obstacle 0's first candidate (+-1, 2 ulps), or safety_dis_st on the first target
candidate's distance: the decisions `within()` takes on squares with a sqrt fallback band.
"""
from __future__ import annotations

import ctypes

import numpy as np

import env_edges as E

# the C library's tan / acos / fma / pow, which the oracle calls (numpy's own float64 tan and arccos differ from them in
# the last bit on a few per cent of arguments, and glibc's pow(m, 2.0) is not always fl(m * m))
_libm = ctypes.CDLL("libm.so.6")
for _f, _n in (("tan", 1), ("acos", 1), ("fma", 3), ("pow", 2)):
    getattr(_libm, _f).restype = ctypes.c_double
    getattr(_libm, _f).argtypes = [ctypes.c_double] * _n
_tan = np.frompyfunc(_libm.tan, 1, 1)
_acos = np.frompyfunc(_libm.acos, 1, 1)
_fma = np.frompyfunc(_libm.fma, 3, 1)
_pow = np.frompyfunc(_libm.pow, 2, 1)


def sqr(x):
    """pow(x, 2.0) of the C library."""
    x = np.asarray(x, np.float64)
    return np.asarray(_pow(x, 2.0), np.float64) if x.size else x.copy()


def c_tan(x):
    return np.asarray(_tan(np.asarray(x, np.float64)), np.float64)


def c_acos(x):
    return np.asarray(_acos(np.asarray(x, np.float64)), np.float64)


def norm2(a, b):
    """np.linalg.norm((a, b)) = sqrt(fma(b, b, a * a)) (oracle ugvo.c norm2), elementwise on arrays."""
    a, b = np.broadcast_arrays(np.asarray(a, np.float64), np.asarray(b, np.float64))
    if a.size == 0:
        return np.zeros(a.shape)
    return np.sqrt(np.asarray(_fma(b, b, a * a), np.float64))


def vector_rad(x1, y1, x2, y2):
    """cal_vector_rad (utils/functions.py:35-46): 0 for a vector shorter than 1e-4, else acos of the clipped cosine."""
    n1, n2 = norm2(x1, y1), norm2(x2, y2)
    with np.errstate(invalid="ignore", divide="ignore"):
        c = np.minimum(np.maximum((x1 * x2 + y1 * y2) / (n1 * n2), -1.0), 1.0)
    return np.where((n2 < 1e-4) | (n1 < 1e-4), 0.0, c_acos(np.where(np.isfinite(c), c, 0.0)))


def ray_angles(p, st):
    """np.linspace(phi - R, phi + R, n_rays) wrapped into [-pi, pi] -> [lanes, n_rays]."""
    phi = np.asarray(st, np.float64)[:, 3:4]
    a0, a1 = phi - p.laser_range, phi + p.laser_range
    step = (a1 - a0) / (p.n_rays - 1)
    ph = np.arange(p.n_rays)[None, :] * step + a0
    ph[:, -1] = a1[:, 0]
    ph = np.where(ph > np.pi, ph - 2 * np.pi, ph)
    return np.where(ph < -np.pi, ph + 2 * np.pi, ph)


def corner_bearings(p, st):
    """th1..th4 of get_fake_laser :304-309 -> [lanes, 4]."""
    x, y = st[:, 0], st[:, 1]
    xm, ym = p.map_x, p.map_y
    return np.stack([vector_rad(1.0, 0.0, xm - x, ym - y), vector_rad(1.0, 0.0, 0 - x, ym - y),
                     -vector_rad(1.0, 0.0, 0 - x, 0 - y), -vector_rad(1.0, 0.0, xm - x, 0 - y)], 1)


def fake_laser(p, st, *, m=None, ray_phi=None, th=None, stats=None):
    """get_fake_laser (:274-397) in float64, the reference's expressions as oracle/c/ugvo.c:47-125 evaluates them, over
    lanes x rays.  `ray_phi` [lanes, rays], `m` [lanes, rays] and `th` [lanes, 4] replace the ray angles, the slopes
    (default tan(ray_phi)) and the corner bearings.  `stats`, a dict, counts the decisions taken (rays that hit a
    circle, the wall branch, the near-vertical guard).  -> laser ranges [lanes, rays]."""
    st = np.asarray(st, np.float64)
    L, NR = len(st), p.n_rays
    LD, LB, xm, ym = p.laser_dis, p.laser_blind, p.map_x, p.map_y
    x, y = st[:, :1], st[:, 1:2]
    ph = ray_angles(p, st) if ray_phi is None else np.asarray(ray_phi, np.float64)
    m = c_tan(ph) if m is None else np.asarray(m, np.float64)
    th = corner_bearings(p, st) if th is None else np.asarray(th, np.float64)
    th1, th2, th3, th4 = (th[:, k:k + 1] for k in range(4))
    with np.errstate(all="ignore"):
        b = y - m * x
        m_2 = sqr(m)
        sq = np.sqrt(1 + m_2)
        cosT, sinT, am = np.abs(m) / sq, 1 / sq, np.abs(m)
        mpos = m >= 0
        rA, rB, rC = (th4 < ph) & (ph <= th1), (th1 < ph) & (ph <= th2), (th3 < ph) & (ph <= th4)
        rA, rB, rC = rA, rB & ~rA, rC & ~rA & ~rB
        rD = ~(rA | rB | rC)
        big = am >= 1e8
        tA, tB, tC, tD = x + LD / sq, y + am * LD / sq, y - am * LD / sq, x - LD / sq
        tx = np.select([rA, rB, rC], [np.where(tA < xm, tA, xm),
                                      np.where(tB < ym, np.where(mpos, x + LD * sinT, x - LD * sinT), np.where(big, x, (ym - b) / m)),
                                      np.where(tC > 0, np.where(mpos, x - LD * sinT, x + LD * sinT), np.where(big, x, -b / m))],
                       np.where(tD > 0, tD, 0.0))
        ty = np.select([rA, rB, rC], [np.where(tA < xm, np.where(mpos, y + cosT * LD, y - cosT * LD), m * xm + b),
                                      np.where(tB < ym, tB, ym), np.where(tC > 0, tC, 0.0)],
                       np.where(tD > 0, np.where(mpos, y - cosT * LD, y + cosT * LD), b))
        tx, ty = np.broadcast_to(tx, (L, NR)).copy(), np.broadcast_to(ty, (L, NR)).copy()
        nobs = st[:, 7].astype(int)
        cx, cy, cr = st[:, 8:56:3], st[:, 9:56:3], st[:, 10:56:3]
        ref = norm2(x - cx, y - cy)
        ref = np.where(np.arange(16)[None, :] < nobs[:, None], ref, np.inf)
        order = np.argsort(ref, axis=1, kind="stable")
        out = np.full((L, NR), np.nan)
        found = np.zeros((L, NR), bool)
        m2p1 = m_2 + 1
        d = tx - x
        sg = np.where(d > 0, 1.0, np.where(d < 0, -1.0, 0.0))
        lo, hi = np.minimum(x, tx), np.maximum(x, tx)
        rows = np.arange(L)
        for j in range(16):
            idx = order[:, j]
            live = (j < nobs)[:, None] & ~found
            x0, y0, r0 = cx[rows, idx][:, None], cy[rows, idx][:, None], cr[rows, idx][:, None]
            rd = ref[rows, idx][:, None]
            live &= ~(rd > LD + r0)
            live &= ~(np.abs(m * x0 - y0 + b) / sq > r0)
            if not live.any():
                continue
            w = np.nonzero(live)
            X0, Y0, R0 = np.broadcast_to(x0, (L, NR))[w], np.broadcast_to(y0, (L, NR))[w], np.broadcast_to(r0, (L, NR))[w]
            xx, yy, mm, bb, TX, TY = np.broadcast_to(x, (L, NR))[w], np.broadcast_to(y, (L, NR))[w], m[w], b[w], tx[w], ty[w]
            ok = ~(vector_rad(TX - xx, TY - yy, X0 - xx, Y0 - yy) > np.pi / 2)
            fx = (X0 + mm * Y0 - mm * bb) / m2p1[w]
            fy = (mm * X0 + m_2[w] * Y0 + bb) / m2p1[w]
            r_dis = norm2(fx - X0, fy - Y0)
            cross = fx - sg[w] * np.sqrt(sqr(R0) - sqr(r_dis)) / np.sqrt(m2p1[w])
            hit = ok & (lo[w] <= cross) & (cross <= hi[w])
            dis = np.abs(cross - xx) * np.sqrt(m2p1[w])
            wi = tuple(a[hit] for a in w)
            out[wi] = np.where(dis[hit] < LB, LB, dis[hit])
            found[wi] = True
        ray_len = norm2(x - tx, y - ty)
        wall = np.where(ray_len > LD, LD, np.where((LB < ray_len) & (ray_len <= LD), ray_len, LB))
        out = np.where(found, out, wall)
    col = E._ugvo_collided(p, st)
    out[col] = LB
    if stats is not None:
        live = ~col[:, None]
        for k, v in (("hit", found), ("right", rA), ("top", rB), ("bottom", rC), ("left", rD), ("guard_1e8", big & (rB | rC)),
                     ("at_laser_dis", ~found & (ray_len > LD))):
            stats[k] = stats.get(k, 0) + int((v & live).sum())
    return out


def laser_obs(p, laser):
    """the observation terms 4.. of get_state: (2 laser / laser_dis - 1) static_gain."""
    return (2 * laser / p.laser_dis - 1) * p.static_gain

# parameter overrides of b200_ugvo_params: name -> {field: value}
MAP_EDGES = {
    # no target candidate is accepted (safety_dis_st above the 4.4 m diagonal of the start box): block 64's draw is
    # kept; no circle is legal either
    "target_fallback": {"safety_dis_st": 10.0},
    # circles of radius 1.2: a few fit, then placement gives up after 2048 candidates
    "give_up_radius": {"r_min": 1.2, "r_max": 1.2},
    # 16 = B200_UGVO_MAX_OBS circles wanted, kept 1.5 m apart: fewer fit
    "give_up_16": {"obs_num": 16, "safety_dis_obs": 1.5},
    # 16 wanted, small and close: every slot is filled
    "full_16": {"obs_num": 16, "r_min": 0.1, "r_max": 0.15, "safety_dis_obs": 0.05, "safety_dis_st": 0.3},
}


def with_params(p, over):
    """a copy of the ctypes parameter struct `p` with the fields of `over` replaced."""
    q = type(p).from_buffer_copy(p)
    for k, v in over.items():
        setattr(q, k, v)
    return q


def tie_rows(p):
    """[lanes, 56] parked states with two circles (slots 0 and 1) at bit-equal centre distance; see the docstring."""
    rows = []
    for x, y in ((1.0, 2.5), (1.5, 2.0), (0.75, 3.0)):
        for a, b in ((1.0, 0.25), (1.25, 0.125), (0.875, 0.3125)):
            for ra, rb in ((0.4, 0.3), (0.3, 0.4)):
                rows.append(E.ugvo_row(p, x, y, phi=0.3, near=[(x + a, y + b, ra), (x + a, y - b, rb)]))
    return np.stack(rows)


def swap_first_two(rows):
    """the same states with circles 0 and 1 exchanged."""
    r = rows.copy()
    r[:, 8:11], r[:, 11:14] = rows[:, 11:14], rows[:, 8:11]
    return r


def oracle_env(name, n, p=None, seed=E.SEED, offset=0):
    from oracle import oracle
    from reinforcementlearningplatform_b200 import _lib
    h = E.host(name)
    sf, od, ad, dd = _lib.dims(h.ENV_ID, h.VARIANT)
    return oracle.OracleEnv(h.ENV_ID, p if p is not None else h._params, n, sf, od, ad, dd, seed=seed,
                            env_index_offset=offset, nthreads=4)


def oracle_observe(name, rows):
    """get_state() of the C oracle at the given states -> [lanes, 41]."""
    o = oracle_env(name, len(rows))
    o.state[:] = np.asarray(rows, np.float64).T
    return o.observe().T.copy()


def oracle_reset(name, n, p, seed=E.SEED, offset=0):
    """reset(random=True) of n instances by the C oracle under parameters p -> (state [n, 56], next_obs [n, 41])."""
    o = oracle_env(name, n, p, seed, offset)
    o.reset()
    return o.state.T.copy(), o.next_obs.T.copy()


def draw2(seed, gid, ep, block):
    """the two U[0, 1) of one Philox4x32-10 block (ugvo.cu / oracle ugvo.c draw2), restated on oracle.philox."""
    from oracle import oracle
    r = oracle.philox([gid & 0xFFFFFFFF, gid >> 32, ep, block], [seed & 0xFFFFFFFF, seed >> 32]).astype(np.float64)
    u0 = ((r[0] // 32) * 67108864.0 + (r[1] // 64)) * (1.0 / 9007199254740992.0)
    u1 = ((r[2] // 32) * 67108864.0 + (r[3] // 64)) * (1.0 / 9007199254740992.0)
    return u0, u1


def lerp_u(lo, hi, u):
    return float(E.fma_exact(np.array([hi - lo]), np.array([u]), np.array([lo]))[0])


# ------------------------------------------------------------------------------------------------------ laser blocks
# Parked lanes (vel = omega = 0, zero action: scan A and scan B are both the laser at the injected pose), one block per
# kind of laser decision, each scanned over +-SCAN ulps of its decisive coordinate.
SCAN = 32
K_SLOPE = 4          # |m_kernel - tan(phi)| in ulps of tan(phi), rays with |m| < 1e3 (sincos + quotient)
K_STEEP = 4          # the same for |m| >= 1e3 (measured on a B200: 4.00 and 2.00 ulps, K included the quotient's 1)


def _scan(rows, col, k=SCAN):
    """each base row repeated over +-k ulps of field `col` -> (rows, ulp offset)."""
    ks = np.arange(-k, k + 1)
    out = np.repeat(rows, len(ks), axis=0)
    out[:, col] = E.ulps(out[:, col], np.tile(ks, len(rows)))
    return out, np.tile(ks, len(rows))


def laser_blocks(p):
    """label -> (rows [lanes, 56], ulp offsets, decisive ray index or None)."""
    B = {}
    x, y, h = 1.5, 2.5, 0.3
    ph = ray_angles(p, np.array([E.ugvo_row(p, x, y, phi=h)]))[0]
    # L1 tangency: r0 on the restated |m x0 - y0 + b| / sqrt(m^2 + 1) of ray k (|m| < 1 and |m| > 1); a second circle
    # further along the ray takes the miss
    rows = []
    for k in (15, 12, 31, 33):
        a = ph[k]
        for side in (1, -1):
            cx, cy = x + 1.0 * np.cos(a) - side * 0.3 * np.sin(a), y + 1.0 * np.sin(a) + side * 0.3 * np.cos(a)
            m = c_tan(a)
            r0 = abs(m * cx - cy + (y - m * x)) / np.sqrt(1 + sqr(m))
            far = (x + 1.7 * np.cos(a), y + 1.7 * np.sin(a), 0.2)
            rows.append(E.ugvo_row(p, x, y, phi=h, near=[(cx, cy, float(r0)), far]))
    B["L1_tangency"] = (*_scan(np.array(rows), 10), None)
    # L2 centre on the normal to a ray through the vehicle, just beyond the collision distance: the dot product of the
    # behind test is 0 +- ulps there, and the line misses the circle
    rows = []
    for k in (10, 18, 26):
        a = ph[k]
        for side in (1, -1):
            d = 0.3 + p.r_vehicle + 1e-6
            rows.append(E.ugvo_row(p, x, y, phi=h, near=[(x - side * d * np.sin(a), y + side * d * np.cos(a), 0.3)]))
    B["L2_perpendicular"] = (*_scan(np.array(rows), 8), None)
    # L3 in-range boundary: |centre - pos| == laser_dis + r0 (the circle then reaches the segment end: L6 too)
    rows = []
    for k in (8, 18, 27):
        a = ph[k]
        cx, cy = x + 2.3 * np.cos(a), y + 2.3 * np.sin(a)
        dd = norm2(x - cx, y - cy)
        rows.append(E.ugvo_row(p, x, y, phi=h, near=[(cx, cy, float(dd - p.laser_dis))]))
    B["L3_in_range"] = (*_scan(np.array(rows), 10), None)
    # L5 first accepted, not nearest: a small nearer-centred circle crossed beyond a large farther-centred one
    rows = []
    for k in (14, 20):
        a = ph[k]
        n = (-np.sin(a), np.cos(a))
        small = (x + 1.0 * np.cos(a) + 0.15 * n[0], y + 1.0 * np.sin(a) + 0.15 * n[1], 0.16)
        large = (x + 1.1 * np.cos(a) - 0.6 * n[0], y + 1.1 * np.sin(a) - 0.6 * n[1], 0.65)
        rows.append(E.ugvo_row(p, x, y, phi=h, near=[large, small]))
    B["L5_first_accepted"] = (*_scan(np.array(rows), 11), None)
    # L7 wall selection: the middle ray on a corner bearing, the corner nearer (1.4 m) and farther (4.2 m) than laser_dis
    rows = []
    for vx, vy in ((4.0, 4.0), (2.0, 2.0), (1.0, 4.0), (4.0, 1.0), (1.2, 1.3)):
        st = E.ugvo_row(p, vx, vy)
        th = corner_bearings(p, st[None])[0]
        for c in range(4):
            s = st.copy()
            s[3] = th[c]
            r = ray_angles(p, s[None])[0, 18]
            s[3] = th[c] + (th[c] - r)     # ray 18 within an ulp or two of the bearing
            rows.append(s)
    B["L7_corner"] = (*_scan(np.array(rows), 3), 18)
    # L8 near-vertical rays: the last ray at fl(pi/2) - 1e-8 + ulps (m straddles the 1e8 guard in steps of ~2), and
    # headings 0, +-pi, +-fl(pi/2); a circle straight above or below the vehicle
    hp = np.pi / 2
    rows = []
    for x8, y8, cy, hd in ((2.5, 1.5, 2.6, -1e-8), (2.5, 3.5, 2.4, np.pi - 1e-8), (2.5, 1.5, 2.6, 0.0), (2.5, 3.5, 2.4, np.pi),
                           (2.5, 3.5, 2.4, -np.pi), (2.5, 1.5, 2.6, hp), (2.5, 3.5, 2.4, -hp)):
        rows.append(E.ugvo_row(p, x8, y8, phi=hd, near=[(2.5, cy, 0.3)]))
    rows = np.array(rows)
    a1 = E.ulps(np.full(2 * SCAN + 1, hp - 1e-8), np.arange(-SCAN, SCAN + 1))
    guard = np.repeat(rows[:1], 2 * SCAN + 1, 0)
    guard[:, 3] = a1 - p.laser_range      # exact: the last ray is a1 again
    rs, ks = _scan(rows[2:], 3)
    keep = np.abs(rs[:, 3]) <= np.pi    # headings beyond +-pi are wrapped by the step: the lane would not be parked
    B["L8_vertical"] = (np.concatenate([guard, rs[keep]]), np.concatenate([np.arange(-SCAN, SCAN + 1), ks[keep]]), None)
    # L9 ray-angle wrap: headings fl(pi / 2) +- ulps, so the last rays cross +-pi
    rows = [E.ugvo_row(p, 2.0, 2.5, phi=s * (np.pi - p.laser_range), near=[(1.0, 2.5, 0.3)]) for s in (1, -1)]
    B["L9_wrap"] = (*_scan(np.array(rows), 3), 36)
    # L10 vehicle on the border: x, y at 0 / map and at the corners (degenerate rays, sg = 0)
    rows = [E.ugvo_row(p, 0.0, 2.5, phi=np.pi), E.ugvo_row(p, 5.0, 2.5, phi=0.0 + 0.3), E.ugvo_row(p, 2.5, 0.0, phi=-1.2),
            E.ugvo_row(p, 2.5, 5.0, phi=1.9), E.ugvo_row(p, 5.0, 5.0, phi=0.7), E.ugvo_row(p, 0.0, 0.0, phi=-2.4)]
    r10 = []
    for s in rows:
        for col in (0, 1):
            if s[col] in (0.0, 5.0):
                r10.append(_scan(s[None], col, 8))
    B["L10_border"] = (np.concatenate([r for r, _ in r10]), np.concatenate([k for _, k in r10]), None)
    # L11 ray length at laser_dis: the vehicle laser_dis from the right / left wall on the heading ray
    rows = [E.ugvo_row(p, p.map_x - p.laser_dis, 2.5, phi=0.0), E.ugvo_row(p, p.laser_dis, 2.5, phi=np.pi),
            E.ugvo_row(p, 2.5, p.map_y - p.laser_dis, phi=np.pi / 2)]
    r11 = [_scan(s[None], 0 if s[3] != np.pi / 2 else 1) for s in rows]
    B["L11_laser_dis"] = (np.concatenate([r for r, _ in r11]), np.concatenate([k for _, k in r11]), None)
    return B


def laser_variants(p, rows, k_slope=K_SLOPE, k_steep=K_STEEP):
    """the restated laser at the lanes over the perturbation set P -> (base [L, R], variants [V, L, R]): the slope
    tan(phi) +- k ulps (k <= k_slope, or <= k_steep on the rays with |m| >= 1e3, sampled at powers of two), the ray angle
    +- 1 ulp (the step's Divisor), each corner bearing +- 1 ulp (libdevice against glibc acos)."""
    ph = ray_angles(p, rows)
    m = c_tan(ph)
    th = corner_bearings(p, rows)
    base = fake_laser(p, rows)
    steep = np.abs(m) >= 1e3
    V = []
    ks = sorted({j for j in range(1, k_slope + 1)} | {2 ** i for i in range(int(np.log2(k_steep)) + 1)})
    for j in ks:
        for sg in (1, -1):
            kk = np.where(steep | (j <= k_slope), sg * j, 0)
            V.append(fake_laser(p, rows, m=E.ulps(m, kk), ray_phi=ph, th=th))
    for sg in (1, -1):
        q = E.ulps(ph, sg)
        V.append(fake_laser(p, rows, ray_phi=q, th=th))
    for c in range(4):
        for sg in (1, -1):
            t = th.copy()
            t[:, c] = E.ulps(t[:, c], sg)
            V.append(fake_laser(p, rows, m=m, ray_phi=ph, th=t))
    return base, np.stack(V)


# ------------------------------------------------------------------------------------------------------ legality at equality
def draw3(seed, gid, ep, block):
    """draw2's pair plus the 22-bit radius draw of an obstacle candidate (ugvo.cu / ugvo.c draw3)."""
    from oracle import oracle
    r = oracle.philox([gid & 0xFFFFFFFF, gid >> 32, ep, block], [seed & 0xFFFFFFFF, seed >> 32]).astype(np.int64)
    u0 = ((r[0] >> 5) * 67108864.0 + (r[1] >> 6)) * (1.0 / 9007199254740992.0)
    u1 = ((r[2] >> 5) * 67108864.0 + (r[3] >> 6)) * (1.0 / 9007199254740992.0)
    low = ((r[0] & 31) << 17) | ((r[1] & 63) << 11) | ((r[2] & 31) << 6) | (r[3] & 63)
    return float(u0), float(u1), float(low) * (1.0 / 4194304.0)


def _start_target(p, gid, s_st, seed=E.SEED):
    lo, hx, hy = p.st_margin, p.map_x - p.st_margin, p.map_y - p.st_margin
    u0, u1 = draw2(seed, gid, 0, 0)
    sx, sy = lerp_u(lo, hx, u0), lerp_u(lo, hy, u1)
    tx, ty = sx, sy
    for j in range(64):
        if not norm2(tx - sx, ty - sy) < s_st:
            break
        u0, u1 = draw2(seed, gid, 0, 1 + j)
        tx, ty = lerp_u(lo, hx, u0), lerp_u(lo, hy, u1)
    return sx, sy, tx, ty


def _sum_on(r, target, k):
    """a double s with fl(r + s) == ulps(target, k), or None."""
    want = float(E.ulps(np.float64(target), k))
    s = want - r
    for j in range(-4, 5):
        c = float(E.ulps(np.float64(s), j))
        if r + c == want:
            return c
    return None


def equality_cases(p, n_inst=6, ks=(-2, -1, 0, 1, 2)):
    """(label, gid, parameter overrides, k) with a decision of the reset on an equality: `start` -- fl(r +
    safety_dis_st) on the distance from the start to obstacle 0's first candidate, +k ulps (illegal for k >= 0);
    `target` -- safety_dis_st on the distance of the first target candidate (accepted for k <= 0); instances whose other
    tests are far from deciding."""
    out = []
    lo, hx, hy = p.st_margin, p.map_x - p.st_margin, p.map_y - p.st_margin
    found = {"start": 0, "target": 0}
    for gid in range(400):
        if min(found.values()) >= n_inst:
            break
        u0, u1 = draw2(E.SEED, gid, 0, 0)
        sx, sy = lerp_u(lo, hx, u0), lerp_u(lo, hy, u1)
        u0, u1 = draw2(E.SEED, gid, 0, 1)
        t1x, t1y = lerp_u(lo, hx, u0), lerp_u(lo, hy, u1)
        dt1 = float(norm2(t1x - sx, t1y - sy))
        if found["target"] < n_inst and dt1 > 1.0:
            found["target"] += 1
            for k in ks:
                out.append(("target", gid, {"safety_dis_st": float(E.ulps(np.float64(dt1), k))}, k))
        if found["start"] < n_inst:
            a, b, c = draw3(E.SEED, gid, 0, 1000)
            cx, cy, r = lerp_u(0., p.map_x, a), lerp_u(0., p.map_y, b), lerp_u(p.r_min, p.r_max, c)
            d = float(norm2(sx - cx, sy - cy))
            ss = [_sum_on(r, d, k) for k in ks]
            if d - r < 0.3 or any(s is None for s in ss):
                continue
            _, _, tx, ty = _start_target(p, gid, max(ss))
            if any(_start_target(p, gid, s)[2:] != (tx, ty) for s in ss) or norm2(tx - cx, ty - cy) < r + max(ss) + 0.05:
                continue
            found["start"] += 1
            for k, s in zip(ks, ss):
                out.append(("start", gid, {"safety_dis_st": s}, k))
    return out


def block_decision(p, label, rows):
    """for the blocks whose two outcomes give the same range: the decisive test on each lane (None for the others).
    L2: the sign of the dot product of the behind test for the ray along the normal's foot (the heading ray of the
    kernel's test is the ray itself; the centre's offset along it is what the scan moves); L3: the in-range cut;
    L11: `t < xm` (`t > 0` on the left wall)."""
    x, y = rows[:, 0], rows[:, 1]
    if label == "L3_in_range":
        return norm2(x - rows[:, 8], y - rows[:, 9]) > p.laser_dis + rows[:, 10]
    if label == "L11_laser_dis":
        xs = np.where(rows[:, 3] == 0.0, x + p.laser_dis, np.where(rows[:, 3] == np.pi, x - p.laser_dis, y + p.laser_dis))
        lim = np.where(rows[:, 3] == 0.0, p.map_x, np.where(rows[:, 3] == np.pi, 0.0, p.map_y))
        return np.where(rows[:, 3] == np.pi, xs > lim, xs < lim)
    if label == "L2_perpendicular":
        ph = ray_angles(p, rows)
        best = np.argmin(np.abs(np.cos(ph) * (rows[:, 8:9] - x[:, None]) + np.sin(ph) * (rows[:, 9:10] - y[:, None])), axis=1)
        a = ph[np.arange(len(rows)), best]
        return np.cos(a) * (rows[:, 8] - x) + np.sin(a) * (rows[:, 9] - y) < 0
    return None
