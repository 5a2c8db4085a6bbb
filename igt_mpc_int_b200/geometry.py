"""Host-side geometry of the four-way intersection (numpy, no CasADi).

Mirrors what the reference derives from common/fourwayint.yaml and evaluate.py:40-62:
start / goal poses per region, the 12 routes as straight-arc-straight paths, the curvature
parameters (b0, b1, Kval) that mpc.py:183-200 turns into a `pw_const`, the closed form
s -> (x, y) of common/utils.py:532-586 (`frenet2global`) and the route heading used by
common/constant_acceleration_model.py:46-64.

Everything here is plain arithmetic on a handful of floats per vehicle; it feeds numbers to
the CUDA solver and is not itself on the GPU path.
"""
import math
import numpy as np

ROAD_WIDTH = 11.4      # fourwayint.yaml:3
ROAD_LENGTH = 50.0     # fourwayint.yaml:5
CA_RADIUS = 2.8        # fourwayint.yaml:9
L_R = 2.235            # fourwayint.yaml:17
L_F = 2.235            # fourwayint.yaml:18

LEFT = ('12', '23', '34', '41')
RIGHT = ('14', '21', '32', '43')
STRAIGHT = ('13', '24', '31', '42')
ROUTES = LEFT + RIGHT + STRAIGHT

# Exit-lane coordinate the reference's frenet2global returns after the arc: it reads the last
# sample of its generated reference track (`ref['x'][-1]` / `ref['y'][-1]`, utils.py:558), which is
# a few millimetres off the nominal lane centre.  Values captured by running the reference's
# ReferenceGenerator (tests/golden/geometry.npz pins them).
EXIT_COORD = {
    '12': 27.89571278670408, '23': 2.8042872132959236, '34': 22.10428721329592, '41': 8.595712786704077,
    '14': 22.099438308054523, '21': 8.600561691945474, '32': 27.90056169194547, '43': 2.7994383080545244,
}

# scenario route-pair sets, common/utils.py:142-149
SCENARIOS = {
    1: [('13', '23'), ('24', '34'), ('31', '41'), ('42', '12')],
    2: [('12', '41'), ('23', '12'), ('34', '23'), ('41', '34')],
    3: [('13', '24'), ('24', '31'), ('31', '42'), ('42', '13')],
    4: [('12', '32'), ('23', '43'), ('34', '14'), ('41', '21')],
    5: [('13', '43'), ('24', '14'), ('31', '21'), ('42', '32')],
    6: [('13', '41'), ('24', '12'), ('31', '23'), ('42', '34')],
    7: [('12', '34'), ('23', '41'), ('34', '12'), ('41', '23')],
    8: [('12', '31'), ('23', '42'), ('34', '13'), ('41', '24')],
}


def start_pose(region, W=ROAD_WIDTH, L=ROAD_LENGTH, ca=CA_RADIUS):
    """evaluate.py:59-62 -- default (s = 0) pose of a vehicle entering from `region`."""
    region = str(region)
    if region == '1':
        return (0.0, ca, 0.0)
    if region == '2':
        return (L / 2 - W / 2 + ca, L / 2 + W / 2, -math.pi / 2)
    if region == '3':
        return (L, W - ca, -math.pi)
    if region == '4':
        return (L / 2 + W / 2 - ca, (W - L) / 2, math.pi / 2)
    raise ValueError('invalid region %r' % region)


def goal_pose(region, W=ROAD_WIDTH, L=ROAD_LENGTH, ca=CA_RADIUS):
    """evaluate.py:51-54."""
    region = str(region)
    if region == '1':
        return (0.0, W - ca, -math.pi)
    if region == '2':
        return (L / 2 + W / 2 - ca, L / 2 + W / 2, math.pi / 2)
    if region == '3':
        return (L, ca, 0.0)
    if region == '4':
        return (L / 2 - W / 2 + ca, (W - L) / 2, -math.pi / 2)
    raise ValueError('invalid region %r' % region)


def turn_sign(route):
    return 1 if route in LEFT else (-1 if route in RIGHT else 0)


def curvature_params(route, W=ROAD_WIDTH, L=ROAD_LENGTH, ca=CA_RADIUS):
    """(b0, b1, Kval) of the piecewise-constant curvature, mpc.py:183-200 / SURVEY 8(a3).

    left : b0 = (L-W)/2,             r = W - ca (= 8.6),  Kval = +1/r
    right: b0 = (L-W)/2 - (W - ca),  r = W      (= 11.4), Kval = -1/r   (ds_right = W - ca,
           evaluate.py:48, :440)
    straight: K == 0 (returned with breakpoints at +inf so that no comparison ever fires).
    """
    sgn = turn_sign(route)
    if sgn == 0:
        return (1e30, 1e30, 0.0)
    if sgn > 0:
        b0 = (L - W) / 2
        r = W - ca
    else:
        b0 = (L - W) / 2 - (W - ca)
        r = (W - ca) + ca
    return (b0, b0 + r * math.pi / 2, sgn / r)


def frenet2global(s, route, ey=0.0, W=ROAD_WIDTH, L=ROAD_LENGTH, ca=CA_RADIUS, exit_coord=None):
    """s (and lateral offset ey, positive to the left) -> (x, y, path heading).

    Closed form of common/utils.py:532-586.  `exit_coord`, when given, replaces the nominal
    exit-lane coordinate after the arc by the value the reference reads from its generated
    track (`ref['x'][-1]` / `ref['y'][-1]`, utils.py:558 -- e.g. 27.8957 instead of 27.9 on
    route 12); None keeps the nominal lane centre.
    """
    x0, y0, th0 = start_pose(route[0], W, L, ca)
    t0 = (math.cos(th0), math.sin(th0))
    n0 = (-t0[1], t0[0])
    sgn = turn_sign(route)
    b0, b1, K = curvature_params(route, W, L, ca)
    if sgn == 0 or s < b0:
        x, y, th = x0 + s * t0[0], y0 + s * t0[1], th0
    else:
        r = 1.0 / abs(K)
        cx, cy = x0 + b0 * t0[0] + sgn * r * n0[0], y0 + b0 * t0[1] + sgn * r * n0[1]
        if s <= b1:
            phi = (s - b0) / r
            x = cx + r * (math.sin(phi) * t0[0] - sgn * math.cos(phi) * n0[0])
            y = cy + r * (math.sin(phi) * t0[1] - sgn * math.cos(phi) * n0[1])
            th = th0 + sgn * phi
        else:
            th = th0 + sgn * math.pi / 2
            t1 = (sgn * n0[0], sgn * n0[1])
            x = cx + r * t0[0] + (s - b1) * t1[0]
            y = cy + r * t0[1] + (s - b1) * t1[1]
            if exit_coord is not None:
                if abs(t1[0]) < 0.5:
                    x = exit_coord
                else:
                    y = exit_coord
    if ey != 0.0:
        x += -math.sin(th) * ey
        y += math.cos(th) * ey
    return x, y, th


def route_descriptor(route, W=ROAD_WIDTH, L=ROAD_LENGTH, ca=CA_RADIUS, exit_coord=None):
    """The 12 numbers the device-side closed loop needs to evaluate `frenet2global_xy` and `route_heading` for this
    route (csrc/episode.cuh route_xy / route_heading): x0, y0, t0x, t0y, turn sign, b0, b1, r, exit axis (0: x, 1: y,
    -1: none), exit coordinate, start heading th0 (stored, not recovered with atan2, so that the device heading is
    bit-identical), flip (1.0 on routes 32 and 41, whose headings the planner takes abs() of, mpc.py:250-253)."""
    x0, y0, th0 = start_pose(route[0], W, L, ca)
    t0 = (math.cos(th0), math.sin(th0))
    sgn = turn_sign(route)
    flip = 1.0 if route in ('32', '41') else 0.0
    if sgn == 0:
        return [x0, y0, t0[0], t0[1], 0.0, 1e30, 1e30, 1.0, -1.0, 0.0, th0, flip]
    b0, b1, K = curvature_params(route, W, L, ca)
    t1x = sgn * (-t0[1])
    axis = -1.0 if exit_coord is None else (0.0 if abs(t1x) < 0.5 else 1.0)
    return [x0, y0, t0[0], t0[1], float(sgn), b0, b1, 1.0 / abs(K), axis, 0.0 if exit_coord is None else float(exit_coord),
            th0, flip]


def frenet2global_xy(s, route, W=ROAD_WIDTH, L=ROAD_LENGTH, ca=CA_RADIUS, exit_coord=None):
    """`frenet2global` (lane centre, ey = 0) for an array of arc lengths: s[...] -> x[...], y[...]."""
    s = np.asarray(s, dtype=np.float64)
    x0, y0, th0 = start_pose(route[0], W, L, ca)
    t0 = (math.cos(th0), math.sin(th0))
    n0 = (-t0[1], t0[0])
    sgn = turn_sign(route)
    if sgn == 0:
        return x0 + s * t0[0], y0 + s * t0[1]
    b0, b1, K = curvature_params(route, W, L, ca)
    r = 1.0 / abs(K)
    cx, cy = x0 + b0 * t0[0] + sgn * r * n0[0], y0 + b0 * t0[1] + sgn * r * n0[1]
    phi = (s - b0) / r
    xa = cx + r * (np.sin(phi) * t0[0] - sgn * np.cos(phi) * n0[0])
    ya = cy + r * (np.sin(phi) * t0[1] - sgn * np.cos(phi) * n0[1])
    t1 = (sgn * n0[0], sgn * n0[1])
    xe = cx + r * t0[0] + (s - b1) * t1[0]
    ye = cy + r * t0[1] + (s - b1) * t1[1]
    if exit_coord is not None:
        if abs(t1[0]) < 0.5:
            xe = np.full_like(s, exit_coord)
        else:
            ye = np.full_like(s, exit_coord)
    x = np.where(s < b0, x0 + s * t0[0], np.where(s <= b1, xa, xe))
    y = np.where(s < b0, y0 + s * t0[1], np.where(s <= b1, ya, ye))
    return x, y


def route_heading(s, route, W=ROAD_WIDTH, L=ROAD_LENGTH, ca=CA_RADIUS):
    """The path heading of `frenet2global` (its third output) for an array of arc lengths: th0 before the arc,
    th0 + sgn * phi on it, th0 + sgn * pi / 2 after it.  No abs() flip (that is the planner's, mpc.py:250-253)."""
    s = np.asarray(s, dtype=np.float64)
    th0 = start_pose(route[0], W, L, ca)[2]
    sgn = turn_sign(route)
    if sgn == 0:
        return np.full_like(s, th0)
    b0, b1, K = curvature_params(route, W, L, ca)
    r = 1.0 / abs(K)
    phi = (s - b0) / r
    return np.where(s < b0, th0, np.where(s <= b1, th0 + sgn * phi, th0 + sgn * math.pi / 2))


def rectangles_overlap(p, q, h=4.47, w=2.0):
    """Do the h x w rectangles centred at (x, y) with heading psi (length along the heading, csrc/obca.cuh) overlap?
    p, q[..., 3] = (x, y, psi) -> bool[...].  Separating-axis test over the four face normals; rectangles that only
    touch do not overlap."""
    p = np.asarray(p, dtype=np.float64); q = np.asarray(q, dtype=np.float64)
    cp, sp, cq, sq = np.cos(p[..., 2]), np.sin(p[..., 2]), np.cos(q[..., 2]), np.sin(q[..., 2])
    dx, dy = q[..., 0] - p[..., 0], q[..., 1] - p[..., 1]
    hl, hw = h / 2, w / 2
    sep = np.zeros(np.broadcast(p[..., 0], q[..., 0]).shape, dtype=bool)
    for ax, ay, he in ((cp, sp, hl), (-sp, cp, hw)):              # p's face normals: p's half-extent he along them
        ho = hl * np.abs(ax * cq + ay * sq) + hw * np.abs(-ax * sq + ay * cq)
        sep |= np.abs(ax * dx + ay * dy) >= he + ho
    for ax, ay, ho in ((cq, sq, hl), (-sq, cq, hw)):              # q's face normals
        he = hl * np.abs(ax * cp + ay * sp) + hw * np.abs(-ax * sp + ay * cp)
        sep |= np.abs(ax * dx + ay * dy) >= he + ho
    return ~sep


def scenario_routes(sc, rotation, order):
    """Route pair of scenario `sc` (1..8): `rotation` picks one of the four rotated pairs
    (utils.py:177-179 does this with an unseeded random.choice) and `order` the agent order
    (the reference's list(set) order is unspecified)."""
    a, b = SCENARIOS[int(sc)][int(rotation) % 4]
    return [a, b] if int(order) % 2 == 0 else [b, a]


def scenario_encoding(routes):
    """common/utils.py:84-169 -- signed scenario index (+-m) for a two-vehicle route pair."""
    pair = {routes[0], routes[1]}
    m = None
    for k, sets in SCENARIOS.items():
        if any(pair == set(p) for p in sets):
            m = k
            break
    if m is None:
        raise ValueError('Scenario not found')
    vh1, vh2 = routes[0][0], routes[1][0]
    if m == 1:
        if routes[0] == '42':
            vh1 = '0'
        elif routes[1] == '42':
            vh2 = '0'
    elif m == 2:
        if routes[0] == '12' and routes[1] == '41':
            vh1 = '5'
        elif routes[1] == '12' and routes[0] == '41':
            vh2 = '5'
    elif m == 3:
        if routes[0] == '13' and routes[1] == '42':
            vh2 = '0'
        elif routes[1] == '13' and routes[0] == '42':
            vh1 = '0'
    if m < 4 or m == 7:
        return [m, -m] if int(vh1) < int(vh2) else [-m, m]
    if m in (4, 6, 8):
        return [m, -m] if routes[0] in LEFT else [-m, m]
    return [m, -m] if routes[0] in STRAIGHT else [-m, m]      # m == 5


def constant_acceleration_forecast(s0, v0, a, route, N, dt=0.1, v_min=-2.0, v_max=20.0,
                                   exit_coord=None):
    """common/constant_acceleration_model.py:66-80 -- N+1 forecast points (x, y, s, v) of a
    vehicle rolling s += v dt + a dt^2/2, v = clip(v + a dt, v_min, v_max)
    (fourwayint.yaml:23-24) along its route."""
    out = np.empty((N + 1, 4))
    s, v = float(s0), float(v0)
    x, y, _ = frenet2global(s, route, exit_coord=exit_coord)
    out[0] = (x, y, s, v)
    for k in range(N):
        s += v * dt + 0.5 * a * dt * dt
        v = min(max(v + a * dt, v_min), v_max)
        x, y, _ = frenet2global(s, route, exit_coord=exit_coord)
        out[k + 1] = (x, y, s, v)
    return out


def filter_obstacle(ego_xy, ego_heading, obs_xy):
    """common/utils.py:365-388 -- if the other vehicle's current position is behind the ego
    (negative dot product with the ego heading vector) all its forecast points become
    (-20, -20).  obs_xy[N+1, 2]; returns a new array."""
    dx, dy = obs_xy[0, 0] - ego_xy[0], obs_xy[0, 1] - ego_xy[1]
    if dx * math.cos(ego_heading) + dy * math.sin(ego_heading) < 0:
        return np.full_like(obs_xy, -20.0)
    return np.array(obs_xy, copy=True)
