"""Every step kernel against the fp64 oracle on pairs placed EXACTLY on the distance thresholds, and on pairs whose fp32
coordinates round the wrong way, at the distances from the map centre where the kernels' fp32 guards change.

Each environment holds one focal UAV i and probes around it, all at their positions AFTER the move:
  T_le   target at d2 in {s*, s* +- 1 ulp} of s* = exact_sq_threshold(dp, <=)     obs_mask (the observation block)
  T_lt   target at d2 in {s*, s* +- 1 ulp} of s* = exact_sq_threshold(dp, <)      cover_mask, covered, tracker_cnt
  U_cn   UAV j < i (moved first) at the same placements around dc                  comm_mask, new position
  U_co   UAV j > i (moves after i) whose OLD position sits there around dc          comm_mask, old position
  U_dup  UAV around 2 dp                                                           dup_mask
  U_nb   UAV around dp                                                             nbr_mask (the PMI reward's neighbour bits)
  T_ah   target truly inside dp whose fp32 offset from the map centre rounds OUTWARD (a hit pushed out)
  T_am   target truly outside dp whose fp32 offset rounds INWARD (a miss pushed in)
Offsets are axis-aligned (a sub-micrometre perpendicular component reaches s* +- 1 ulp where no square does),
Pythagorean diagonals ((120, 160) -> 200, (300, 400) -> 500, (240, 320) -> 400 at the shipped constants), or zero.

Every entity whose new position enters a decision moves along a cardinal heading (cos / sin are +-1, or ~1e-16 that the
addition absorbs), so `x + dt v cos h` is the same double in the oracle and in every kernel: the test checks that first.
A partner j > i is seen by i at its OLD position; its new position gets a non-cardinal heading (the 64 x 64 fast kernel
rebuilds the old position from it in fp32) and is kept at least ~2e-6 relative away from every threshold.

Distances from the map centre: in the map, and just inside / just outside 1.3 * the half map (the tile kernel's first
band), r_tile, r_fast (a marker UAV sets the environment's largest offset R; one environment keeps its probes at the
centre and only the marker near r_fast), 32 000 m, and the generic kernel's prefilter radius rmax = 32 768 m
(|x - cx| == rmax exactly, and the next double).
"""
import math

import numpy as np
import pytest
import torch

from gpu_util import MASKS, max_scaled_err, oracle_params_from_config

TOL_TIGHT = 2e-6
CARD = (0.0, math.pi / 2, math.pi, -math.pi / 2)

# scenario constants: (dp, dc, uav v_max) with dt = 1 and the target speed 5
CONSTS = {
    "shipped": (200.0, 500.0, 20.0),
    "nonint": (140.003, 420.009, 20.0),     # s_le != fl(thr^2) for dp, 2 dp and dc; s_dp_lt two doubles below s_dp_le
    "wide_dup": (200.0, 300.0, 20.0),       # 2 dp > dc + dt v: the duplicate radius is the widest UAV-UAV test
    "nondyadic": (200.0, 500.0, 20.3),      # dt v = 20.3 is not a binary fraction: the moves round
}
# (step path, n, m): 4 small-swarm, 1 generic (64x64 and 10x10 compile-time, others run-time), 2 fast, 3 tile
KERNELS = [(4, 10, 10), (4, 16, 16), (4, 7, 5), (4, 3, 16), (4, 16, 2),
           (1, 64, 64), (1, 10, 10), (1, 33, 7), (1, 128, 150), (2, 64, 64), (3, 64, 64)]
RANGES = ("map", "tile0_in", "tile0_out", "rtile_in", "rtile_out", "rfast_in", "rfast_out", "wide", "r32000",
          "rmax_in", "rmax_out")
ON_KINDS = ("T_le", "T_lt", "U_cn", "U_co", "U_dup", "U_nb")
ADV_KINDS = ("T_ah", "T_am")
MASK_OF = {"T_le": "obs_mask", "T_lt": "cover_mask", "U_cn": "comm_mask", "U_co": "comm_mask", "U_dup": "dup_mask",
           "U_nb": "nbr_mask", "T_ah": "obs_mask", "T_am": "obs_mask"}
AXIS_DIR = {"T_le": (1, 0), "T_lt": (-1, 0), "U_cn": (0, 1), "U_co": (0, -1), "U_dup": (0, 1), "U_nb": (-1, 0)}
DIAG_DIR = {"T_le": (0.6, 0.8), "T_lt": (-0.8, 0.6), "U_cn": (-0.6, 0.8), "U_co": (0.8, -0.6), "U_dup": (0.8, 0.6),
            "U_nb": (-0.6, -0.8)}


# ---------------------------------------------------------------------------------------------------- host arithmetic
def exact_sq_threshold(thr, strict):
    """Python copy of uavsim.cu's exact_sq_threshold: the largest double s with sqrt(s) <= thr (< thr if strict)."""
    s = thr * thr
    ok = (lambda v: math.sqrt(v) < thr) if strict else (lambda v: math.sqrt(v) <= thr)
    while not ok(s):
        s = math.nextafter(s, -math.inf)
    while ok(math.nextafter(s, math.inf)):
        s = math.nextafter(s, math.inf)
    return s


def ulps(v, k):
    for _ in range(abs(k)):
        v = math.nextafter(v, math.inf if k > 0 else -math.inf)
    return v


def d2_of(ax, ay, bx, by):
    """The oracle's squared distance: (x1 - x2)**2 + (y1 - y2)**2 in fp64, no contraction."""
    dx, dy = ax - bx, ay - by
    return dx * dx + dy * dy


def f32_d2(ax, ay, bx, by, cx, cy):
    """The kernels' fp32 squared distance: offsets from the map centre rounded to fp32, differenced in fp32, then
    fma(dx, dx, dy * dy) (the product of two floats is exact in fp64, so one rounding of the sum is the fma)."""
    f = np.float32
    dx = f(f(ax - cx) - f(bx - cx))
    dy = f(f(ay - cy) - f(by - cy))
    return float(f(float(dx) * float(dx) + float(f(dy * dy))))


def f32_floor(v):
    g = np.float32(v)
    if float(g) > v:
        g = np.nextafter(g, np.float32(-np.inf))
    return g


def pre_move(X, step):
    """A double x with fl(x + step) == X (so the move lands on X exactly in the oracle and the kernels)."""
    x0 = X - step
    for k in range(64):
        for x in (ulps(x0, k), ulps(x0, -k)):
            if x + step == X:
                return x
    raise AssertionError("no pre-move coordinate lands on %r (step %r)" % (X, step))


def pre_move_cardinal(X, Y, h, dtv):
    """Pre-move coordinates for a cardinal heading, starting with h: a move towards zero across a power of two cannot
    land on every double, the opposite heading always can."""
    for hh in (h,) + tuple(c for c in CARD if c != h):
        try:
            return pre_move(X, dtv * math.cos(hh)), pre_move(Y, dtv * math.sin(hh)), hh
        except AssertionError:
            pass
    raise AssertionError("no cardinal move lands on (%r, %r)" % (X, Y))


def solve_offset(x0, y0, S, ux, uy, side=0):
    """(x, y) near (x0, y0) + sqrt(S) (ux, uy) with d2_of(x, y, x0, y0) == S exactly (axis-aligned offsets always; a
    diagonal where S is reachable, else the nearest reachable d2 on the side `side`)."""
    if S == 0.0:
        return x0, y0
    d = math.sqrt(S)
    K = 24

    def around(v):
        up, dn = [v], [v]
        for _ in range(K):
            up.append(math.nextafter(up[-1], math.inf))
            dn.append(math.nextafter(dn[-1], -math.inf))
        return np.array(dn[::-1][:-1] + up)

    X, Y = around(x0 + d * ux), around(y0 + d * uy)
    DX, DY = X - x0, Y - y0
    D2 = DX[:, None] * DX[:, None] + DY[None, :] * DY[None, :]
    hit = np.argwhere(D2 == S)
    if len(hit):
        k = hit[np.argmin(np.abs(hit - K).sum(1))]
        return float(X[k[0]]), float(Y[k[1]])
    if ux != 0 and uy != 0:
        # a diagonal reaches only every few doubles (both coordinates move in steps of their ulp): the reachable d2
        # nearest to S on the side `side` asks for (0: at or below S)
        sel = (D2 > S) if side > 0 else (D2 < S)
        k = np.argwhere(sel)[np.argmin(np.abs(D2[sel] - S))]
        return float(X[k[0]]), float(Y[k[1]])
    # no square of a coordinate difference lands on S: take the primary axis just below and add a sub-micrometre
    # perpendicular offset whose square supplies the last ulps
    P, p0 = (X, x0) if uy == 0 else (Y, y0)
    q0 = y0 if uy == 0 else x0
    DP = P - p0
    base = DP * DP
    ok = np.nonzero((base < S) & (base <= ulps(S, -2)))[0]
    a = float(P[ok[np.argmax(base[ok])]])
    r = S - (a - p0) * (a - p0)
    q = q0 + math.sqrt(r)
    for k in range(32):
        for qq in (ulps(q, k), ulps(q, -k)):
            pair = (a, qq) if uy == 0 else (qq, a)
            if d2_of(pair[0], pair[1], x0, y0) == S:
                return pair
    raise AssertionError("no placement for d2 = %r" % S)


def adversarial(x0, y0, cx, cy, S, thr, hit):
    """A target whose fp32 offset rounds the wrong way: `hit` -> true d2 <= S (east of the focal UAV, its offset rounds
    up while the focal one rounds down: the fp32 distance is pushed OUT); else true d2 > S (west, pushed IN).
    Returns the candidate with the largest push past thr^2."""
    best = None
    x0r = x0 - cx
    for k in range(160):
        b = 17.0 + 0.37 * k
        y1 = y0 + b
        dyt = y1 - y0
        A = math.sqrt(S - dyt * dyt)
        v = x0r + A + 0.48 * float(np.spacing(np.float32(x0r + A))) if hit else x0r - A + 0.48 * float(np.spacing(np.float32(x0r - A)))
        G = f32_floor(v)
        if not hit and float(G) >= v:
            G = np.nextafter(G, np.float32(-np.inf))
        for g in (G, np.nextafter(G, np.float32(-np.inf))):
            x1 = cx + (float(g) - 0.48 * float(np.spacing(g)))
            t = d2_of(x1, y1, x0, y0)
            s = f32_d2(x1, y1, x0, y0, cx, cy)
            if hit and t <= S:
                score = s - thr * thr
            elif not hit and t > S:
                score = thr * thr - s
            else:
                continue
            if best is None or score > best[0]:
                best = (score, x1, y1)
            break
    assert best is not None and best[0] > 0, "no adversarial placement"
    return best[1], best[2]


# ---------------------------------------------------------------------------------------------------- scene building
class Limits:
    """The radii the kernels switch at, as uavsim.cu computes them."""

    def __init__(self, dp, dc, x_max=2000.0, y_max=2000.0):
        self.cx, self.cy = x_max / 2, y_max / 2
        rf = min(2e-6 * 16777216.0 * min(dp, dc), 32768.0)
        self.r_fast = float(np.float32(rf))
        self.r_tile = float(np.float32(min(rf, 4096.0)))
        cmax = max(self.cx, self.cy)
        r0 = min(1.3 * cmax, self.r_tile)
        t0 = np.float32(r0)
        if float(t0) > r0:
            t0 = np.nextafter(t0, np.float32(0))
        self.tile0 = float(t0)

    def marker(self, rng_name):
        """(x offset of the marker UAV from the centre, x offset of the cluster), or None for no marker."""
        nxt = lambda r: float(np.nextafter(np.float32(r), np.float32(np.inf)))  # noqa: E731
        table = {"tile0_in": self.tile0, "tile0_out": nxt(self.tile0), "rtile_in": self.r_tile,
                 "rtile_out": nxt(self.r_tile), "rfast_in": self.r_fast, "rfast_out": nxt(self.r_fast),
                 "wide": self.r_fast, "rmax_in": 32768.0, "rmax_out": math.nextafter(32768.0, math.inf)}
        if rng_name == "map":
            return None, 200.0
        if rng_name == "r32000":
            return None, 31500.0
        r = table[rng_name]
        return r, (200.0 if rng_name == "wide" else r - 700.0)


class Scenario:
    def __init__(self, name, n, m):
        self.name, self.n, self.m = name, n, m
        dp, dc, v = CONSTS[name]
        self.dp, self.dc = dp, dc
        self.dtv, self.dtv_t = 1.0 * v, 1.0 * 5.0
        self.lim = Limits(dp, dc)
        self.S = {"le": exact_sq_threshold(dp, False), "lt": exact_sq_threshold(dp, True),
                  "dc": exact_sq_threshold(dc, False), "2dp": exact_sq_threshold(2 * dp, False)}
        self.kind_S = {"T_le": self.S["le"], "T_lt": self.S["lt"], "U_cn": self.S["dc"], "U_co": self.S["dc"],
                       "U_dup": self.S["2dp"], "U_nb": self.S["le"], "T_ah": self.S["le"], "T_am": self.S["le"]}
        self.kind_thr = {"T_le": dp, "T_lt": dp, "U_cn": dc, "U_co": dc, "U_dup": 2 * dp, "U_nb": dp,
                         "T_ah": dp, "T_am": dp}

    def config(self, method):
        from marl_uavs_targets_tracking_b200 import default_config
        dp, dc, v = CONSTS[self.name]
        return default_config(method, self.n, self.m, uav__dp=dp, uav__dc=dc, uav__v_max=v)

    def index_cases(self):
        """(focal i, partner below i or None, partner above i or None): adjacent pairs, j = 0 and j = n - 1, and the pairs
        across the 32-partner chunks and 64-bit neighbour words."""
        n = self.n
        c = [(n // 2, n // 2 - 1, n // 2 + 1), (n - 1, 0, None), (0, None, n - 1)]
        if n >= 33:
            c += [(32, 31, 33), (31, 30, 32), (96, 95, 97) if n > 97 else (32, 0, n - 1)]
        if n >= 65:
            c += [(64, 63, 65), (63, 62, 64), (127, 126, None) if n >= 128 else (64, 0, n - 1)]
        if n >= 128:
            c += [(0, None, 127), (126, 64, 127)]
        return [tuple(None if v is not None and (v < 0 or v >= n) else v for v in t) for t in c]

    def scenes(self):
        """One scene per environment: (range, offset variant, geometry, index case, rotation).  The rotation decides which
        probe kinds come first; a swarm too small for all of them gets more blocks, so that every kind meets every range
        on both sides of its threshold."""
        out = []
        cases = self.index_cases()
        reps = 1 if self.n >= 8 else 2
        blk = 0

        def case_for(b):  # the block's first UAV kind needs a partner on its side of i
            first = ("U_cn", "U_co", "U_dup", "U_nb")[b % 4]
            for q in range(len(cases)):
                c = cases[(b + q) % len(cases)]
                if (first != "U_cn" or c[1] is not None) and (first != "U_co" or c[2] is not None):
                    return c
            return cases[b % len(cases)]
        for rng_name in RANGES:
            for _ in range(reps):
                for geom in ("axis", "diag"):
                    for vi, var in enumerate((0, 1, -1)):
                        out.append((rng_name, var, geom, case_for(blk), 3 * blk + vi))
                    blk += 1
            out.append((rng_name, 0, "adv", case_for(blk), 3 * blk))
            blk += 1
        out.append(("map", 0, "zero", cases[0], 0))
        out.append(("map", 1, "zero", cases[1 % len(cases)], 3))
        return out


def build_env(sc, scene, seed):
    """Pre-move state of one environment, its probes [(kind, uav i, partner, intended d2)] and the entities that move
    along a non-cardinal heading."""
    rng_name, var, geom, (fi, jlo, jhi), rot = scene
    rs = np.random.default_rng(seed)
    n, m, L = sc.n, sc.m, sc.lim
    cx, cy = L.cx, L.cy
    uxn, uyn, uh = np.zeros(n), np.zeros(n), np.zeros(n)
    txn, tyn, th = np.zeros(m), np.zeros(m), np.zeros(m)
    uxo, uyo = {}, {}   # old positions set directly (non-cardinal movers)
    placed_u, placed_t = {}, set()
    marker_x, clx = L.marker(rng_name)

    # focal UAV: its offset from the centre rounds DOWN to fp32 by 0.48 ulp
    g0 = f32_floor(clx)
    x0 = cx + (float(g0) + 0.48 * float(np.spacing(g0)))
    y0 = cy + 37.0 + 0.25 * (rot % 4)
    uxn[fi], uyn[fi] = x0, y0
    placed_u[fi] = "focal"

    free_u = [j for j in range(n) if j != fi and j not in (jlo, jhi)]
    free_t = list(range(m))
    probes = []
    if geom == "adv":
        kinds = [k for k in ADV_KINDS]
    elif geom == "zero":
        kinds = ["T_le", "U_cn", "U_nb"]
    else:
        tk, uk = ["T_le", "T_lt"], ["U_cn", "U_co", "U_dup", "U_nb"]
        r = (rot // 3) % 4
        kinds = tk[rot % 2:] + tk[:rot % 2] + uk[r:] + uk[:r]  # which kinds fit in a small environment rotates
    if marker_x is not None:
        reserve = 1
    else:
        reserve = 0
    # partner indices: the chunk / word boundary pair takes the class the rotation gives it
    for kind in kinds:
        S0 = sc.kind_S[kind]
        if kind.startswith("T"):
            if not free_t:
                continue
            t = free_t.pop(0) if (rot + len(probes)) % 2 == 0 else free_t.pop()
            if kind in ADV_KINDS:
                tx, ty = adversarial(x0, y0, cx, cy, S0, sc.kind_thr[kind], kind == "T_ah")
                S = d2_of(tx, ty, x0, y0)
            else:
                S = 0.0 if geom == "zero" else ulps(S0, var)
                ux, uy = (AXIS_DIR if geom in ("axis", "zero") else DIAG_DIR)[kind]
                tx, ty = solve_offset(x0, y0, S, ux, uy, var)
                S = d2_of(tx, ty, x0, y0)
            txn[t], tyn[t] = tx, ty
            th[t] = CARD[rs.integers(4)]
            placed_t.add(t)
            probes.append((kind, fi, t, S))
            continue
        if kind == "U_cn":
            cand = [jlo] if jlo is not None and jlo not in placed_u else [j for j in free_u if j < fi]
        elif kind == "U_co":
            cand = [jhi] if jhi is not None and jhi not in placed_u else [j for j in free_u if j > fi]
        else:
            cand = [j for j in (jlo, jhi) if j is not None and j not in placed_u] + free_u
        cand = [j for j in cand if j not in placed_u]
        if len(placed_u) + reserve >= n or not cand:
            continue
        j = cand[0] if kind != "U_dup" else cand[-1]
        if j in free_u:
            free_u.remove(j)
        S = 0.0 if geom == "zero" else ulps(S0, var)
        ux, uy = (AXIS_DIR if geom in ("axis", "zero") else DIAG_DIR)[kind]
        px, py = solve_offset(x0, y0, S, ux, uy, var)
        S = d2_of(px, py, x0, y0)
        if kind == "U_co":
            uxo[j], uyo[j] = px, py
            if geom == "axis":     # straight away from i: the new position sits on dc + dt v, the prefilter radius
                uh[j] = -math.pi / 2
            else:                  # non-cardinal: the fp32 rebuild of the old position is inexact
                base = math.atan2(uy, ux)
                uh[j] = base + math.radians(rs.uniform(20, 70)) * (1 if rs.integers(2) else -1)
        else:
            uxn[j], uyn[j] = px, py
            uh[j] = CARD[rs.integers(4)]
        placed_u[j] = kind
        probes.append((kind, fi, j, S))
    uh[fi] = CARD[rs.integers(4)]

    # the marker UAV sets the environment's largest offset from the centre
    if marker_x is not None:
        j = [q for q in range(n) if q not in placed_u][-1]
        uxn[j], uyn[j] = cx + marker_x, cy + 1250.0
        uh[j] = math.pi / 2 if rs.integers(2) else -math.pi / 2
        placed_u[j] = "marker"
    # everything else parked at random in the map, cardinal headings
    for j in range(n):
        if j not in placed_u:
            uxn[j], uyn[j] = cx + rs.uniform(-900, 900), cy + rs.uniform(-900, 900)
            uh[j] = CARD[rs.integers(4)]
    for t in range(m):
        if t not in placed_t:
            txn[t], tyn[t] = cx + rs.uniform(-900, 900), cy + rs.uniform(-900, 900)
            th[t] = CARD[rs.integers(4)]

    noncard = [j for j in uxo if uh[j] not in CARD]
    ux, uy = np.zeros(n), np.zeros(n)
    for j in range(n):
        if j in uxo:
            ux[j], uy[j] = uxo[j], uyo[j]
            uxn[j] = uxo[j] + sc.dtv * math.cos(uh[j])
            uyn[j] = uyo[j] + sc.dtv * math.sin(uh[j])
        else:
            ux[j], uy[j], uh[j] = pre_move_cardinal(uxn[j], uyn[j], uh[j], sc.dtv)
    tx, ty = np.zeros(m), np.zeros(m)
    for t in range(m):
        tx[t], ty[t], th[t] = pre_move_cardinal(txn[t], tyn[t], th[t], sc.dtv_t)

    # a non-cardinal mover's NEW position (rounded differently by the oracle's libm and the kernels' sine) must stay
    # clear of every threshold it meets
    def clear(d2, thr):
        return abs(d2 / (thr * thr) - 1.0) > 4e-6
    for j in noncard:
        for k in range(n):
            if k != j:
                d2 = d2_of(uxn[j], uyn[j], uxn[k], uyn[k])
                assert all(clear(d2, t) for t in (sc.dp, 2 * sc.dp, sc.dc)), (scene, j, k)
                if k > j:
                    assert clear(d2_of(uxn[j], uyn[j], ux[k], uy[k]), sc.dc), (scene, j, k)
        for t in range(m):
            assert clear(d2_of(uxn[j], uyn[j], txn[t], tyn[t]), sc.dp), (scene, j, t)
    st = {"ux": ux, "uy": uy, "uh": uh, "ua": rs.integers(0, 12, n).astype(np.int32), "tx": tx, "ty": ty, "th": th}
    new = {"ux": uxn, "uy": uyn, "tx": txn, "ty": tyn}
    return st, new, probes, noncard


def build_batch(sc, E_min=0, group=1, seed=0):
    scenes = sc.scenes()
    while len(scenes) < E_min or (group > 1 and len(scenes) % group == 0):
        scenes.append(scenes[len(scenes) % len(sc.scenes())])  # a partial last group of the small-swarm kernel
    envs = [build_env(sc, s, seed * 100003 + e) for e, s in enumerate(scenes)]
    st = {k: np.stack([e[0][k] for e in envs]) for k in envs[0][0]}
    return scenes, envs, st


def env_R(st_e, new_e, cx, cy):
    """Largest |fp32 offset from the centre| over old and new positions: what the 64 x 64 kernels compare."""
    vals = [np.abs(np.float32(a - c)) for a, c in ((st_e["ux"], cx), (st_e["uy"], cy), (st_e["tx"], cx), (st_e["ty"], cy),
                                                    (new_e["ux"], cx), (new_e["uy"], cy), (new_e["tx"], cx), (new_e["ty"], cy))]
    return float(max(v.max() for v in vals))


def small_group(n, m):
    return min(32 // max(n, m), 8)


# ---------------------------------------------------------------------------------------------------- CPU check
@pytest.mark.parametrize("name", sorted(CONSTS))
def test_constructed_geometry_sits_on_the_thresholds(oracle, name):
    """No GPU: the construction places what it claims -- probe d2 on s* and one double to either side (or 0), fp32 rounding
    in the intended direction for the adversarial targets, the intended offset R from the centre, exact moves in the
    oracle -- and the oracle's decisions for every (kind, range) fall on both sides of the threshold."""
    shapes = sorted({(n, m) for _, n, m in KERNELS})
    for n, m in shapes:
        sc = Scenario(name, n, m)
        L = sc.lim
        assert sc.S["lt"] < sc.S["le"]
        if name == "nonint":
            assert sc.S["le"] != sc.dp * sc.dp and sc.S["dc"] != sc.dc * sc.dc and sc.S["2dp"] != (2 * sc.dp) ** 2
            assert sc.S["lt"] != math.nextafter(sc.S["le"], -math.inf)
        scenes, envs, st = build_batch(sc)
        P = oracle_params_from_config(sc.config("MAAC-G"), n, m)
        sides = {}
        for e, (scene, (st_e, new_e, probes, noncard)) in enumerate(zip(scenes, envs)):
            rng_name, var, geom = scene[0], scene[1], scene[2]
            for kind, i, j, S in probes:
                a = (new_e["ux"][i], new_e["uy"][i])
                b = (st_e["ux"][j], st_e["uy"][j]) if kind == "U_co" else \
                    (new_e["tx"][j], new_e["ty"][j]) if kind[0] == "T" else (new_e["ux"][j], new_e["uy"][j])
                d2 = d2_of(b[0], b[1], a[0], a[1])
                assert d2 == S, (scene, kind)
                S0 = sc.kind_S[kind]
                if geom == "axis":
                    assert d2 == ulps(S0, var), (scene, kind)
                elif geom == "diag":   # on s* +- 1 ulp where reachable, else the nearest reachable double on that side
                    want = ulps(S0, var)
                    assert d2 == want or ((d2 > S0) if var > 0 else (d2 < want)), (scene, kind)
                    assert abs(d2 - want) <= 16 * (ulps(S0, 1) - S0), (scene, kind)
                elif geom == "zero":
                    assert d2 == 0.0
                else:
                    thr2 = sc.kind_thr[kind] ** 2
                    s32 = f32_d2(b[0], b[1], a[0], a[1], L.cx, L.cy)
                    if kind == "T_ah":
                        assert d2 <= S0 and s32 > thr2, (scene, d2, s32)
                    else:
                        assert d2 > S0 and s32 < thr2, (scene, d2, s32)
            marker_x, _ = L.marker(rng_name)
            R = env_R(st_e, new_e, L.cx, L.cy)
            lim = {"tile0": L.tile0, "rtile": L.r_tile, "rfast": L.r_fast, "wide": L.r_fast}.get(rng_name.split("_")[0])
            if lim is not None:
                assert (R <= lim) == (rng_name.endswith("_in") or rng_name == "wide"), (scene, R, lim)
            if rng_name.startswith("rmax"):
                far = max(np.abs(np.concatenate([new_e["ux"] - L.cx, new_e["uy"] - L.cy, new_e["tx"] - L.cx,
                                                 new_e["ty"] - L.cy]))) > 32768.0
                assert far == (rng_name == "rmax_out")
            one = {k: np.ascontiguousarray(v.copy()) for k, v in st_e.items()}
            ref = oracle.step(P, 1, 0.3, None, one, np.zeros(n, np.int32), masks=True)
            for k in ("ux", "uy", "tx", "ty"):   # the moves land where the construction put them
                idx = [q for q in range(len(one[k])) if not (k[0] == "u" and q in noncard)]
                assert np.array_equal(one[k][idx], new_e[k][idx]), (scene, k)
            for kind, i, j, S in probes:
                sides.setdefault((kind, rng_name), set()).add(int(ref[MASK_OF[kind]][i, j]))
        for key, s in sides.items():
            if key[0] in ON_KINDS:
                assert s == {0, 1}, (n, m, key, s)
        for kind in ADV_KINDS:   # adversarial targets: a hit and a miss in every range
            assert all(sides.get((kind, r)) == {1 if kind == "T_ah" else 0} for r in RANGES), kind
        kinds_seen = {k for k, _ in sides}
        assert kinds_seen >= set(ON_KINDS) | set(ADV_KINDS), (n, m, kinds_seen)


# ---------------------------------------------------------------------------------------------------- GPU against the oracle
def _make_env(sc, path, E, masks, seed):
    from marl_uavs_targets_tracking_b200 import BatchedEnvironment
    env = BatchedEnvironment(sc.n, sc.m, 2000, 2000, 12, n_envs=E, device="cuda:0", seed=seed,
                             record_masks=masks, track_counts=masks)
    env.set_step_path(path)
    return env


def _check_step(oracle, sc, cfg, method, env, scenes, envs, st, actions, masks, tag):
    """One step on the GPU against the oracle, environment by environment; returns the oracle's outcome per
    (kind, range)."""
    obs, rew4, cov = env.step_device(cfg, None, None if actions is None else torch.as_tensor(actions, device="cuda:0"))
    if actions is None:
        actions = env.actions.cpu().numpy().copy()
    got = {k: v.cpu().numpy() for k, v in env.get_state().items()}
    obs, rew4, cov = obs.double().cpu().numpy(), rew4.double().cpu().numpy(), cov.cpu().numpy()
    gm = {k: env.masks[k].cpu().numpy() for k in MASKS} if masks else None
    trk = env.tracker_counts.cpu().numpy() if masks else None
    P = oracle_params_from_config(cfg, sc.n, sc.m)
    omode = {"MAAC": 0, "MAAC-G": 1}[method]
    sides = {}
    for e, (scene, (st_e, new_e, probes, noncard)) in enumerate(zip(scenes, envs)):
        one = {k: np.ascontiguousarray(v[e].copy()) for k, v in st.items()}
        ref = oracle.step(P, omode, float(cfg["cooperative"]), None, one, actions[e], masks=True)
        where = (tag, e, scene)
        # the precondition: every position that enters an exact decision is the same double on both sides
        for k in ("ux", "uy", "tx", "ty"):
            exact = [q for q in range(one[k].size) if not (k[0] == "u" and q in noncard)]
            assert np.array_equal(got[k][e][exact], one[k][exact]), (where, k)
            assert max_scaled_err(got[k][e], one[k]) <= 1e-9, (where, k)
        assert np.array_equal(got["ua"][e], one["ua"]), where
        assert int(cov[e]) == ref["covered"], (where, int(cov[e]), ref["covered"])
        if masks:
            for k in MASKS:
                assert np.array_equal(gm[k][e], ref[k]), (where, k, np.argwhere(gm[k][e] != ref[k])[:4])
            assert np.array_equal(trk[e], ref["tracker_cnt"]), where
        assert max_scaled_err(obs[e], ref["obs"]) <= TOL_TIGHT, where
        r4 = np.stack([ref["rewards"], ref["tt"], ref["bp"], ref["dup"]])
        assert max_scaled_err(rew4[:, e], r4) <= TOL_TIGHT, where
        for kind, i, j, S in probes:
            sides.setdefault((kind, scene[0]), set()).add(int(ref[MASK_OF[kind]][i, j]))
    return sides


def _cases():
    out = []
    for path, n, m in KERNELS:
        for name in sorted(CONSTS):
            for masks, method in ((True, "MAAC-G"), (False, "MAAC-G"), (False, "MAAC")):
                out.append(pytest.param(path, n, m, name, masks, method,
                                        id="p%d-%dx%d-%s-%s-%s" % (path, n, m, name, "masks" if masks else "plain", method)))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("path,n,m,name,masks,method", _cases())
def test_pair_decisions_match_the_oracle(oracle, path, n, m, name, masks, method):
    """Masks, coverage and per-target counts bit-equal to the oracle, observations and rewards within 2e-6, on every
    placement of the module docstring; the oracle's outcomes for every (probe kind, range) fall on both sides.  With
    masks and counts off (the plain instance) the decisions reach the outputs through `covered`, the observation blocks
    and the reward planes."""
    sc = Scenario(name, n, m)
    cfg = sc.config(method)
    scenes, envs, st = build_batch(sc, group=small_group(n, m) if path == 4 else 1, seed=path * 7 + n)
    E = len(scenes)
    env = _make_env(sc, path, E, masks, seed=3)
    env.reset(cfg)
    env.set_state(cfg, *(st[k] for k in ("ux", "uy", "uh", "ua", "tx", "ty", "th")))
    rs = np.random.default_rng(n * 1000 + m)
    actions = rs.integers(0, 12, (E, n)).astype(np.int32)
    sides = _check_step(oracle, sc, cfg, method, env, scenes, envs, st, actions, masks, "step")
    for key, s in sides.items():
        if key[0] in ON_KINDS:
            assert s == {0, 1}, (key, s)
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("path", [4, 0])
def test_random_policy_step_on_the_thresholds(oracle, path):
    """One step of the random-policy loop below the FFI (the small-swarm kernel draws the actions itself): the drawn
    actions, read back, drive the oracle, which must agree on every placement."""
    sc = Scenario("shipped", 10, 10)
    cfg = sc.config("MAAC-G")
    scenes, envs, st = build_batch(sc, group=small_group(10, 10), seed=5)
    env = _make_env(sc, path, len(scenes), True, seed=3)
    env.reset(cfg)
    env.set_state(cfg, *(st[k] for k in ("ux", "uy", "uh", "ua", "tx", "ty", "th")))
    before = env.actions.clone()
    obs, rew4, cov = env.run_random_policy(cfg, None, 99, 0, 1)
    assert not torch.equal(before, env.actions)
    # the step has been taken: replay it in the oracle with the drawn actions and compare every output
    actions = env.actions.cpu().numpy().copy()
    got_obs, got_rew, got_cov = obs.double().cpu().numpy(), rew4.double().cpu().numpy(), cov.cpu().numpy()
    got = {k: v.cpu().numpy() for k, v in env.get_state().items()}
    P = oracle_params_from_config(cfg, 10, 10)
    for e, (scene, (st_e, new_e, probes, noncard)) in enumerate(zip(scenes, envs)):
        one = {k: np.ascontiguousarray(v[e].copy()) for k, v in st.items()}
        ref = oracle.step(P, 1, float(cfg["cooperative"]), None, one, actions[e], masks=True)
        for k in ("ux", "uy", "tx", "ty"):
            exact = [q for q in range(one[k].size) if not (k[0] == "u" and q in noncard)]
            assert np.array_equal(got[k][e][exact], one[k][exact]), (e, k)
        assert int(got_cov[e]) == ref["covered"], (e, scene)
        for k in MASKS:
            assert np.array_equal(env.masks[k][e].cpu().numpy(), ref[k]), (e, scene, k)
        assert np.array_equal(env.tracker_counts[e].cpu().numpy(), ref["tracker_cnt"]), (e, scene)
        assert max_scaled_err(got_obs[e], ref["obs"]) <= TOL_TIGHT
        r4 = np.stack([ref["rewards"], ref["tt"], ref["bp"], ref["dup"]])
        assert max_scaled_err(got_rew[:, e], r4) <= TOL_TIGHT
    env.close()
