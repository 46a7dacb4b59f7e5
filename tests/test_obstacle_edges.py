"""The obstacle path at its decision boundaries, one crafted env per case, one step from an injected state, against the
CPU oracle stepped from the same state.

The pipeline layout decides visibility and collision in float, on float obstacle records relative to the goal, with
explicit slack (cull_pair_rec); pairs within 2 mm of the collision threshold are re-decided in double; the in-view
envs go to work lists by the number of obstacles in view.  Random rollouts almost never put a surface within a few mm of
a field-of-view plane, the range limit or the collision threshold, so every case here is built to sit there:

  A  range limit: a ray through a sphere centre / capsule axis hits at max_dist - delta (centre and corner ray)
  B  field-of-view edge: a close obstacle whose surface crosses the plane of an outermost ray column / row by delta at a
     ray of that column / row (spheres; capsules parallel, oblique and perpendicular to the plane); the x = 0 plane
  C  capsule axis clipping: 40 m pillars seen from near one end, vertical pillars at zero roll and pitch (alpha == 0),
     an axis tilted by a subnormal angle (the ftz branch), foot points at bot / top
  D  collision band: centre / axis distance = radius + safety_radius + delta (sphere, capsule side, end cap, foot point
     at bot / top, vehicle inside an obstacle)
  E  work lists: 8 capsules + 8 spheres with exactly k in view (k = 0..16), every slot alone, two-obstacle type mixes
  F  float record counts: (capsules, spheres) = (8, 4), (8, 5), (0, 1), (1, 0)
  G  1985 m from the goal: max_dist_from_goal + max_dist = 2000 (float records) and 2000.5 (exact culls)
  H  non-finite pose (NaN / inf in position or velocity) with obstacles in view

Placement is two-pass: the oracle steps the pre-step state once, the obstacles are placed around its post-step pose
(geometry is decided there; obstacles do not feed back into the dynamics), then both sides step from the pre-step state.

w_oa is raised from 0.2 to 2000: a ray of the outermost column carries beta_oa weight 0.01, so with the stock factor a
hit 1e-4 m inside the range limit moves the reward by ~3e-10 and no bar could see a wrongly culled obstacle; at 2000 every
inside case of A-D moves it by more than 1e-7 relative (test_cases_discriminate checks that on the oracle alone).  For
the same reason the max-timestep done (reward -100) is injected only into cases whose edge is a collision or a list.
"""
import copy

import numpy as np
import pytest

from oracle import oracle as orc
from tests.golden_utils import rel_err

W_OA = 2000.0
WINDOW = 1e-9             # |delta| up to this: the reference formulas and the kernels may round either way
TIGHT = 0.05              # obstacles at least this far outside the view and range must not be listed
DELTAS_EDGE = (2.5e-3, -2.5e-3, 1e-3, -1e-3, 1e-4, -1e-4, 3e-5, -3e-5)
DELTAS_BAND = (0.0, 1e-9, -1e-9, 1e-6, -1e-6, 1e-4, -1e-4, 1.9e-3, -1.9e-3, 2e-3, -2e-3, 2.1e-3, -2.1e-3, 1e-2, -1e-2)
DEG = np.pi / 180
POSES = [(0.0, 0.0, 0.3), (55 * DEG, 0.0, 1.2), (-55 * DEG, 20 * DEG, -2.0), (10 * DEG, 55 * DEG, 3.1),
         (-15 * DEG, -55 * DEG, -3.1), (30 * DEG, -30 * DEG, np.pi - 1e-3)]
# name: (n_capsules, n_spheres, max_dist_from_goal)
GROUPS = {"c4": (5, 3, 20.0), "e": (8, 8, 20.0), "f84": (8, 4, 20.0), "f85": (8, 5, 20.0), "f01": (0, 1, 20.0),
          "f10": (1, 0, 20.0), "g_float": (5, 3, 1990.0), "g_exact": (5, 3, 1990.5)}
LAYOUTS = ("pipeline", "warp_rays", "thread_per_env")


def _config(max_dist_from_goal):
    from gym_dockauv_b200.config import BASE_CONFIG, RADAR_64
    cfg = copy.deepcopy(BASE_CONFIG)
    cfg["radar"] = dict(RADAR_64)
    cfg["reward_factors"]["w_oa"] = W_OA
    cfg["max_dist_from_goal"] = float(max_dist_from_goal)
    return cfg


def _unit(v):
    v = np.asarray(v, dtype=float)
    return v / np.linalg.norm(v)


class _Frame:
    """Post-step pose of one case: position, rotation, world ray directions, outward normals of the fan's planes."""

    def __init__(self, P, pos, att):
        self.pos = np.array(pos, dtype=float)
        self.R = orc.rzyx(*att)
        self.u = orc.ray_directions(P, att)
        self.n_v, self.n_h, self.max_dist = P.n_vert, P.n_horiz, P.radar_max_dist
        rd = np.ctypeslib.as_array(P.rd_b)[:3 * P.n_rays].reshape(-1, 3)
        sy, sz = rd[-1, 1] / rd[-1, 0], rd[-1, 2] / rd[-1, 0]          # last ray: outermost column and row
        # plane name -> (outward body normal, rays lying in the plane)
        col = lambda ih: [iv * self.n_h + ih for iv in range(self.n_v)]  # noqa: E731
        row = lambda iv: [iv * self.n_h + ih for ih in range(self.n_h)]  # noqa: E731
        self.planes = {"y+": (_unit([-sy, 1, 0]), col(self.n_h - 1)), "y-": (_unit([-sy, -1, 0]), col(0)),
                       "z+": (_unit([-sz, 0, 1]), row(self.n_v - 1)), "z-": (_unit([-sz, 0, -1]), row(0))}

    def ray(self, iv, ih):
        return iv * self.n_h + ih

    def world(self, v_body):
        return self.R @ np.asarray(v_body, dtype=float)


class Case:
    def __init__(self, group, family, label):
        self.group, self.family, self.label = group, family, label
        self.delta = None          # signed distance from the decision boundary (> 0: inside / colliding side)
        self.ray = None            # the ray designed to hit (delta > 0) or miss (delta < 0) the edge obstacle
        self.hit_at = None         # designed hit distance along that ray (family A)
        self.collide = None        # designed collision flag (family D)
        self.edge = []             # (kind, slot) of the obstacles the case is about
        self.tight = False         # every obstacle at least TIGHT outside view and range
        self.n_in_view = None      # family E: number of obstacles placed well inside the view

    @property
    def window(self):
        return self.delta is not None and abs(self.delta) <= WINDOW


class _Scene:
    """Pre-step state + obstacle slots of one case; unused slots are parked 15+ m behind the vehicle."""

    def __init__(self, P, group, rng, pose, goal_dist=8.0, state=None, action=None, t_steps=None):
        nc, ns, _ = GROUPS[group]
        self.P, self.nc, self.ns = P, nc, ns
        if state is None:
            goal = rng.uniform(-30, 30, 3)
            pos = goal + goal_dist * _unit(rng.normal(size=3))
            nu = rng.uniform(-0.2, 0.2, 6) * np.array([1, 1, 1, 0.3, 0.3, 0.3])
            state = np.concatenate([pos, pose, nu])
        else:
            goal = state[:3] + goal_dist * _unit(rng.normal(size=3))
        self.state = np.asarray(state, dtype=float)
        self.goal = goal
        self.heading = rng.uniform(-np.pi, np.pi)
        self.u0 = rng.uniform(-0.5, 0.5, 6)
        self.action = rng.uniform(-1, 1, 6) if action is None else np.asarray(action, dtype=float)
        self.t_steps = int(rng.integers(0, 990)) if t_steps is None else t_steps
        self.ep_return = float(rng.uniform(-50, 50))
        self.caps = np.zeros((nc, 7))
        self.sph = np.zeros((ns, 4))
        E = self.oracle_env()
        orc.step(P, E, self.action)
        post = np.array(E.state[:])
        if not np.all(np.isfinite(post[:6])):
            post = self.state          # non-finite pose: place around the pre-step pose
        self.f = _Frame(P, post[:3], post[3:6])
        back = -self.f.world([1, 0, 0])
        side = self.f.world([0, 1, 0])
        for k in range(nc):
            b = self.f.pos + (15 + 2 * k) * back
            self.caps[k] = [*b, *(b + side), 0.3]
        for k in range(ns):
            self.sph[k] = [*(self.f.pos + (15 + 2 * k) * back + 3 * side), 0.3]

    def oracle_env(self, caps=None, sph=None):
        E = orc.OrcEnv()
        orc.set_env(E, self.state, self.goal, self.heading, self.caps if caps is None else caps,
                    self.sph if sph is None else sph, np.zeros(5), u=self.u0, t_steps=self.t_steps)
        E.cum_reward = self.ep_return
        return E

    def put_sphere(self, slot, centre, r):
        self.sph[slot] = [*centre, r]

    def put_capsule(self, slot, bot, top, r):
        self.caps[slot] = [*bot, *top, r]


def _pick_slot(scene, kind, rng):
    return int(rng.integers(0, scene.nc if kind == "cap" else scene.ns))


def _mk(scene, case, kind, slot):
    case.scene = scene
    case.edge.append((kind, slot))
    return case


# ----------------------------------------------------------------------------------------------------- case families
def _family_a(P, group, rng, poses, deltas, kinds=("sph", "cap")):
    """Range limit: the ray through the centre / axis hits at max_dist - delta."""
    out = []
    for pi, pose in enumerate(poses):
        for ray_name, (iv, ih) in (("centre", (4, 4)), ("corner", (7, 0))):
            for kind in kinds:
                for d in deltas:
                    sc = _Scene(P, group, rng, pose)
                    f = sc.f
                    i = f.ray(iv, ih)
                    u = f.u[i]
                    r = rng.uniform(0.3, 0.8)
                    c = f.pos + (f.max_dist - d + r) * u
                    cs = Case(group, "A", f"pose{pi}-{ray_name}-{kind}-{d:+g}")
                    cs.delta, cs.ray, cs.hit_at, cs.tight = d, i, f.max_dist - d, d <= -TIGHT
                    slot = _pick_slot(sc, kind, rng)
                    if kind == "sph":
                        sc.put_sphere(slot, c, r)
                    else:
                        w = _unit(np.cross(u, rng.normal(size=3)))     # axis perpendicular to the ray
                        a = rng.uniform(0.2, 1.5)
                        sc.put_capsule(slot, c - a * w, c + (2.0 - a) * w, r)
                    out.append(_mk(sc, cs, kind, slot))
    return out


def _plane_obstacle(sc, slot, kind, plane, i_ray, D, r, d, shape, rng, L=1.0, a=0.5):
    """An obstacle whose surface crosses `plane` by d at the point of ray i_ray at distance D (d < 0: outside)."""
    f = sc.f
    n = f.world(f.planes[plane][0])
    u = f.u[i_ray]
    F = f.pos + D * u + (r - d) * n          # the centre / axis point nearest to the plane, r - d outside it
    m = _unit(np.cross(n, u))                 # in the plane, perpendicular to the ray
    if kind == "sph":
        sc.put_sphere(slot, F, r)
    elif shape == "parallel":                 # axis in a plane parallel to the fan plane, not parallel to the ray
        phi = rng.uniform(-0.6, 0.6)
        w = np.cos(phi) * m + np.sin(phi) * u
        sc.put_capsule(slot, F - a * w, F + (L - a) * w, r)
    else:                                     # the end cap at F is the nearest part; the axis leaves the plane
        beta = {"perpendicular": 0.0, "oblique": 45 * DEG, "oblique70": 70 * DEG}[shape]
        w = np.cos(beta) * n + np.sin(beta) * m
        sc.put_capsule(slot, F, F + L * w, r)


def _family_b(P, group, rng, poses, deltas):
    out = []
    shapes = [("sph", None), ("cap", "parallel"), ("cap", "oblique"), ("cap", "oblique70"), ("cap", "perpendicular")]
    for pi, pose in enumerate(poses):
        for plane, (iv, ih) in (("y+", (3, 7)), ("y-", (4, 0)), ("z+", (7, 2)), ("z-", (0, 5))):
            for kind, shape in shapes:
                for d in deltas:
                    sc = _Scene(P, group, rng, pose)
                    i = sc.f.ray(iv, ih)
                    assert i in sc.f.planes[plane][1]
                    slot = _pick_slot(sc, kind, rng)
                    _plane_obstacle(sc, slot, kind, plane, i, rng.uniform(1.5, 5.0), rng.uniform(0.2, 0.6), d, shape, rng)
                    cs = Case(group, "B", f"pose{pi}-{plane}-{kind}-{shape}-{d:+g}")
                    cs.delta, cs.ray, cs.tight = d, i, d <= -TIGHT
                    out.append(_mk(sc, cs, kind, slot))
        # the x = 0 plane: no ray of a +-35 deg fan passes near it, so these cases pin the collision decision and (when
        # the obstacle is 5 cm or more behind) the tightness of the cull -- a sphere directly behind the vehicle
        # collides with it but must not be listed
        for where in ("behind", "beside"):
            for d in (-TIGHT, -0.2):
                sc = _Scene(P, group, rng, pose)
                r = 0.5
                cb = [-(r - d), 0.0, 0.0] if where == "behind" else [-(r - d), r, 0.0]
                slot = _pick_slot(sc, "sph", rng)
                sc.put_sphere(slot, sc.f.pos + sc.f.world(cb), r)
                cs = Case(group, "B", f"pose{pi}-x0-{where}-{d:+g}")
                cs.delta, cs.tight = d, where == "behind"
                out.append(_mk(sc, cs, "sph", slot))
    return out


def _family_c(P, group, rng):
    out = []
    # 40 m pillars seen from near one end, under roll and pitch: the axis runs in a plane parallel to a fan plane,
    # the nearest axis point (foot of the designed ray) at 0, 1 m or L from bot
    for pi, pose in enumerate(POSES[1:5]):
        for plane, (iv, ih) in (("y+", (4, 7)), ("z-", (0, 3))):
            for a in (0.0, 1.0, 40.0):
                for d in (1e-3, -1e-3, 1e-4, -1e-4, -TIGHT):
                    sc = _Scene(P, group, rng, pose)
                    i = sc.f.ray(iv, ih)
                    slot = _pick_slot(sc, "cap", rng)
                    _plane_obstacle(sc, slot, "cap", plane, i, rng.uniform(1.0, 4.0), 0.5, d, "parallel", rng, L=40.0, a=a)
                    cs = Case(group, "C", f"pillar-pose{pi}-{plane}-a{a:g}-{d:+g}")
                    cs.delta, cs.ray, cs.tight = d, i, d <= -TIGHT and a == 1.0
                    out.append(_mk(sc, cs, "cap", slot))
    # vertical pillars at zero roll and pitch: the body-frame axis has db[0] == 0 exactly (the alpha == 0 branch of
    # the clip), and tilted by a subnormal angle: alpha flushes to zero in rcp.approx.ftz
    for yaw in (0.0, 0.7, -2.5, np.pi - 1e-3):
        for tilt in (0.0, 1e-40):
            for d in (1e-3, -1e-3, 1e-4, -1e-4, 3e-5, -3e-5, -TIGHT):
                state = np.zeros(12)
                state[5] = yaw
                sc = _Scene(P, group, rng, None, state=np.concatenate([rng.uniform(-20, 20, 3), state[3:]]),
                            action=np.zeros(6))
                sc.u0[:] = 0.0
                # re-run the placement with the zeroed command: the pose must stay exactly level
                E = sc.oracle_env()
                orc.step(P, E, sc.action)
                post = np.array(E.state[:])
                sc.f = _Frame(P, post[:3], post[3:6])
                i = sc.f.ray(3, 7)
                D, r = rng.uniform(1.5, 4.0), 0.5
                n = sc.f.world(sc.f.planes["y+"][0])
                F = sc.f.pos + D * sc.f.u[i] + (r - d) * n
                if tilt:
                    # the axis is x = 0 in world coordinates so that a 1e-40 relative offset survives in double: shift
                    # the whole scene along x by -F[0]
                    shift = np.array([F[0], 0.0, 0.0])
                    sc.state[:3] -= shift
                    sc.goal = sc.goal - shift
                    F = F - shift
                    F[0] = 0.0
                    sc.f.pos = sc.f.pos - shift
                    for k in range(sc.nc):
                        sc.caps[k, [0, 3]] -= shift[0]
                    for k in range(sc.ns):
                        sc.sph[k, 0] -= shift[0]
                bot = F - np.array([0, 0, 20.0])
                top = F + np.array([0, 0, 20.0])
                if tilt:
                    top[0] = tilt * 40.0           # F[0] == 0
                slot = _pick_slot(sc, "cap", rng)
                sc.put_capsule(slot, bot, top, r)
                cs = Case(group, "C", f"vertical-yaw{yaw:.2f}-tilt{tilt:g}-{d:+g}")
                cs.delta, cs.ray, cs.tight = d, i, d <= -TIGHT
                cs.level = True
                out.append(_mk(sc, cs, "cap", slot))
    return out


def _family_d(P, group, rng, poses, deltas, kinds=("sph", "cap")):
    out = []
    shapes = [s for s in ("sph", "cap_side", "cap_end", "cap_foot_bot", "cap_foot_top") if s[:3] in kinds]
    for pi, pose in enumerate(poses):
        for shape in shapes:
            for d in deltas:
                sc = _Scene(P, group, rng, pose)
                f = sc.f
                u = f.u[f.ray(4, 3)]
                r = rng.uniform(0.3, 0.8)
                thr = r + P.safety_radius
                m = _unit(np.cross(u, rng.normal(size=3)))
                kind = "sph" if shape == "sph" else "cap"
                slot = _pick_slot(sc, kind, rng)
                c = f.pos + (thr + d) * u
                if shape == "sph":
                    sc.put_sphere(slot, c, r)
                elif shape == "cap_side":
                    sc.put_capsule(slot, c - 0.7 * m, c + 0.9 * m, r)
                elif shape == "cap_foot_bot":
                    sc.put_capsule(slot, c, c + 1.2 * m, r)
                elif shape == "cap_foot_top":
                    sc.put_capsule(slot, c - 1.2 * m, c, r)
                else:                               # end cap: the axis leaves the vehicle at an angle to every ray
                    w = _unit(u + 0.3 * m)
                    b = f.pos + (thr + d) * w
                    sc.put_capsule(slot, b, b + 1.5 * w, r)
                cs = Case(group, "D", f"pose{pi}-{shape}-{d:+g}")
                cs.delta, cs.collide = d, d < 0
                out.append(_mk(sc, cs, kind, slot))
        for kind in kinds:                          # the vehicle inside an obstacle
            sc = _Scene(P, group, rng, pose)
            u = sc.f.u[sc.f.ray(4, 4)]
            slot = _pick_slot(sc, kind, rng)
            c = sc.f.pos + 0.3 * u
            if kind == "sph":
                sc.put_sphere(slot, c, 2.0)
            else:
                m = _unit(np.cross(u, rng.normal(size=3)))
                sc.put_capsule(slot, c - m, c + 2 * m, 1.5)
            cs = Case(group, "D", f"pose{pi}-inside-{kind}")
            cs.collide = True
            out.append(_mk(sc, cs, kind, slot))
    return out


def _family_e(P, rng):
    """8 capsules + 8 spheres: exactly k in view (k = 0..16), every slot alone, two-obstacle type mixes."""
    group = "e"
    sets = [list(rng.permutation(16)[:k]) for k in range(17)]
    sets += [[s] for s in range(16)]
    sets += [[0, 7], [2, 5], [3, 10], [7, 15], [8, 15], [9, 12], [6, 13, 14], [1, 8, 11]]
    out = []
    for j, slots in enumerate(sets):
        sc = _Scene(P, group, rng, POSES[j % len(POSES)])
        f = sc.f
        rays = rng.permutation(P.n_rays)[:len(slots)]
        for s, i in zip(slots, rays):
            u = f.u[i]
            c = f.pos + rng.uniform(3.0, 8.0) * u
            if s < 8:
                w = _unit(np.cross(u, rng.normal(size=3)))
                sc.put_capsule(s, c - 0.3 * w, c + 0.3 * w, 0.2)
            else:
                sc.put_sphere(s - 8, c, 0.25)
        cs = Case(group, "E", f"slots{'-'.join(map(str, slots)) or 'none'}")
        cs.n_in_view = len(slots)
        cs.scene = sc
        cs.edge = [("cap", s) if s < 8 else ("sph", s - 8) for s in slots]
        out.append(cs)
    return out


def _family_f(P, group, rng):
    """Edge cases in the last slot of each obstacle type (the last float record of the env)."""
    nc, ns, _ = GROUPS[group]
    out = []
    kinds = [k for k, n in (("cap", nc), ("sph", ns)) if n > 0]
    for kind in kinds:
        last = (nc if kind == "cap" else ns) - 1
        for c in _family_a(P, group, rng, POSES[:2], (1e-4, -1e-4), kinds=(kind,)) + \
                _family_d(P, group, rng, POSES[2:3], (1e-4, -1e-4, 1e-9), kinds=(kind,)):
            if c.edge[0][0] != kind:
                continue
            _move_edge(c, last)
            c.family = "F"
            out.append(c)
        for d in (1e-3, -1e-3):
            sc = _Scene(P, group, rng, POSES[3])
            i = sc.f.ray(3, 7)
            _plane_obstacle(sc, last, kind, "y+", i, 2.5, 0.4, d, "oblique", rng)
            cs = Case(group, "F", f"{kind}-plane-{d:+g}")
            cs.delta, cs.ray = d, i
            out.append(_mk(sc, cs, kind, last))
    return out


def _move_edge(case, slot):
    kind, old = case.edge[0]
    sc = case.scene
    arr = sc.caps if kind == "cap" else sc.sph
    arr[[old, slot]] = arr[[slot, old]]
    case.edge = [(kind, slot)]


def _family_g(P, group, rng):
    """1985 m from the goal, families A, B and D around the vehicle."""
    out = []
    for fam in (_family_a(P, group, rng, POSES[:2], (1e-3, -1e-3, 1e-4, -1e-4, -TIGHT)),
                _family_b(P, group, rng, POSES[2:3], (1e-3, -1e-3, 1e-4, -1e-4, -TIGHT)),
                _family_d(P, group, rng, POSES[3:4], (1e-6, -1e-6, 1e-4, -1e-4, 2.1e-3, -2.1e-3, 0.0))):
        for c in fam:
            c.family = "G" + c.family
            out.append(c)
    return out


def _family_h(P, group, rng):
    out = []
    for idx, val in ((0, np.nan), (2, np.inf), (6, np.nan), (8, np.inf), (10, -np.inf), (7, -np.inf)):
        sc = _Scene(P, group, rng, POSES[1])
        f = sc.f
        cs = Case(group, "H", f"state{idx}={val}")
        if sc.ns:
            sc.put_sphere(0, f.pos + 3.0 * f.u[f.ray(4, 4)], 0.5)
            cs.edge.append(("sph", 0))
        if sc.nc:
            w = _unit(np.cross(f.u[f.ray(2, 5)], [0, 0, 1]))
            c = f.pos + 4.0 * f.u[f.ray(2, 5)]
            sc.put_capsule(0, c - w, c + w, 0.4)
            cs.edge.append(("cap", 0))
        sc.state[idx] = val
        cs.scene = sc
        out.append(cs)
    return out


def _padding_scene(P, group):
    """The env the large batches are padded with: nothing in view, episode not ending."""
    return _Scene(P, group, np.random.default_rng(99), POSES[0], t_steps=5)


_CACHE = {}


def build_cases(group):
    """All cases of a group, each with its oracle result (deterministic)."""
    if group in _CACHE:
        return _CACHE[group]
    nc, ns, mdg = GROUPS[group]
    P = orc.make_params(_config(mdg))
    rng = np.random.default_rng(list(GROUPS).index(group) + 1)
    if group == "c4":
        cases = (_family_a(P, group, rng, POSES, DELTAS_EDGE + (-TIGHT,)) + _family_b(P, group, rng, POSES, DELTAS_EDGE + (-TIGHT,))
                 + _family_c(P, group, rng) + _family_d(P, group, rng, POSES[:3], DELTAS_BAND) + _family_h(P, group, rng))
    elif group == "e":
        cases = _family_e(P, rng)
    elif group.startswith("f"):
        # with and without capsules the reference treats a non-finite pose differently (see radar_env)
        cases = _family_f(P, group, rng) + _family_h(P, group, rng)
    else:
        # vehicles 1985 m from the goal (the goal 1985 m away from a vehicle near the origin of a far-off patch)
        cases = []
        for c in _family_g(P, group, rng):
            cases.append(c)
        for c in cases:
            sc = c.scene
            off = sc.goal - sc.state[:3]
            shift = 1985.0 * _unit(off) - off           # move the goal, keep the vehicle and its obstacles
            sc.goal = sc.goal + shift
    for k, c in enumerate(cases):
        if k % 9 == 4 and c.family in ("D", "E", "GD"):
            c.scene.t_steps = 1000                       # the max-timestep done on top of whatever else happens
    for c in cases:
        E = c.scene.oracle_env()
        c.out = orc.step(P, E, c.scene.action)
        c.post_state = np.array(E.state[:])
        c.cum_reward = E.cum_reward
        c.t_after = E.t_steps
    pad = _padding_scene(P, group)
    E = pad.oracle_env()
    pad.out = orc.step(P, E, pad.action)
    pad.post_state = np.array(E.state[:])
    _CACHE[group] = (P, cases, pad)
    return _CACHE[group]


def _reward_without_edge(P, case):
    """Oracle reward of the case with its edge obstacles moved to the parking places."""
    sc = case.scene
    caps, sph = sc.caps.copy(), sc.sph.copy()
    back = -sc.f.world([1, 0, 0])
    side = sc.f.world([0, 1, 0])
    for kind, slot in case.edge:
        b = sc.f.pos + 40 * back + slot * side
        if kind == "cap":
            caps[slot] = [*b, *(b + side), 0.3]
        else:
            sph[slot] = [*(b + 2 * side), 0.3]
    E = sc.oracle_env(caps, sph)
    return orc.step(P, E, sc.action).reward


# ------------------------------------------------------------------------------------ CPU: the generator is right
@pytest.mark.parametrize("group", list(GROUPS))
def test_cases_discriminate(group):
    """On the oracle alone: every designed ray hits inside cases below max_dist and misses outside ones; the collision
    flag follows the sign of delta; an inside case of A-D loses at least 1e-7 relative of its reward when its edge
    obstacle is removed (100x the 1e-9 bar), so a wrongly culled obstacle cannot pass; level poses stay exactly level;
    tight cases see nothing at all."""
    P, cases, pad = build_cases(group)
    assert np.all(np.array(pad.out.ray_dist[:P.n_rays]) == P.radar_max_dist) and not pad.out.done
    n_checked = 0
    for c in cases:
        o = c.out
        rd = np.array(o.ray_dist[:P.n_rays])
        if c.collide is not None and c.delta != 0.0:
            assert bool(o.collision) == c.collide, (c.label, c.delta)
        if c.window or c.family == "H":
            continue
        if c.ray is not None:
            inside = c.delta > 0
            if inside:
                assert rd[c.ray] < P.radar_max_dist, c.label
            else:
                assert rd[c.ray] == P.radar_max_dist, c.label
            if c.hit_at is not None and inside:
                assert abs(rd[c.ray] - c.hit_at) < 1e-9, (c.label, rd[c.ray], c.hit_at)
        if c.tight:
            assert np.all(rd == P.radar_max_dist), c.label
        if getattr(c, "level", False):
            assert c.post_state[3] == 0.0 and c.post_state[4] == 0.0, c.label
        if c.family.lstrip("G") in "ABCDF" and (c.collide or (c.delta is not None and c.delta > 0)):
            r0 = _reward_without_edge(P, c)
            assert abs(o.reward - r0) >= 1e-7 * max(abs(o.reward), 1e-3), (c.label, o.reward, r0)
            n_checked += 1
        if c.family == "E":
            assert (np.sum(rd < P.radar_max_dist) > 0) == (c.n_in_view > 0), c.label
    if group not in ("e",):
        assert n_checked > 0
    sub = [c for c in cases if "tilt1e-40" in c.label]
    for c in sub:
        kind, slot = c.edge[0]
        b = c.scene.caps[slot]
        d0 = (b[3] - b[0]) / np.linalg.norm(b[3:6] - b[:3])
        assert 0 < abs(np.float32(d0)) < np.finfo(np.float32).tiny, (c.label, d0)


# ------------------------------------------------------------------------------------------------ GPU runs
def _make_env(group, n, layout, auto_reset, debug):
    from gym_dockauv_b200 import envs
    nc, ns, mdg = GROUPS[group]
    return envs.ObstaclesDocking3d(_config(mdg), num_envs=n, seed=3, layout=layout, n_capsules=nc, n_spheres=ns,
                                   auto_reset=auto_reset, debug_outputs=debug)


def _inject(env, scenes):
    n = len(scenes)
    nc, ns = env.n_capsules, env.n_spheres
    env.set_state(state=np.stack([s.state for s in scenes]), u_prev=np.stack([s.u0 for s in scenes]),
                  goal=np.stack([s.goal for s in scenes]), heading_goal=np.array([s.heading for s in scenes]),
                  current=np.zeros((n, 5)), capsules=np.stack([s.caps for s in scenes]).reshape(n, nc * 7) if nc else None,
                  spheres=np.stack([s.sph for s in scenes]).reshape(n, ns * 4) if ns else None,
                  t_steps=np.array([s.t_steps for s in scenes]), ep_return=np.array([s.ep_return for s in scenes]))


def _step(env, scenes):
    import torch
    _inject(env, scenes)
    a = torch.as_tensor(np.stack([s.action for s in scenes]), device=env.device)
    obs, reward, done, info = env.step(a)
    return dict(obs=obs.cpu().numpy(), reward=reward.cpu().numpy(), done=done.cpu().numpy(),
                cond=info["cond_bits"].cpu().numpy(), state=env.state.t().cpu().numpy(),
                term=info["terminal_observation"].cpu().numpy(), ep_ret=info["episode_return"].cpu().numpy(),
                ep_len=info["episode_length"].cpu().numpy(), delta_d=info["delta_d"].cpu().numpy(),
                ray=None if env.debug is None else env.debug["ray_dist"].t().cpu().numpy())


def _cond_bits(o):
    return sum(int(o.cond[k]) << k for k in range(5))


def _ulp_ok(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    same = (a == b) | (np.isnan(a) & np.isnan(b))
    close = np.abs(a.astype(np.float64) - b) <= np.spacing(np.maximum(np.abs(a), np.abs(b)))
    return same | close


def _check_vs_oracle(P, cases, res, rows, where):
    """Every case outside the ambiguity window against its oracle step; returns the cases inside the window."""
    n_obs = P.n_obs
    inside = []
    for c, i in zip(cases, rows):
        o = c.out
        tag = (where, c.group, c.family, c.label)
        if c.window:
            inside.append(c)
            continue
        assert int(res["done"][i]) == int(o.done), tag
        assert int(res["cond"][i]) == _cond_bits(o), tag
        assert rel_err(res["reward"][i], o.reward) < 1e-9, (tag, res["reward"][i], o.reward)
        if res.get("auto_reset") and o.done:      # re-initialised: the state is the next episode's
            assert not res["obs"][i].any(), tag
            assert _ulp_ok(res["term"][i], np.array(o.obs[:n_obs])).all(), tag
            assert rel_err(res["ep_ret"][i], c.cum_reward) < 1e-9, tag
            assert res["ep_len"][i] == c.t_after, tag
        else:
            assert rel_err(res["state"][i], c.post_state) < 1e-9, tag
            assert _ulp_ok(res["obs"][i], np.array(o.obs[:n_obs])).all(), (tag, res["obs"][i], np.array(o.obs[:n_obs]))
        if res.get("ray") is not None:
            assert rel_err(res["ray"][i], np.array(o.ray_dist[:P.n_rays])) < 1e-9, tag
    return inside


@pytest.mark.gpu
@pytest.mark.parametrize("group", list(GROUPS))
def test_families_through_every_layout(group):
    """Each case as one env, auto_reset off, through the pipeline and both single-launch layouts (those with per-ray
    debug outputs): against the oracle outside the ambiguity window; inside it the pipeline and warp_rays, which both
    decide in double, agree bitwise on the flags."""
    P, cases, _ = build_cases(group)
    scenes = [c.scene for c in cases]
    rows = range(len(cases))
    res = {}
    for layout in LAYOUTS:
        env = _make_env(group, len(cases), layout, auto_reset=False, debug=layout != "pipeline")
        res[layout] = _step(env, scenes)
        if layout == "pipeline":
            n_listed = env.last_list_counts()[0]
        env.close()
        inside = _check_vs_oracle(P, cases, res[layout], rows, layout)
    win = [cases.index(c) for c in inside]
    for k in ("done", "cond"):
        assert np.array_equal(res["pipeline"][k][win], res["warp_rays"][k][win]), group
    fams = sorted({c.family for c in cases})
    print(f"\n[{group}] {len(cases)} cases, listed by the pipeline cull: {n_listed}; inside the ambiguity window: " +
          ", ".join(f"{f} {sum(c.family == f for c in inside)}" for f in fams))
    if group == "e":
        # every obstacle placed in view is well inside it, every parked one far outside: the listed count is exact
        assert n_listed == sum(c.n_in_view > 0 for c in cases)


@pytest.mark.gpu
@pytest.mark.parametrize("group", ["c4", "g_float", "g_exact"])
def test_cull_is_tight(group):
    """Cases whose obstacles all sit at least 5 cm outside the view or range: no env may be listed for the ray launch
    (a cull that kept everything would pass every other assertion)."""
    P, cases, _ = build_cases(group)
    tight = [c for c in cases if c.tight]
    assert tight
    env = _make_env(group, len(tight), "pipeline", auto_reset=False, debug=False)
    _step(env, [c.scene for c in tight])
    assert env.last_list_counts()[0] == 0, [getattr(c, "label", "pad") for c in tight]
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("auto_reset", [False, True])
def test_all_cases_in_one_large_batch(auto_reset):
    """Each group's cases shuffled into 2^17 + 4,099 envs (stepped in two parts on two streams), padded with envs that
    have nothing in view, pipeline only.  With auto-reset: terminal observation, episode return and length of the done
    envs against the oracle, and the statistics deltas against sums over the oracle."""
    N = (1 << 17) + 4099
    for group in GROUPS:
        P, cases, pad = build_cases(group)
        rng = np.random.default_rng(7)
        rows = rng.choice(N, size=len(cases), replace=False)
        scenes = [pad] * N
        for c, i in zip(cases, rows):
            scenes[i] = c.scene
        env = _make_env(group, N, "pipeline", auto_reset=auto_reset, debug=False)
        s0 = env.get_stats()
        res = _step(env, scenes)
        res["auto_reset"] = auto_reset
        _check_vs_oracle(P, cases, res, rows, f"batch auto_reset={auto_reset}")
        padm = np.ones(N, bool)
        padm[rows] = False
        assert not res["done"][padm].any()
        assert rel_err(res["reward"][padm], pad.out.reward) < 1e-9 and rel_err(res["state"][padm], pad.post_state) < 1e-9
        assert _ulp_ok(res["obs"][padm], np.array(pad.out.obs[:P.n_obs])).all()
        if auto_reset:
            s1 = env.get_stats()
            d = {k: s1[k] - s0[k] for k in s1}
            # per ended episode: (condition bits, length, return, final delta_d, NaN reward) -- from the oracle, except
            # inside the ambiguity window, where the flags are the kernel's own (checked against warp_rays above)
            ends = [(_cond_bits(c.out), c.t_after, c.cum_reward, c.out.delta_d, np.isnan(c.out.reward))
                    for c in cases if not c.window and c.out.done]
            ends += [(int(res["cond"][i]), int(res["ep_len"][i]), float(res["ep_ret"][i]), float(res["delta_d"][i]),
                      np.isnan(res["reward"][i])) for c, i in zip(cases, rows) if c.window and res["done"][i]]
            assert d["episodes"] == len(ends) and d["env_steps"] == N, group
            for k, name in enumerate(("done_goal_reached", "done_out_pos", "done_out_att", "done_max_t", "done_collision")):
                assert d[name] == sum(e[0] >> k & 1 for e in ends), (group, name)
            assert d["sum_length"] == sum(e[1] for e in ends), group
            assert d["nan_envs"] == sum(e[4] for e in ends), group
            assert rel_err(d["sum_return"], sum(e[2] for e in ends)) < 1e-9, group
            assert rel_err(d["sum_final_delta_d"], sum(e[3] for e in ends)) < 1e-9, group
        env.close()
