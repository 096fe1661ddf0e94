"""Pin the CPU oracle ("port") to the reference.

Three anchors, all CPU-only:
  1. the reference's OWN known-answer vectors, re-expressed from test/src/test_raycast_dda.cpp,
     test_chunked_kdtree.cpp, test_quat.cpp, test_pf.cpp (cited per test);
  2. tests/golden/*.npz — outputs of the reference's own sources (oracle/_ref), committed with the
     generating script tests/golden/make_golden.py;
  3. port == reference bit-for-bit on seeded random scenes, against the reference build's answers recorded in
     tests/golden/reference_calls.npz (the `reference` fixture, tests/recorded_reference.py).
"""
import math

import numpy as np
import pytest

from conftest import golden
from oracle import cpu_checker as cc
from mcl_3dl_b200 import synth


def frange(a, b, step):
    """`for (float v = a; v < b; v += step)` with float32 accumulation, as the reference tests loop."""
    v = np.float32(a)
    out = []
    while v < np.float32(b):
        out.append(float(v))
        v = np.float32(v + np.float32(step))
    return out


def wall_map(ystep, zstep, extent=2.05):
    pts = [(0.5, y, z) for y in frange(-1.0, 1.0, ystep) for z in frange(-1.0, 1.0, zstep)]
    pts += [(-extent, -extent, -extent), (extent, extent, extent)]
    return cc.points(pts)


def any_collision(chk, m, ctor, begin, end):
    c, coll, _ = chk.dda_walk(m, ctor, begin, end, stop_at_collision=False)
    return c, coll


# ---------------------------------------------------------------- test_raycast_dda.cpp:185-244
WAYPOINTS_1 = [(0.1, 0.0, 0.0), (0.1, 0.1, 0.0), (0.2, 0.1, 0.0), (0.2, 0.2, 0.0), (0.3, 0.2, 0.0),
               (0.4, 0.2, 0.0), (0.4, 0.3, 0.0), (0.5, 0.3, 0.0), (0.5, 0.4, 0.0), (0.6, 0.4, 0.0),
               (0.7, 0.4, 0.0), (0.7, 0.5, 0.0), (0.8, 0.5, 0.0), (0.8, 0.6, 0.0), (0.9, 0.6, 0.0)]
WAYPOINTS_2 = [(0.0, 0.1, 0.0), (0.1, 0.1, 0.0), (0.1, 0.2, 0.0), (0.2, 0.2, 0.0), (0.3, 0.2, 0.0),
               (0.3, 0.3, 0.0), (0.4, 0.3, 0.0), (0.4, 0.4, 0.0), (0.5, 0.4, 0.0), (0.6, 0.4, 0.0),
               (0.6, 0.5, 0.0), (0.7, 0.5, 0.0), (0.7, 0.6, 0.0), (0.8, 0.6, 0.0), (0.9, 0.6, 0.0)]


@pytest.mark.parametrize("begin,end,expected", [
    ((0.0, 0.0, 0.0), (1.2, 0.8, 0.0), WAYPOINTS_1),
    ((-0.04, 0.04, 0.0), (1.16, 0.84, 0.0), WAYPOINTS_2),
])
def test_dda_waypoints(port, begin, end, expected):
    m = cc.points([(0.9, 0.6, 0.0), (-2.05, -2.05, -2.05), (2.05, 2.05, 2.05)])
    c, coll, cid = port.dda_walk(m, [0.1, 0.1, 0.1, 0.1, 0.5, 0.0], begin, end, stop_at_collision=True)
    assert len(c) == len(expected)
    assert np.abs(c - np.array(expected, dtype=np.float32)).max() <= 1.0e-6
    assert coll[-1] and not coll[:-1].any() and cid == 0


# ---------------------------------------------------------------- test_raycast_dda.cpp:246-286
def test_dda_intersection(port):
    m = cc.points([(0.6, -0.4, 0.0), (-2.1, -2.1, -2.1), (2.1, 2.1, 2.1)])
    ctor = [0.05, 0.05, 0.05, 0.2, 0.01, 0.0]
    exp1 = [(0.2, 0.0, 0.0), (0.2, -0.2, 0.0), (0.4, -0.2, 0.0), (0.6, -0.2, 0.0), (0.6, -0.4, 0.0)]
    c, coll, _ = port.dda_walk(m, ctor, (0, 0, 0), (1.0, -0.55, 0.0))
    assert len(c) == 5 and np.abs(c - np.array(exp1, np.float32)).max() <= 1e-6 and coll[-1]
    exp2 = exp1 + [(0.8, -0.4, 0.0), (1.0, -0.4, 0.0)]
    c, coll, _ = port.dda_walk(m, ctor, (0, 0, 0), (1.1, -0.55, 0.0))
    assert len(c) == 7 and np.abs(c - np.array(exp2, np.float32)).max() <= 1e-6 and not coll.any()


# ---------------------------------------------------------------- test_raycast_dda.cpp:40-104
def test_dda_collision(port):
    m = wall_map(0.1, 0.1)
    hit_range = float(np.float32(math.sqrt(3.0) * 0.1))
    ctor = [0.1, 0.1, 0.1, 0.1, 0.5, hit_range]
    for y in frange(-0.8, 0.8, 0.11):
        for z in frange(-0.8, 0.8, 0.13):
            end = (1.0, float(np.float32(y * 2.0)), float(np.float32(z * 2.0)))
            c, coll, _ = port.dda_walk(m, ctor, (0, 0, 0), end, stop_at_collision=True)
            assert coll.any(), (y, z)
            first = c[np.argmax(coll)]
            assert np.linalg.norm(first - np.array([0.5, y, z])) <= 0.2
    eps = 0.05
    for y in frange(-1.0, 1.0, 0.11):
        for z in frange(-1.0, 1.0, 0.13):
            end = (float(np.float32(0.5 - hit_range - eps)), y, z)
            _, coll = any_collision(port, m, ctor, (0, 0, 0), end)
            assert not coll.any(), (y, z)
    _, coll = any_collision(port, m, ctor, (0, 0, 0), (0.5, 3.0, 0.0))
    assert not coll.any()


# ---------------------------------------------------------------- test_raycast_dda.cpp:106-155
def test_dda_collision_tolerance(port):
    m = wall_map(0.05, 0.1)
    _, coll = any_collision(port, m, [0.05, 0.1, 0.1, 0.1, 0.5, math.sqrt(3.0) * 0.1], (0, 0, 0), (0.5, 0, 0))
    assert coll.any()
    hr = float(np.float32(math.sqrt(3.0) * 0.15))
    _, coll = any_collision(port, m, [0.1, 0.15, 0.15, 0.15, 0.5, hr], (0, 0, 0),
                            (float(np.float32(0.5 - hr)), 0, 0))
    assert not coll.any()


# ---------------------------------------------------------------- test_raycast.cpp:40-147 (KD-tree caster)
def plain_wall(ystep, zstep):
    return cc.points([(0.5, y, z) for y in frange(-1.0, 1.0, ystep) for z in frange(-1.0, 1.0, zstep)])


def test_kd_raycast_collision(port):
    m = plain_wall(0.1, 0.1)
    hit_range = float(np.float32(0.1) * np.sqrt(np.float32(3.0)))
    ctor = [0.1, 0.1, 0.1, hit_range]
    for y in frange(-0.8, 0.8, 0.11):
        for z in frange(-0.8, 0.8, 0.13):
            end = (1.0, float(np.float32(y * 2.0)), float(np.float32(z * 2.0)))
            pos, coll, _, _ = port.kd_walk(m, ctor, (0, 0, 0), end, stop_at_collision=True)
            assert coll.any(), (y, z)
            assert np.linalg.norm(pos[np.argmax(coll)] - np.array([0.5, y, z])) <= 0.2
    for y in frange(-1.0, 1.0, 0.11):
        for z in frange(-1.0, 1.0, 0.13):
            end = (float(np.float32(0.5 - hit_range * 2.0)), y, z)
            _, coll, _, _ = port.kd_walk(m, ctor, (0, 0, 0), end, stop_at_collision=False)
            assert not coll.any(), (y, z)
    _, coll, _, _ = port.kd_walk(m, ctor, (0, 0, 0), (0.5, 3.0, 0.0), stop_at_collision=False)
    assert not coll.any()


# ---------------------------------------------------------------- test_raycast.cpp:149-208 (SinAng)
def test_kd_raycast_sin_angle(port):
    m = plain_wall(0.1, 0.1)
    ctor = [0.1, 0.1, 0.1, float(np.float32(0.1) * np.sqrt(np.float32(3.0)))]
    for begin, end, want, tol in [((0, 0, 0), (1, 0, 0), 1.0, 0.1), ((0, 5, 0), (1, -5, 0), math.sin(0.5 / 5.0), 0.05),
                                  ((0, 3, 0), (1, -3, 0), math.sin(0.5 / 3.0), 0.05)]:
        pos, coll, sa, _ = port.kd_walk(m, ctor, begin, end, stop_at_collision=True)
        assert coll.any()
        assert abs(sa[np.argmax(coll)] - want) <= tol


# ---------------------------------------------------------------- test_chunked_kdtree.cpp:38-88
def test_chunked_kdtree_radius_search(port):
    pts = cc.points([(0.5, 0.5, 0.5), (0.8, 0.0, 0.0), (1.3, 0.0, 0.0), (0.0, 0.2, 0.0), (0.0, -0.3, 0.0)])
    m = port.create(pts, None, None, chunk_length=1.0, max_search_radius=0.3)
    for q, want in [((0.5, 0.5, 0.5), 0), ((0.5, 0.4, 0.5), 0), ((1.05, 0.0, 0.0), 1), ((1.1, 0.0, 0.0), 2),
                    ((0.0, -0.05, 0.0), 3), ((0.0, -0.15, 0.0), 4)]:
        i, _ = m.radius_search(q, 0.3)
        assert i == want, (q, i, want)
    # radius > chunk length: the reference throws (chunked_kdtree.h:224-225); the checker reports -2
    assert m.radius_search((0, 0, 0), 1.5)[0] == -2


# ---------------------------------------------------------------- test_quat.cpp:234-290
def axis_angle(axis, ang):
    a = np.array(axis, dtype=np.float64)
    a /= np.linalg.norm(a)
    s = math.sin(ang / 2)
    return np.array([a[0] * s, a[1] * s, a[2] * s, math.cos(ang / 2)], dtype=np.float32)


def test_quat_rotate_axes(port):
    v = [(1, 0, 0), (0, 1, 0), (0, 0, 1)]
    r = [axis_angle((1, 0, 0), math.pi / 2), axis_angle((0, 1, 0), -math.pi / 2), axis_angle((0, 0, 1), -math.pi / 2)]
    ans = [[(1, 0, 0), (0, 0, 1), (0, -1, 0)], [(0, 0, 1), (0, 1, 0), (-1, 0, 0)], [(0, -1, 0), (1, 0, 0), (0, 0, 1)]]
    for i in range(3):
        for j in range(3):
            out = port.quat_rotate(r[j], v[i])
            assert np.abs(out - np.array(ans[j][i], np.float32)).max() < 1e-6
    # the survey's probe of the reference build: Quat((0,0,1),0.5)*Vec3(1,2,3)
    out = port.quat_rotate(axis_angle((0, 0, 1), 0.5), (1, 2, 3))
    assert np.allclose(out, [-0.081268549, 2.23459053, 3.0], atol=1e-6)


# ---------------------------------------------------------------- test_pf.cpp:330-391 (Entropy)
def test_pf_entropy(port):
    n = 10
    prior = np.full(n, 1.0 / n, dtype=np.float32)
    lik = np.zeros(n, np.float32)
    lik[0] = 1.0
    _, ent, kept = port.pf_update(prior, lik)
    assert kept and ent == 0
    _, ent, kept = port.pf_update(prior, np.full(n, 0.1, np.float32))
    assert kept and abs(ent - 2.303) < 1e-3
    l1 = np.full(n, 0.025, np.float32)
    l1[4:6] = 0.4
    l2 = np.full(n, 0.025, np.float32)
    l2[2:8] = 0.15
    assert port.pf_update(prior, l2)[1] > port.pf_update(prior, l1)[1]
    # all-zero likelihood -> particles restored (pf.h:274-278)
    p, _, kept = port.pf_update(prior, np.zeros(n, np.float32))
    assert not kept and np.array_equal(p, prior)


# ---------------------------------------------------------------- test_pf.cpp:210-289 (ResampleFirstAndLastParticle)
@pytest.mark.parametrize("probs,expected", [
    ([1.0e-6, 0.2, 0.2, 0.2, 0.4 - 1.0e-6], [1.0, 2.0, 3.0, 4.0, 4.0]),
    ([0.2, 0.2, 0.2, 0.4 - 1.0e-6, 1.0e-6], [0.0, 1.0, 2.0, 3.0, 3.0]),
])
def test_pf_resample_known_answers(port, probs, expected):
    probs = np.array(probs, dtype=np.float64).astype(np.float32)
    probs[np.argmax(probs)] = np.float32(0.4) - np.float32(1.0e-6)  # `0.4f - small_prob` in float, as the test writes it
    out_s, out_p = port.pf_resample_1d(probs, [0.0, 1.0, 2.0, 3.0, 4.0], seed=12345)
    assert np.array_equal(out_s, np.array(expected, dtype=np.float32))
    assert np.all(out_p == np.float32(1.0 / 5))


# test_pf.cpp:190-208 (ResampleFlatLikelihood): equal weights keep every particle where it is
def test_pf_resample_flat_likelihood_is_identity(port):
    rng = np.random.default_rng(3)
    states = (12.3 + 0.45 * rng.normal(size=10)).astype(np.float32)
    out_s, _ = port.pf_resample_1d(np.full(10, 0.1, np.float32), states, seed=99)
    assert np.array_equal(out_s, states)


def test_pf_resample_port_equals_reference_build(port, reference):
    rng = np.random.default_rng(17)
    for n in (2, 5, 64, 1000):
        for sigma in (0.0, 0.3):
            probs = rng.random(n).astype(np.float32) ** 4
            probs[rng.integers(0, n, n // 4)] = 0.0
            states = rng.normal(size=n).astype(np.float32)
            a = reference.pf_resample_1d(probs, states, seed=12345 + n, sigma=sigma)
            b = port.pf_resample_1d(probs, states, seed=12345 + n, sigma=sigma)
            assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


# ---------------------------------------------------------------- groundwork for scope row f3 (motion prediction)
def test_motion_prediction_port_equals_reference_build(port, reference):
    rng = np.random.default_rng(23)
    for trial in range(20):
        def pose():
            q = rng.normal(size=4)
            q /= np.linalg.norm(q)
            return cc.poses([rng.uniform(-5, 5, 3)], [q])[0]
        a, b = pose(), pose()
        if trial % 4 == 0:
            b = a.copy()  # no rotation: the |w| >= 1 - 1e-6 branch of getAxisAng (quat.h:224-229)
            b["px"] += np.float32(0.3)
        st = np.zeros(64, dtype=cc.MOTION_STATE)
        st["pos"] = rng.uniform(-10, 10, (64, 3))
        q = rng.normal(size=(64, 4))
        st["rot"] = q / np.linalg.norm(q, axis=1, keepdims=True)
        for f in ("noise_ll", "noise_la", "noise_al", "noise_aa"):
            st[f] = rng.normal(0, 0.05, 64)
        st["odom_err_integ_lin"] = rng.normal(0, 0.02, (64, 3))
        st["odom_err_integ_ang"] = rng.normal(0, 0.02, (64, 3))
        ra = reference.motion_predict(a, b, 0.05, 10.0, 10.0, st)
        rb = port.motion_predict(a, b, 0.05, 10.0, 10.0, st)
        for f in cc.MOTION_STATE.names:
            assert np.array_equal(ra[f], rb[f]), (trial, f)
        assert not np.array_equal(ra["pos"], st["pos"])


def test_state6dof_resample_port_equals_reference_build(port, reference):
    """The node's resample call (src/mcl_3dl.cpp:809-815) on State6DOF particles: duplicates get position /
    rpy noise through State6DOF::generateNoise and operator+ (state_6dof.h:226-261)."""
    rng = np.random.default_rng(31)
    for n, sp, sr in ((8, (0.05, 0.05, 0.0), (0.0, 0.0, 0.02)), (300, (0.05, 0.05, 0.05), (0.05, 0.05, 0.05)),
                      (64, (0, 0, 0), (0, 0, 0))):
        st = np.zeros(n, dtype=cc.MOTION_STATE)
        st["pos"] = rng.uniform(-10, 10, (n, 3))
        q = rng.normal(size=(n, 4))
        st["rot"] = q / np.linalg.norm(q, axis=1, keepdims=True)
        for f in ("noise_ll", "noise_la", "noise_al", "noise_aa"):
            st[f] = rng.normal(0, 0.05, n)
        st["odom_err_integ_lin"] = rng.normal(0, 0.02, (n, 3))
        st["odom_err_integ_ang"] = rng.normal(0, 0.02, (n, 3))
        probs = (rng.random(n) ** 6).astype(np.float32)   # a few heavy particles -> many duplicates
        a = reference.pf_resample_6dof(probs, st, 4242 + n, sp, sr)
        b = port.pf_resample_6dof(probs, st, 4242 + n, sp, sr)
        for f in cc.MOTION_STATE.names:
            assert np.array_equal(a[0][f], b[0][f]), (n, f)
        assert np.array_equal(a[1], b[1])
        if any(sp) or any(sr):
            assert (b[0]["noise_ll"] == 0).sum() > 0   # duplicates lose their odometry-noise draw


# ---------------------------------------------------------------- groundwork for scope row f4 (scan filtering)
def test_filter_clip_and_point_budget_port_equals_reference_build(port, reference):
    rng = np.random.default_rng(29)
    pts = cc.points(rng.uniform(-12, 12, (5000, 3)) * np.array([1, 1, 0.3]))
    # points exactly on the clip boundaries (the comparisons are strict, likelihood.cpp:85-90)
    pts["x"][:4], pts["y"][:4], pts["z"][:4] = [0.5, 10.0, 3.0, 3.0], 0.0, [0.0, 0.0, 2.0, -2.0]
    for args in ((0.5, 10.0, -2.0, 2.0), (0.5, 4.0, -2.0, 2.0), (1.0, 6.5, -0.3, 4.1)):
        ka, kb = reference.filter_clip(pts, *args), port.filter_clip(pts, *args)
        assert np.array_equal(ka, kb) and 0 < kb.sum() < len(pts)
    assert port.filter_clip(pts)[:4].all()  # boundary points are kept
    # the test of test_beam_likelihood.cpp:140-146: z = +-5 is clipped with clip_z = (-0.3, 4.1)
    two = cc.points([[0, 0, 5.0], [0, 0, -5.0], [2, 0, 0.0]])
    assert list(port.filter_clip(two, 0.5, 4.0, -0.3, 4.1)) == [False, False, True]
    for d, g, n, cur in ((96, 8, 64, 64), (96, 8, 64, 65), (96, 8, 64, 768), (96, 8, 64, 100000), (3, 0, 64, 1000)):
        assert reference.global_localization_points(d, g, n, cur) == port.global_localization_points(d, g, n, cur)
    assert port.global_localization_points(96, 8, 64, 768) == 8 and port.global_localization_points(96, 8, 64, 128) == 48


# ---------------------------------------------------------------- golden fixtures (reference outputs)
def test_golden_beam_likelihood_world(port):
    g = golden("beam_likelihood_world.npz")
    pc_map, pc, xs = cc.points(g["map"]), cc.points(g["scan"]), g["xs"]
    k = 0
    for method, mode in ((1, 0), (1, 1), (0, 0), (0, 1)):
        for hr in g["hit_ranges"]:
            assert g["mode"][k] == mode and g["method"][k] == method
            braw = cc.beam_raw(map_grid=(0.1, 0.1, 0.1), num_points_default=len(pc) + 2, beam_likelihood_min=0.2,
                               hit_range=float(hr), add_penalty_short_only_mode=(mode == 1), dda_grid_size=0.1,
                               use_raycast_using_dda=(method == 1))
            m = port.create(pc_map, None, braw, chunk_length=10.0, max_search_radius=1.0)
            ident = cc.poses([[0, 0, 0]], [[0, 0, 0, 1]])
            for i, x in enumerate(xs):
                r = m.measure(cc.poses([[x, 0, 0]], [[0, 0, 0, 1]]), None, pc, np.array([[x, 0, 0]], np.float32))
                assert r["score_beam"][0] == g["likelihood"][k, i], (mode, hr, i)
                s = m.beam_status(ident, cc.points([[x, 0, 0]]), np.zeros((1, 3), np.float32))
                assert s[0, 0] == g["status"][k, i], (mode, hr, i)
            m.close()
            k += 1


@pytest.mark.parametrize("name", ["room_iso", "room_aniso", "room_spread", "room_kd_iso", "room_kd_aniso"])
def test_golden_rooms(port, name):
    g = golden(name + ".npz")
    n_beam, flm, short_only = [int(v) for v in g["beam_cfg"]]
    lik = cc.lik_params(dist_weight=tuple(float(v) for v in g["dist_weight"]))
    braw = cc.beam_raw(num_points_default=n_beam, filter_label_max=flm, add_penalty_short_only_mode=bool(short_only),
                       dda_grid_size=float(g["dda_grid"]), use_raycast_using_dda=bool(int(g["use_dda"])))
    m = port.create(g["map"], lik, braw)
    res = m.measure(g["particles"], g["lik"], g["beam"], g["origins"])
    for f in res.dtype.names:
        assert np.array_equal(res[f], g["result"][f]), f
    assert np.array_equal(m.beam_status(g["particles"], g["beam"], g["origins"]), g["status"])
    # sanity: the fixture exercises every branch
    assert g["result"]["n_short"].sum() and g["result"]["n_hit"].sum() and g["result"]["n_long"].sum()
    if not int(g["use_dda"]):
        assert (g["status"] == 3).sum() > 0  # TOTAL_REFLECTION is live with the KD-tree caster (beam.cpp:186-189)


@pytest.mark.parametrize("tag", ["iso", "aniso"])
def test_golden_radius_search(port, tag):
    g = golden("chunked_radius_search_%s.npz" % tag)
    m = port.create(cc.points(g["pts"]), cc.lik_params(dist_weight=tuple(float(v) for v in g["w"])), None,
                    chunk_length=1.0, max_search_radius=0.3)
    for q, gid, gd2 in zip(g["q"], g["ids"], g["d2"]):
        i, d2 = m.radius_search(q, 0.3)
        assert (i >= 0) == (gid >= 0)
        if gid >= 0:
            assert np.float32(d2) == gd2  # the distance is the contract; equidistant ids may differ
    assert (g["ids"] >= 0).sum() > 500 and (g["ids"] < 0).sum() > 500


def test_golden_transform(port):
    g = golden("transform.npz")
    for i in range(len(g["v"])):
        assert np.array_equal(port.transform_point(g["poses"][i], g["v"][i]), g["transformed"][i])
        q = np.array([g["poses"][i][k] for k in ("qx", "qy", "qz", "qw")], np.float32)
        assert np.array_equal(port.quat_rotate(q, g["v"][i]), g["rotated_raw"][i])


# ---------------------------------------------------------------- cross-check with the recorded reference build
@pytest.mark.parametrize("seed,w,spread,use_dda", [(1, (1, 1, 1), False, True), (2, (1, 1, 5), False, True),
                                                   (3, (1, 1, 5), True, True), (4, (2, 0.5, 3), False, True),
                                                   (5, (1, 1, 1), False, False), (6, (1, 1, 5), False, False),
                                                   (7, (1, 1, 5), True, False)])
def test_port_equals_reference_build(port, reference, seed, w, spread, use_dda):
    s = synth.scene(30_000, 96, 128, 48, spread=spread, seed=seed)
    lik = cc.lik_params(dist_weight=w)
    braw = cc.beam_raw(num_points_default=48, dda_grid_size=0.2 if seed % 2 else 0.1,
                       filter_label_max=1 if seed in (2, 6) else 0xFFFFFFFF, add_penalty_short_only_mode=seed != 3,
                       use_raycast_using_dda=use_dda)
    # max_search_radius as the node derives it: max(match_dist_min, 4*map_grid) = 0.4 (mcl_3dl.cpp:1320-1326);
    # the (2,0.5,3) weights need a larger halo for the chunk search to stay complete.
    msr = 0.4 if min(w) >= 1 else 1.0
    a = reference.create(s["map"], lik, braw, 20.0, msr)
    b = port.create(s["map"], lik, braw, 20.0, msr)
    assert a.beam_params().as_tuple() == b.beam_params().as_tuple()
    ra = a.measure(s["particles"], s["lik"], s["beam"], s["origins"])
    rb = b.measure(s["particles"], s["lik"], s["beam"], s["origins"])
    for f in ra.dtype.names:
        assert np.array_equal(ra[f], rb[f]), f
    assert np.array_equal(a.beam_status(s["particles"], s["beam"], s["origins"]),
                          b.beam_status(s["particles"], s["beam"], s["origins"]))
    # degenerate inputs: empty scans return (1, 0) (likelihood.cpp:111-114, beam.cpp:130-133)
    for m in (a, b):
        r = m.measure(s["particles"][:3], None, None, s["origins"])
        assert (r["score_like"] == 1).all() and (r["score_beam"] == 1).all() and (r["match_cnt"] == 0).all()


def test_pose_estimate_port_equals_reference_build(port, reference):
    """bias + expectationBiased + max + covariance (src/mcl_3dl.cpp:428-452,704-724; pf.h:246-251,281-374): the port's
    restatement against the reference's own pf::ParticleFilter / ParticleWeightedMeanQuat / State6DOF::covElement /
    NormalLikelihood, bit for bit."""
    from oracle import cpu_checker as cc
    from mcl_3dl_b200 import synth
    for seed, n, with_prev in ((1, 64, True), (2, 777, False), (3, 4096, True)):
        rng = np.random.default_rng(seed)
        st = np.zeros(n, dtype=cc.MOTION_STATE)
        st["pos"] = rng.normal([3, 4, 0.5], [0.2, 0.2, 0.05], (n, 3))
        st["rot"] = synth.quat_from_rpy(rng.normal([0, 0, 3.0], [0.02, 0.02, 0.3], (n, 3))) * \
            (1 + rng.normal(0, 1e-3, (n, 1))).astype(np.float32)
        p = rng.uniform(0.1, 1, n).astype(np.float32)
        p /= p.sum()
        prev = synth.make_poses([[3.1, 4.0, 0.5]], synth.quat_from_rpy([[0, 0, 3.05]])) if with_prev else None
        a = port.pf_estimate(p, st, prev, 0.2, 0.1)
        b = reference.pf_estimate(p, st, prev, 0.2, 0.1)
        assert a[0].tobytes() == b[0].tobytes() and a[1] == b[1] and a[2].tobytes() == b[2].tobytes()
