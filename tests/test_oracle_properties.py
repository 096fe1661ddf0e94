"""Property tests (hypothesis): the repo-owned oracle equals the reference's own sources bit for bit on random
small worlds — DDA walks (every visited voxel), KD-tree walks (positions, sin_angle_), radius search, per-ray
BeamStatus and per-particle records.  The reference's answers are recorded (tests/recorded_reference.py), so every
test runs a fixed, seeded set of examples drawn from its strategies' domain rather than fresh draws."""
import numpy as np
from hypothesis import HealthCheck, Phase, example, given, settings
from hypothesis import strategies as st

from oracle import cpu_checker as cc


def recorded_examples(count, **domain):
    """@given over `domain` (name -> (lo, hi) integer range or list of choices), run as `count` explicit examples drawn
    from it with a fixed seed and nothing else: the reference's answers exist for exactly these inputs."""
    rng = np.random.default_rng(count * 7919 + len(domain))
    cases = [{k: (int(rng.integers(v[0], v[1] + 1)) if isinstance(v, tuple) else v[int(rng.integers(len(v)))])
              for k, v in domain.items()} for _ in range(count)]
    strategies = {k: st.integers(*v) if isinstance(v, tuple) else st.sampled_from(v) for k, v in domain.items()}

    def deco(f):
        f = given(**strategies)(f)
        for c in cases:
            f = example(**c)(f)
        return settings(phases=[Phase.explicit], deadline=None,
                        suppress_health_check=[HealthCheck.function_scoped_fixture])(f)
    return deco


def world(seed, n):
    rng = np.random.default_rng(seed)
    kind = seed % 3
    if kind == 0:      # scattered points
        pts = rng.uniform(-2, 2, (n, 3))
    elif kind == 1:    # lattice wall: exact ties and voxel-boundary coordinates
        g = np.arange(-1.0, 1.0, 0.1, dtype=np.float32)
        yy, zz = np.meshgrid(g, g)
        pts = np.stack([np.full(yy.size, 0.5), yy.ravel(), zz.ravel()], 1)[:max(n, 8)]
    else:              # two noisy planes
        a = np.c_[rng.uniform(-2, 2, n // 2), rng.uniform(-2, 2, n // 2), rng.normal(0, 0.01, n // 2)]
        b = np.c_[rng.normal(1.0, 0.01, n - n // 2), rng.uniform(-2, 2, n - n // 2), rng.uniform(-1, 2, n - n // 2)]
        pts = np.vstack([a, b])
    pts = np.vstack([pts, [[-2.55, -2.55, -2.55], [2.55, 2.55, 2.55]]]).astype(np.float32)
    lab = (rng.random(len(pts)) < 0.2).astype(np.uint32) * 2
    return cc.points(pts, lab), rng


@recorded_examples(60, seed=(0, 10_000), n=(4, 120), grid=[0.05, 0.1, 0.2, 0.37], tol=[0.0, 0.1, 0.3])
def test_dda_walk_matches_reference(port, reference, seed, n, grid, tol):
    m, rng = world(seed, n)
    ctor = [0.1, 0.1, 0.1, grid, 0.25 * np.pi / 180.0 if seed % 2 else 0.5, tol]
    for _ in range(4):
        b = rng.uniform(-2.6, 2.6, 3) if rng.random() < 0.8 else rng.uniform(-4, 4, 3)
        e = rng.uniform(-3, 3, 3)
        if seed % 5 == 0:
            e[2] = b[2]   # axis-aligned components: infinite t_delta path (raycast_using_dda.h:88-92)
        a = reference.dda_walk(m, ctor, b, e, stop_at_collision=bool(seed % 2))
        p = port.dda_walk(m, ctor, b, e, stop_at_collision=bool(seed % 2))
        assert np.array_equal(a[0], p[0]) and np.array_equal(a[1], p[1]) and a[2] == p[2]


@recorded_examples(60, seed=(0, 10_000), n=(4, 120), hit=[0.0, 0.17, 0.3])
def test_kd_walk_matches_reference(port, reference, seed, n, hit):
    m, rng = world(seed, n)
    ctor = [0.1, 0.1 if seed % 2 else 0.05, 0.1, hit]
    for _ in range(3):
        b, e = rng.uniform(-2, 2, 3), rng.uniform(-2, 2, 3)
        a = reference.kd_walk(m, ctor, b, e, stop_at_collision=False)
        p = port.kd_walk(m, ctor, b, e, stop_at_collision=False)
        assert np.array_equal(a[0], p[0]) and np.array_equal(a[1], p[1]) and np.array_equal(a[2], p[2])
        # the colliding point may differ only between exactly equidistant map points; both pick the lowest index
        assert a[3] == p[3]


@recorded_examples(25, seed=(0, 10_000), n=(20, 400), use_dda=[False, True], w=[(1, 1, 1), (1, 1, 5), (2, 1, 3)])
def test_records_match_reference(port, reference, seed, n, use_dda, w):
    m, rng = world(seed, n)
    lik = cc.lik_params(dist_weight=w, match_dist_min=0.2 if seed % 2 else 0.35)
    braw = cc.beam_raw(num_points_default=6, use_raycast_using_dda=use_dda, dda_grid_size=0.2 if seed % 3 else 0.1,
                       filter_label_max=1 if seed % 4 == 0 else 0xFFFFFFFF, hit_range=0.3 if seed % 2 else 0.1,
                       add_penalty_short_only_mode=bool(seed % 3))
    a = reference.create(m, lik, braw, 20.0, 1.0)
    b = port.create(m, lik, braw, 20.0, 1.0)
    P = 5
    q = rng.normal(0, 1, (P, 4))
    poses = cc.poses(rng.uniform(-1.5, 1.5, (P, 3)), q)
    scan_l = cc.points(rng.uniform(-2, 2, (9, 3)))
    scan_b = cc.points(rng.uniform(-2, 2, (6, 3)), rng.integers(0, 2, 6))
    org = rng.uniform(-0.3, 0.3, (2, 3)).astype(np.float32)
    ra, rb = a.measure(poses, scan_l, scan_b, org), b.measure(poses, scan_l, scan_b, org)
    for f in ra.dtype.names:
        assert np.array_equal(ra[f], rb[f]), f
    assert np.array_equal(a.beam_status(poses, scan_b, org), b.beam_status(poses, scan_b, org))
    for _ in range(5):
        qq = rng.uniform(-2.5, 2.5, 3).astype(np.float32)
        ia, da = a.radius_search(qq, 0.3)
        ib, db = b.radius_search(qq, 0.3)
        assert (ia >= 0) == (ib >= 0) and (ia < 0 or np.float32(da) == np.float32(db))
