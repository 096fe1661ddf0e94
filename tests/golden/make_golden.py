"""Regenerate tests/golden/*.npz by running the REFERENCE's own sources (oracle/_ref).

Only runnable in the development container (needs /root/reference to build oracle/_ref).
    python tests/golden/make_golden.py           # the fixtures below
    python tests/golden/make_golden.py --calls   # reference_calls.npz
The committed .npz files hold inputs AND the reference outputs, so the GPU box (which has no
/root/reference) can check both the port oracle and the CUDA engine against them.

Fixtures
  beam_likelihood_world.npz  the world and parameter sweep of test/src/test_beam_likelihood.cpp:81-138
                             (both casters; rows 0-11 DDA, 12-23 KD-tree): the 100-position likelihood row and
                             the 100 BeamStatus codes the reference test only prints.
  room_kd_iso / room_kd_aniso  rooms measured with the KD-tree raycaster (the node's default).
  room_iso.npz / room_aniso.npz / room_spread.npz
                             synthetic room scenes (mcl_3dl_b200.synth) -> per-particle records + per-ray status.
  chunked_radius_search.npz  random ChunkedKdtree::radiusSearch queries (ids + d2), incl. chunk borders.
  transform.npz              State6DOF::transform of random points by random (non-unit) quaternions.
  reference_calls.npz        the reference's answers to every call of the tests that compare the port with it call by
                             call (the `reference` fixture, tests/recorded_reference.py): those tests run once against
                             the live build and record what it returned.
"""
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from mcl_3dl_b200 import synth  # noqa: E402
from oracle import cpu_checker as cc  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


def beam_likelihood_world():
    """test/src/test_beam_likelihood.cpp:81-116 restated: 5x5 patch at x=2, two clip-test points,
    two map-extent dummies."""
    raw = []
    y = np.float32(-0.2)
    while y <= np.float32(0.2):
        z = np.float32(-0.2)
        while z <= np.float32(0.2):
            raw.append((2.0, float(y), float(z)))
            z = np.float32(z + np.float32(0.1))
        y = np.float32(y + np.float32(0.1))
    raw_pc = raw + [(0.0, 0.0, 5.0), (0.0, 0.0, -5.0)]
    pc_map = raw_pc + [(-100.05, 100.0, -0.05), (100.0, -100.05, 4.0)]
    return np.array(raw_pc, dtype=np.float32), np.array(pc_map, dtype=np.float32)


def gen_beam_likelihood(ref):
    raw_pc, pc_map = beam_likelihood_world()
    # LidarMeasurementModelBeam::filter with clip_z_min=-0.3, clip_z_max=4.1 and the defaults
    # clip_near=0.5, clip_far=4.0 keeps exactly the 25... the test asserts size()-2 (:140)
    r2 = raw_pc[:, 0] ** 2 + raw_pc[:, 1] ** 2
    keep = ~((r2 > 16.0) | (r2 < 0.25) | (raw_pc[:, 2] < np.float32(-0.3)) | (np.float32(4.1) < raw_pc[:, 2]))
    pc = raw_pc[keep]
    assert len(pc) == len(raw_pc) - 2
    out = {"map": pc_map, "scan": pc}
    xs = np.array([np.float32(0.1 * i) for i in range(-50, 50)], dtype=np.float32)
    out["xs"] = xs
    hrs = []
    hr = 0.0
    while hr <= 1.0:
        hrs.append(hr)
        hr += 0.2
    out["hit_ranges"] = np.array(hrs, dtype=np.float64)
    lik_rows, status_rows, modes, methods = [], [], [], []
    for method, mode in ((1, 0), (1, 1), (0, 0), (0, 1)):  # DDA rows first (kept at indices 0..11), then the KD-tree caster
        for hr in hrs:
            braw = cc.beam_raw(map_grid=(0.1, 0.1, 0.1), num_points_default=len(raw_pc), beam_likelihood_min=0.2,
                               hit_range=hr, add_penalty_short_only_mode=(mode == 1), dda_grid_size=0.1,
                               use_raycast_using_dda=(method == 1))
            m = ref.create(cc.points(pc_map), None, braw, chunk_length=10.0, max_search_radius=1.0)
            row = []
            for x in xs:
                p = cc.poses([[x, 0, 0]], [[0, 0, 0, 1]])
                # origins = {pos}; State6DOF(pos, Quat())  (test_beam_likelihood.cpp:165-170)
                r = m.measure(p, None, cc.points(pc), np.array([[x, 0, 0]], dtype=np.float32))
                row.append(r["score_beam"][0])
            lik_rows.append(row)
            # getBeamStatus(kdtree, Vec3(), p=(x,0,0)) (:196-198): identity pose, origin 0, one-point scan
            st = []
            ident = cc.poses([[0, 0, 0]], [[0, 0, 0, 1]])
            for x in xs:
                s = m.beam_status(ident, cc.points([[x, 0, 0]]), np.zeros((1, 3), dtype=np.float32))
                st.append(int(s[0, 0]))
            status_rows.append(st)
            modes.append(mode)
            methods.append(method)
            m.close()
    out["likelihood"] = np.array(lik_rows, dtype=np.float32)
    out["status"] = np.array(status_rows, dtype=np.uint8)
    out["mode"] = np.array(modes, dtype=np.int32)
    out["method"] = np.array(methods, dtype=np.int32)  # 1 = RaycastUsingDDA, 0 = RaycastUsingKDTree
    np.savez_compressed(os.path.join(OUT, "beam_likelihood_world.npz"), **out)
    print("beam_likelihood_world", out["likelihood"].shape)


def gen_room(ref, name, dist_weight, spread, seed, n_map=12000, P=48, n_lik=64, n_beam=24, filter_label_max=0xFFFFFFFF,
             short_only=True, dda_grid=0.2, use_dda=True):
    s = synth.scene(n_map, P, n_lik, n_beam, spread=spread, n_origins=2, seed=seed)
    lik = cc.lik_params(dist_weight=dist_weight)
    braw = cc.beam_raw(num_points_default=n_beam, filter_label_max=filter_label_max,
                       add_penalty_short_only_mode=short_only, dda_grid_size=dda_grid, use_raycast_using_dda=use_dda)
    m = ref.create(s["map"], lik, braw, chunk_length=20.0, max_search_radius=0.4)
    res = m.measure(s["particles"], s["lik"], s["beam"], s["origins"])
    st = m.beam_status(s["particles"], s["beam"], s["origins"])
    np.savez_compressed(os.path.join(OUT, name + ".npz"), map=s["map"], particles=s["particles"], lik=s["lik"],
                        beam=s["beam"], origins=s["origins"], result=res, status=st,
                        dist_weight=np.array(dist_weight, dtype=np.float32),
                        beam_cfg=np.array([n_beam, filter_label_max, 1 if short_only else 0], dtype=np.uint64),
                        use_dda=np.int32(1 if use_dda else 0),
                        dda_grid=np.float32(dda_grid))
    print(name, len(s["map"]), "matched", res["match_cnt"].mean(), "short/hit/long/total_ref",
          res["n_short"].mean(), res["n_hit"].mean(), res["n_long"].mean(), (st == 3).sum(axis=1).mean())
    m.close()


def gen_radius_search(ref):
    rng = np.random.default_rng(7)
    pts = rng.uniform(-3, 3, (4000, 3)).astype(np.float32)
    # cluster some points around chunk borders (chunk length 1.0)
    pts[:1000] = np.round(pts[:1000]) + rng.normal(0, 0.05, (1000, 3)).astype(np.float32)
    for w, tag in (((1, 1, 1), "iso"), ((1, 1, 5), "aniso")):
        m = ref.create(cc.points(pts), cc.lik_params(dist_weight=w), None, chunk_length=1.0, max_search_radius=0.3)
        q = rng.uniform(-3.2, 3.2, (3000, 3)).astype(np.float32)
        q[:800] = np.round(q[:800]) + rng.normal(0, 0.03, (800, 3)).astype(np.float32)
        ids, d2 = [], []
        for v in q:
            i, d = m.radius_search(v, 0.3)
            ids.append(i)
            d2.append(d if i >= 0 else -1.0)
        np.savez_compressed(os.path.join(OUT, "chunked_radius_search_%s.npz" % tag), pts=pts, q=q,
                            ids=np.array(ids, dtype=np.int32), d2=np.array(d2, dtype=np.float32),
                            w=np.array(w, dtype=np.float32))
        print("radius_search", tag, "found", int((np.array(ids) >= 0).sum()))
        m.close()


def gen_transform(ref):
    rng = np.random.default_rng(11)
    q = rng.normal(0, 1, (256, 4)).astype(np.float32)
    pos = rng.uniform(-50, 50, (256, 3)).astype(np.float32)
    v = rng.uniform(-10, 10, (256, 3)).astype(np.float32)
    P = cc.poses(pos, q)
    t = np.array([ref.transform_point(P[i], v[i]) for i in range(256)], dtype=np.float32)
    r = np.array([ref.quat_rotate(q[i], v[i]) for i in range(256)], dtype=np.float32)
    np.savez_compressed(os.path.join(OUT, "transform.npz"), poses=P, v=v, transformed=t, rotated_raw=r)
    print("transform ok")


def gen_calls():
    env = dict(os.environ, MCL3DL_RECORD_REFERENCE="1")
    tests = [os.path.join(ROOT, "tests", t) for t in ("test_oracle_golden.py", "test_oracle_properties.py")]
    subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", "-k", "reference"] + tests,
                   env=env, check=True)


if __name__ == "__main__":
    assert cc.build("reference"), "oracle/_ref cannot be built here (no /root/reference)"
    if "--calls" in sys.argv:
        gen_calls()
        sys.exit(0)
    ref = cc.CpuChecker("reference")
    gen_beam_likelihood(ref)
    gen_room(ref, "room_iso", (1, 1, 1), False, seed=100)
    gen_room(ref, "room_aniso", (1, 1, 5), False, seed=200, filter_label_max=1, short_only=False)
    gen_room(ref, "room_spread", (1, 1, 5), True, seed=300, dda_grid=0.1)
    gen_room(ref, "room_kd_iso", (1, 1, 1), False, seed=400, use_dda=False)
    gen_room(ref, "room_kd_aniso", (1, 1, 5), False, seed=500, use_dda=False, filter_label_max=1, short_only=False)
    gen_radius_search(ref)
    gen_transform(ref)
