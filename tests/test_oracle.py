"""CPU tests: pin the oracle against the reference's own compiled function / committed golden vectors,
and against independent numpy restatements (float64) of the algorithms it restates."""
from pathlib import Path

import numpy as np
import pytest

GOLD = Path(__file__).parent / "golden"


def test_brute_force_orb_matches_golden_vectors(oracle_mod):
    """Golden vectors were produced by the reference's bruteForceSearchORB (features.cpp:168-182)."""
    g = np.load(GOLD / "brute_force_orb.npz")
    for name in ("a", "b", "c", "d", "ties"):
        hd, idx = oracle_mod.brute_force_orb(g[f"{name}_q"], g[f"{name}_t"])
        assert np.array_equal(hd, g[f"{name}_hd"]), name
        assert np.array_equal(idx, g[f"{name}_idx"]), name
    # quirk: the last train row is never examined (features.cpp:174)
    assert g["a_idx"].max() <= len(g["a_t"]) - 2
    assert (g["c_hd"] == 257).all() and (g["c_idx"] == -1).all()


def test_brute_force_orb_matches_reference_binary(oracle_mod):
    """Uniformly random cases; the expected values are the reference's bruteForceSearchORB outputs (make_golden.py)."""
    g = np.load(GOLD / "brute_force_orb_random.npz")
    for i, (nq, nt) in enumerate([(50, 300), (7, 2), (3, 1), (128, 1000)]):
        q, t = g[f"r{i}_q"], g[f"r{i}_t"]
        assert q.shape == (nq, 32) and t.shape == (nt, 32)
        hd, idx = oracle_mod.brute_force_orb(q, t)
        assert np.array_equal(hd, g[f"r{i}_hd"]) and np.array_equal(idx, g[f"r{i}_idx"]), (nq, nt)


def test_hamming_against_numpy(oracle_mod):
    rng = np.random.default_rng(1)
    q = rng.integers(0, 256, (40, 32), dtype=np.uint8)
    t = rng.integers(0, 256, (90, 32), dtype=np.uint8)
    hd, idx = oracle_mod.brute_force_orb(q, t)
    d = np.unpackbits(q[:, None, :] ^ t[None, :-1, :], axis=2).sum(2)
    assert np.array_equal(hd, d.min(1))
    assert np.array_equal(idx, d.argmin(1))  # argmin returns the first minimum == lowest index wins


def test_rng_known_answers(oracle_mod):
    """Pins the counter-based generator shared with the CUDA path (DESIGN.md)."""
    L = oracle_mod.lib()
    vals = [L.oracle_rand31(0, 0, 0, 0), L.oracle_rand31(1, 2, 3, 4), L.oracle_rand31(2**63, 12345, 200, 7)]
    def mix(z):
        z = (z + 0x9E3779B97F4A7C15) % 2**64
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) % 2**64
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) % 2**64
        return z ^ (z >> 31)
    def r31(seed, pair, stream, ctr):
        k = mix(seed ^ mix(pair))
        return mix(k ^ ((stream << 32) | ctr)) >> 33
    assert vals == [r31(0, 0, 0, 0), r31(1, 2, 3, 4), r31(2**63, 12345, 200, 7)]
    assert all(0 <= v < 2**31 for v in vals)


def test_match_distance_formula(oracle_mod):
    """distance = hd/256.0 + (float)rand()/(1000.0*RAND_MAX), stored as float (node.cpp:573)."""
    L = oracle_mod.lib()
    for hd, r in [(0, 0), (17, 123456789), (127, 2**31 - 1), (64, 2**24 + 1)]:
        want = np.float32(hd / 256.0 + float(np.float32(r)) / (1000.0 * 2147483647.0))
        assert L.oracle_match_distance(hd, r) == want
    # jitter never reorders different Hamming distances
    assert L.oracle_match_distance(10, 2**31 - 1) < L.oracle_match_distance(11, 0)


def test_feature_matching_filters_and_sorts(oracle_mod):
    from rgbdslam_v2_b200 import synth
    p = synth.make_pair(3, 600)
    m = oracle_mod.feature_matching_orb(p["desc_newer"], p["desc_older"], 300, seed=9, pair=4)
    assert len(m) <= 300
    assert (np.diff(m["distance"]) >= 0).all()
    hd, idx = oracle_mod.brute_force_orb(p["desc_newer"], p["desc_older"])
    assert (hd[m["queryIdx"]] < 128).all()
    assert np.array_equal(idx[m["queryIdx"]], m["trainIdx"])
    assert (m["imgIdx"] == -1).all()
    # kept matches are the strongest ones
    kept = np.zeros(len(hd), bool)
    kept[m["queryIdx"]] = True
    rest = hd[(~kept) & (hd < 128)]
    if len(rest):
        assert rest.min() >= hd[m["queryIdx"]].max() - 0  # jitter < 1/256


def _kabsch_weighted(P, Q, w):
    """float64 closed form: R,t minimising sum w |R p + t - q|^2."""
    w = w / w.sum()
    mp, mq = (w[:, None] * P).sum(0), (w[:, None] * Q).sum(0)
    Cm = ((Q - mq) * w[:, None]).T @ (P - mp)
    U, S, Vt = np.linalg.svd(Cm)
    D = np.diag([1, 1, np.sign(np.linalg.det(U) * np.linalg.det(Vt))])
    R = U @ D @ Vt
    return R, mq - R @ mp


def test_transform_from_matches_against_numpy_kabsch(oracle_mod):
    from rgbdslam_v2_b200 import synth
    rng = np.random.default_rng(11)
    for n in (4, 7, 50, 300):
        T = synth.random_rigid(rng, 0.3, 20)
        P = synth._random_points(rng, n)
        Q = P @ T[:3, :3].T + T[:3, 3] + rng.normal(size=(n, 3)) * 1e-3
        x1 = np.concatenate([P, np.ones((n, 1))], 1).astype(np.float32)
        x2 = np.concatenate([Q, np.ones((n, 1))], 1).astype(np.float32)
        m = np.zeros(n, oracle_mod.DMATCH_DTYPE)
        m["queryIdx"] = m["trainIdx"] = np.arange(n)
        To = oracle_mod.get_transform_from_matches(x1, x2, m)
        w = 1.0 / (x1[:, 2].astype(np.float64) * x2[:, 2])  # transformation_estimation_euclidean.cpp:25
        R, t = _kabsch_weighted(x1[:, :3].astype(np.float64), x2[:, :3].astype(np.float64), w)
        assert np.abs(To[:3, :3] - R).max() < 5e-5
        assert np.abs(To[:3, 3] - t).max() < 5e-5
        assert np.allclose(To[3], [0, 0, 0, 1])
        assert abs(np.linalg.det(To[:3, :3].astype(np.float64)) - 1) < 1e-5


def test_transform_from_matches_reflection_case(oracle_mod):
    """Coplanar correspondences with noise can give det(U)det(V) < 0; R must still be a rotation."""
    rng = np.random.default_rng(2)
    P = np.concatenate([rng.uniform(-1, 1, (6, 2)), np.full((6, 1), 2.0)], 1)
    T = np.eye(4); T[:3, 3] = [0.1, -0.05, 0.02]
    Q = P + T[:3, 3] + rng.normal(size=P.shape) * 1e-4
    x1 = np.concatenate([P, np.ones((6, 1))], 1).astype(np.float32)
    x2 = np.concatenate([Q, np.ones((6, 1))], 1).astype(np.float32)
    m = np.zeros(6, oracle_mod.DMATCH_DTYPE)
    m["queryIdx"] = m["trainIdx"] = np.arange(6)
    To = oracle_mod.get_transform_from_matches(x1, x2, m)
    assert abs(np.linalg.det(To[:3, :3].astype(np.float64)) - 1) < 1e-5
    assert np.abs(To[:3, 3] - T[:3, 3]).max() < 5e-3


def _error_function2_numpy(x1, x2, T, sigma, z0):
    """misc.cpp:697-770 restated with numpy float64 (np.linalg.solve instead of LLT)."""
    rcx = (3 * np.tan(58.0 / 180 * np.pi / 640)) ** 2
    rcy = (3 * np.tan(45.0 / 180 * np.pi / 480)) ** 2
    cz = lambda z: (sigma * (z0 if z0 > 0 else z) ** 2) ** 2
    a, b = x1.astype(np.float64), x2.astype(np.float64)
    mu = (T @ a)[:3]
    d = mu - b[:3]
    if d @ d > 2 * (max(rcx, cz(a[2])) + max(rcx, cz(b[2]))):
        return np.finfo(np.float64).max
    R = T[:3, :3]
    S = R.T @ np.diag([rcx * a[2], rcy * a[2], cz(a[2])]) @ R + np.diag([rcx * b[2], rcy * b[2], cz(b[2])])
    return float(d @ np.linalg.solve(S, d))


@pytest.mark.parametrize("z0", [2.0, -1.0])
def test_error_function2_against_numpy(oracle_mod, z0):
    from rgbdslam_v2_b200 import synth
    rng = np.random.default_rng(4)
    prm = oracle_mod.make_params(depth_cov_z0=z0)
    n_fin = 0
    for _ in range(200):
        T = synth.random_rigid(rng, 0.2, 10)
        p = synth._random_points(rng, 1)[0]
        q = T[:3, :3] @ p + T[:3, 3] + rng.normal(size=3) * rng.choice([1e-3, 2e-2, 0.2])
        x1 = np.array([*p, 1], np.float32)
        x2 = np.array([*q, 1], np.float32)
        Tf = T.astype(np.float32).astype(np.float64)
        got = oracle_mod.error_function2(prm, x1, x2, Tf)
        want = _error_function2_numpy(x1, x2, Tf, 0.01, z0)
        if want > 1e300:
            assert got > 1e300
        else:
            n_fin += 1
            assert abs(got - want) <= 1e-9 * max(1.0, abs(want))
    assert n_fin > 20
    nan = np.array([0, 0, np.nan, 1], np.float32)
    assert oracle_mod.error_function2(prm, nan, x2, Tf) > 1e300


def test_ransac_recovers_ground_truth(oracle_mod):
    from rgbdslam_v2_b200 import synth
    b = synth.make_batch(6, 800, seed0=40)
    prm = oracle_mod.make_params(depth_cov_z0=2.0)
    res, allm, inl = oracle_mod.match_pairs(prm, b["desc_newer"], b["xyz_newer"], b["n_newer"], b["desc_older"],
                                            b["xyz_older"], b["n_older"], b["id_newer"], b["id_older"], seed=3)
    ok = 0
    for i in range(6):
        if res[i]["id1"] < 0:
            continue
        ok += 1
        assert res[i]["id1"] == b["id_older"][i] and res[i]["id2"] == b["id_newer"][i]  # node.cpp:1337-1338
        T = res[i]["ransac_trafo"].reshape(4, 4).T
        assert np.abs(T[:3, 3] - b["T_true"][i][:3, 3]).max() < 5e-3
        assert np.abs(T[:3, :3] - b["T_true"][i][:3, :3]).max() < 5e-3
        n = res[i]["n_inliers"]
        assert res[i]["info_scale"] == pytest.approx(n / float(res[i]["rmse"]) ** 2, rel=1e-5)  # node.cpp:1335
        assert (np.diff(inl[i, :n]["distance"]) >= 0).all()  # inliers keep the sorted all_matches order
    assert ok >= 5


def test_too_few_matches_gives_invalid_edge(oracle_mod):
    """< min_matches correspondences -> edge ids -1,-1, rmse 0, identity trafo (node.cpp:1319,1420)."""
    rng = np.random.default_rng(0)
    d1 = rng.integers(0, 256, (10, 32), dtype=np.uint8)
    d2 = rng.integers(0, 256, (12, 32), dtype=np.uint8)
    x = np.ones((12, 4), np.float32)
    prm = oracle_mod.make_params(depth_cov_z0=2.0)
    res, allm, inl = oracle_mod.match_pairs(prm, d1, x[:10], [10], d2, x, [12], [5], [4], seed=1)
    assert res[0]["id1"] == -1 and res[0]["id2"] == -1 and res[0]["rmse"] == 0
    assert np.array_equal(res[0]["ransac_trafo"].reshape(4, 4), np.eye(4, dtype=np.float32))
    # empty nodes
    res, _, _ = oracle_mod.match_pairs(prm, d1[:0], x[:0], [0], d2[:0], x[:0], [0], seed=1)
    assert res[0]["id1"] == -1 and res[0]["n_all_matches"] == 0


def test_project_to_3d_and_remove_depthless(oracle_mod):
    """node.cpp:67-97, 900-965 + misc2.h:49-65: rounding lookup, NaN drop, sub-pixel back-projection."""
    import ctypes as C
    L = oracle_mod.lib()
    L.oracle_project_to_3d.restype = C.c_int
    w, h = 64, 48
    depth = np.full((h, w), 2.0, np.float32)
    depth[10, 20] = np.nan
    depth[11, 20] = 3.0
    xy = np.array([[20.4, 10.4], [20.4, 10.6], [63.6, 5.0], [-1.0, 3.0], [5.25, 7.75]], np.float32)
    keep = np.zeros(len(xy), np.uint8)
    xyz = np.zeros((len(xy), 4), np.float32)
    n = L.oracle_project_to_3d(xy.ctypes.data_as(C.c_void_p), C.c_int(len(xy)), depth.ctypes.data_as(C.c_void_p),
                               C.c_int(w), C.c_int(h), C.c_double(525.0), C.c_double(525.0), C.c_double(31.5),
                               C.c_double(23.5), C.c_double(1.0), C.c_int(600), xyz.ctypes.data_as(C.c_void_p),
                               keep.ctypes.data_as(C.c_void_p))
    # (20.4,10.4) -> depth[10,20] NaN dropped; (20.4,10.6) -> depth[11,20]=3; (63.6,5) rounds to col 64 = out of
    # the row (reads the next row's first pixel in the reference; x < cols so it is kept) ; (-1,3) dropped
    assert list(keep) == [0, 1, 1, 0, 1]
    assert n == 3
    fxinv = np.float32(1.0 / 525.0)
    assert xyz[0, 2] == 3.0 and xyz[0, 0] == (np.float32(20.4) - np.float32(31.5)) * np.float32(3.0) * fxinv
    assert xyz[2, 3] == 1.0
