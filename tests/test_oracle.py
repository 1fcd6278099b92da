"""CPU suite: the C oracle against its independent numpy restatement, against the committed golden
values on the reference's femur fixtures, and against analytic known answers (SURVEY.md 8c i-vii)."""
import struct

import numpy as np
import pytest

from conftest import random_theta
from icp_proposal_b200 import fixtures_io as fx, synth
from oracle import np_oracle as npo
from oracle import oracle as orc


def _objs(m):
    om = orc.Model(m["ref"], m["cells"], m["basis"], m["variance"])
    ot = orc.Mesh(m["target"], m["target_cells"])
    nm = npo.Model(m["ref"], m["cells"], m["basis"], m["variance"])
    return om, ot, nm


def test_closest_point_tree_equals_brute_force(twin31):
    mesh = orc.Mesh(twin31["target"], twin31["target_cells"])
    for q in (synth.near_surface_queries(twin31["target"], twin31["target_cells"], 1500),
              synth.far_field_queries(twin31["target"], 1500)):
        t1, f1, c1, d1 = mesh.closest_point(q, brute=True)
        t2, f2, c2, d2 = mesh.closest_point(q)
        assert np.array_equal(d1, d2) and np.array_equal(t1, t2) and np.array_equal(f1, f2)
        tn, cn, dn = npo.closest_point_on_triangles(q[:300], twin31["target"], twin31["target_cells"])
        np.testing.assert_allclose(dn, d1[:300], rtol=1e-12, atol=1e-18)
        np.testing.assert_allclose(cn, c1[:300], rtol=0, atol=1e-10)


def test_point_on_vertex_edge_face():
    a, b, c = np.array([0., 0, 0]), np.array([2., 0, 0]), np.array([0., 2, 0])
    for q, feat, cp in ((a + [-1, -1, 3], 0, a), ([1, -1, 0.5], 1, [1, 0, 0]), ([0.5, 0.5, 2], 2, [0.5, 0.5, 0]),
                        ([3, 3, 0], 1, [1, 1, 0]), ([5, -1, 0], 0, b)):
        d2, p, f = orc.point_triangle_d2(q, a, b, c)
        assert f == feat
        np.testing.assert_allclose(p, cp, atol=1e-15)
        np.testing.assert_allclose(d2, ((np.asarray(q, float) - cp) ** 2).sum(), rtol=1e-15)


def test_kdtree_boundary_normals(open_twin):
    mesh = orc.Mesh(open_twin["ref"], open_twin["cells"])
    q = synth.far_field_queries(open_twin["ref"], 500)
    i1, _ = mesh.closest_vertex(q, brute=True)
    i2, _ = mesh.closest_vertex(q)
    assert np.array_equal(i1, i2)
    assert np.array_equal(mesh.boundary_flags(), npo.boundary_flags(len(open_twin["ref"]), open_twin["cells"]))
    side = 33
    expect = np.zeros((side, side), bool); expect[0] = expect[-1] = True; expect[:, 0] = expect[:, -1] = True
    assert np.array_equal(mesh.boundary_flags(), expect.ravel())
    np.testing.assert_allclose(mesh.vertex_normals(), npo.vertex_normals(open_twin["ref"], open_twin["cells"]), atol=1e-12)


def test_surface_noise_matches_numpy_and_closed_form():
    rng = np.random.default_rng(0)
    for _ in range(20):
        n = rng.normal(size=3)
        c = orc.surface_noise_cov(n, 5.0, 10.0)
        np.testing.assert_allclose(c, npo.surface_noise_cov(n, 5.0, 10.0), atol=1e-12)
        u = n / np.linalg.norm(n)
        inv = np.outer(u, u) / 25.0 + (np.eye(3) - np.outer(u, u)) / 100.0
        np.testing.assert_allclose(np.linalg.inv(c), inv, atol=1e-12)
    # Appendix B2: the inverted fallback yields NaN for n = +-e_y
    assert np.isnan(orc.surface_noise_cov([0, 1.0, 0], 5.0, 10.0)).any()


@pytest.mark.parametrize("direction", [0, 1])
def test_posterior_propose_transition_vs_numpy(twin31, direction):
    om, ot, nm = _objs(twin31)
    K = 31
    rng = np.random.default_rng(5)
    theta = random_theta(twin31, rng, 1, pose=True)[0]
    ids = np.arange(2 * K)
    tp = twin31["target"][rng.choice(len(twin31["target"]), 2 * K, replace=False)] + rng.normal(0, 0.2, (2 * K, 3))
    p = orc.IcpProposal(om, ot, 0.1, 10.0, 5.0, direction, True, ids, tp)
    po = p.posterior(theta, with_obs=True)
    obs = npo.icp_observations(nm, twin31["target"], twin31["target_cells"], theta, direction, True, ids, tp, 10.0, 5.0)
    pn = npo.icp_posterior(nm, obs)
    assert po["n"] == len(obs) and np.array_equal(po["ids"], [o[0] for o in obs])
    np.testing.assert_allclose(po["mu"], pn["mu"], rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(po["M"], pn["M"], rtol=1e-11)
    np.testing.assert_allclose(po["Minv"], pn["Minv"], rtol=1e-8, atol=1e-14)
    z0 = np.zeros(K)
    np.testing.assert_allclose(p.propose(theta, z0), npo.propose(nm, pn, theta, z0, 0.1), rtol=0, atol=1e-11)
    z = rng.normal(size=K)
    to = p.propose(theta, z)
    # with the shared sign rule of the singular vectors the two independent restatements (tred2/tql2 vs LAPACK gesdd) draw
    # the same sample for the same z
    np.testing.assert_allclose(to, npo.propose(nm, pn, theta, z, 0.1), rtol=0, atol=1e-9)
    lt = p.log_transition(theta, to)
    np.testing.assert_allclose(lt, npo.log_transition(nm, pn, theta, to, 0.1), rtol=1e-10)
    # Appendix A6/A7: the sample drawn with z has transition density N(z; 0, I) up to the 1e-5 regulariser
    np.testing.assert_allclose(lt, -0.5 * (K * np.log(2 * np.pi) + z @ z), rtol=1e-6)
    # closed forms (what the device computes) agree with the reference structure within the stated tolerance
    np.testing.assert_allclose(p.log_transition(theta, to, closed_form=True), lt, rtol=1e-6)
    np.testing.assert_allclose(p.propose(theta, z0, closed_form=True), p.propose(theta, z0), rtol=0, atol=1e-9)
    # guard: anything but alpha differs -> -inf (NonRigidIcpProposal.scala:72-74)
    bad = to.copy(); bad[1] += 1e-3
    assert p.log_transition(theta, bad) == -np.inf


def test_propose_covariance_factor(twin31):
    """W W^T = M^-1 for the closed-form factor (Cholesky) and for the reference's SVD factor."""
    om, ot, _ = _objs(twin31)
    K = 31
    theta = random_theta(twin31, np.random.default_rng(1), 1)[0]
    p = orc.IcpProposal(om, ot, 1.0, 10.0, 5.0, 0, True, np.arange(62), np.zeros((0, 3)))
    post = p.posterior(theta)
    base = {cf: p.propose(theta, np.zeros(K), closed_form=cf)[10:] for cf in (False, True)}
    for cf in (False, True):
        W = np.stack([p.propose(theta, np.eye(K)[i], closed_form=cf)[10:] - base[cf] for i in range(K)], axis=1)
        np.testing.assert_allclose(W @ W.T, post["Minv"], rtol=1e-5, atol=1e-9)


def test_evaluators_vs_numpy(twin31):
    om, ot, nm = _objs(twin31)
    rng = np.random.default_rng(2)
    theta = random_theta(twin31, rng, 1, pose=True)[0]
    ids = np.arange(124)
    tp = twin31["target"][::13][:124]
    for mode in (0, 1, 2):
        a = orc.eval_independent(om, ot, mode, 0.0, 2.0, ids, tp, theta)
        b = npo.eval_independent(nm, twin31["target"], twin31["target_cells"], mode, 0.0, 2.0, ids, tp, theta)
        np.testing.assert_allclose(a, b, rtol=1e-12)
    np.testing.assert_allclose(orc.eval_hausdorff(om, ot, 100.0, theta),
                               npo.eval_hausdorff(nm, twin31["target"], twin31["target_cells"], 100.0, theta), rtol=1e-12)
    np.testing.assert_allclose(orc.eval_prior(31, theta), -0.5 * (31 * np.log(2 * np.pi) + theta[10:] @ theta[10:]), rtol=1e-14)


def test_collective_boundary_and_empty_set(open_twin):
    om = orc.Model(open_twin["ref"], open_twin["cells"], open_twin["basis"], open_twin["variance"])
    ot = orc.Mesh(open_twin["target"], open_twin["target_cells"])
    K = 21
    theta = random_theta(open_twin, np.random.default_rng(3), 1)[0]
    ids = np.arange(0, len(open_twin["ref"]), 7)
    tp = open_twin["target"][::9]
    v, st, am = orc.eval_collective(om, ot, 2, 0.1, 0.3, 1.0, ids, tp, theta)
    assert st == 0 and np.isfinite(v) and am[1] >= am[0] > 0
    # only boundary hits -> empty filtered list (the reference throws, CollectiveAverage...:51)
    corner = np.array([0])
    v, st, _ = orc.eval_collective(om, ot, 0, 0.1, 0.3, 1.0, corner, tp, theta)
    assert st == 1


def test_posterior_mean_is_least_squares_as_sigma_to_zero(twin31):
    """SURVEY 8c (iii): model.posterior(corr, 1e-15).mean == least squares on the correspondences."""
    om, ot, nm = _objs(twin31)
    K = 31
    alpha = np.random.default_rng(4).normal(0, 0.3, K)
    ids = np.arange(0, 1622, 3)
    out = orc.std_icp_iteration(om, ot, 0, ids, np.zeros((0, 3)), 1e-15, 1.0, alpha)
    theta = np.zeros(K + 10); theta[0] = 1; theta[10:] = alpha
    cur = nm.transformed_mesh(theta)
    _, cp, _ = npo.closest_point_on_triangles(cur[ids], twin31["target"], twin31["target_cells"])
    rows = (3 * ids[:, None] + np.arange(3)).ravel()
    ls = np.linalg.lstsq(nm.Q[rows], (cp - nm.ref[ids]).ravel(), rcond=None)[0]
    np.testing.assert_allclose(out, ls, rtol=1e-5, atol=1e-7)


def test_S_is_identity_to_regulariser(femur):
    """SURVEY 8c (vi): coefficients(instance(alpha)) = S alpha with |S - I| ~ 1e-5 / lambda_min(G)."""
    g = femur["gpmm_100"]
    q = g["basis"] * np.sqrt(g["variance"])
    G = q.T @ q
    S = np.linalg.solve(G / 1e-5 + np.eye(len(G)), G / 1e-5)
    assert 1e-8 < np.abs(S - np.eye(len(G))).max() < 1e-6


def test_fp32_reconstruction_error_exceeds_budget(femur):
    """SURVEY 8c (vii): FP32 reconstruction error vs the 1e-5-relative budget on ~1 mm distances."""
    g = femur["gpmm_100"]
    q = g["basis"] * np.sqrt(g["variance"])
    alpha = np.random.default_rng(0).normal(0, 1, len(g["variance"]))
    x64 = femur["ref"].ravel() + q @ alpha
    x32 = (femur["ref"].ravel().astype(np.float32) + q.astype(np.float32) @ alpha.astype(np.float32)).astype(np.float64)
    err = np.abs(x64 - x32).max()
    assert 1e-6 < err < 1e-4   # of the order of 1e-5 mm: FP32 coordinates cannot carry 1e-5 relative on 1 mm


def test_golden_femur_values(femur):
    """The oracle reproduces the committed golden values on the reference's femur fixtures."""
    for key, gk in (("gpmm_50", "gpmm_50"), ("gpmm_100", "gpmm_100"), ("gpmm_200", "gpmm_200")):
        g = femur["golden"][gk]
        m = femur[key]
        K = len(m["variance"])
        om = orc.Model(femur["ref"], femur["cells"], m["basis"], m["variance"])
        ot = orc.Mesh(femur["target"], femur["target_cells"])
        theta = np.array(g["theta"])
        ids = np.arange(g["n_icp"]); eids = np.arange(g["n_eval"])
        tp = femur["target"][:: max(1, len(femur["target"]) // (2 * K))][: 2 * K]
        xyz = om.transformed_mesh(theta)
        np.testing.assert_allclose([xyz.sum(), np.abs(xyz).sum()], g["mesh_checksum"], rtol=1e-12)
        for direction, name in ((0, "model_sampling"), (1, "target_sampling")):
            p = orc.IcpProposal(om, ot, 0.1, 10.0, 5.0, direction, True, ids, tp)
            post = p.posterior(theta)
            assert post["n"] == g[name]["n_obs"]
            np.testing.assert_allclose(post["mu"], g[name]["mu"], rtol=1e-8, atol=1e-11)
            np.testing.assert_allclose(np.diag(post["M"]), g[name]["M_diag"], rtol=1e-11)
            if key == "gpmm_50":  # the reference-structure propose/transition are the slow part: K = 51 only
                to = p.propose(theta, np.zeros(K))
                np.testing.assert_allclose(to[10:], g[name]["propose_z0"], rtol=1e-7, atol=1e-10)
                np.testing.assert_allclose(p.log_transition(theta, to), g[name]["log_transition_to_z0"], rtol=1e-9)
        np.testing.assert_allclose(orc.eval_independent(om, ot, 0, 0.0, 2.0, eids, tp, theta), g["independent_m2t"], rtol=1e-11)
        np.testing.assert_allclose(orc.eval_independent(om, ot, 2, 0.0, 2.0, eids, tp, theta), g["independent_sym"], rtol=1e-11)
        np.testing.assert_allclose(orc.eval_hausdorff(om, ot, 100.0, theta), g["hausdorff"], rtol=1e-11)
        np.testing.assert_allclose(orc.eval_prior(K, theta), g["prior"], rtol=1e-13)


def test_femur_target_is_explained_by_the_model(femur):
    """SURVEY 8c: after landmark alignment the 101-component model explains the target to sub-mm."""
    g = femur["gpmm_100"]
    q = g["basis"] * np.sqrt(g["variance"])
    alpha = np.linalg.lstsq(q, (femur["target"] - femur["ref"]).ravel(), rcond=None)[0]
    res = np.linalg.norm((femur["ref"].ravel() + q @ alpha).reshape(-1, 3) - femur["target"], axis=1)
    assert res.mean() < 0.5 and res.max() < 2.0


def _binary_stl(verts, tris):
    """Binary STL of a triangle mesh: one float32 facet per triangle (corners in the triangle's vertex order, the facet
    normal, a running attribute word)."""
    rec = np.zeros(len(tris), dtype=[("n", "<f4", 3), ("v", "<f4", (3, 3)), ("a", "<u2")])
    rec["v"] = verts[tris]
    rec["n"] = np.cross(rec["v"][:, 1] - rec["v"][:, 0], rec["v"][:, 2] - rec["v"][:, 0])
    rec["a"] = np.arange(len(tris)) & 0xFFFF
    return b"binary STL".ljust(80) + struct.pack("<I", len(tris)) + rec.tobytes()


def _hdf5_file(tree):
    """An HDF5 file holding `tree`: name -> ndarray, bytes (a fixed-length string) or dict (a group, whose '@name' keys are
    string attributes). It uses the constructs of the file format the statismo model files are written in: superblock v0,
    v1 object headers (the layout message of every dataset in a continuation block), symbol-table groups with B-trees of
    one and of two levels, scalar datasets, and both the v1 and the v3 contiguous-layout message."""
    undef = 0xFFFFFFFFFFFFFFFF
    buf = bytearray(96)                                   # superblock + root symbol-table entry, written last

    def put(b):
        addr = len(buf)
        buf.extend(b + bytes(-len(b) % 8))
        return addr

    def messages(msgs):
        return b"".join(struct.pack("<HHB3x", t, len(m) + -len(m) % 8, 0) + m + bytes(-len(m) % 8) for t, m in msgs)

    def object_header(msgs, continued=()):
        if continued:
            more = messages(continued)
            msgs = msgs + [(0x10, struct.pack("<QQ", put(more), len(more)))]
        body = messages(msgs)
        return put(struct.pack("<BBHII4x", 1, 0, len(msgs) + len(continued), 1, len(body)) + body)

    def space(shape):
        return struct.pack("<BBB5x", 1, len(shape), 0) + struct.pack(f"<{len(shape)}Q", *shape)

    def string_type(n):
        return struct.pack("<BBxxI", 0x13, 0, n)

    def attribute(name, value):
        parts = [name.encode() + b"\0", string_type(len(value)), space(())]
        return struct.pack("<BxHHH", 1, *map(len, parts)) + b"".join(p + bytes(-len(p) % 8) for p in parts) + value

    def dataset(a):
        if isinstance(a, bytes):
            layout = struct.pack("<BBQQ", 3, 1, put(a), len(a))
            return object_header([(0x1, space(())), (0x3, string_type(len(a)))], [(0x8, layout)])
        a = np.ascontiguousarray(a)
        addr, bits = put(a.tobytes()), 8 * a.itemsize
        if a.dtype.kind == "f":
            exp, mant = {4: (8, 23), 8: (11, 52)}[a.itemsize]
            dtype = struct.pack("<BBBxIHHBBBBI", 0x11, 0x20, bits - 1, a.itemsize, 0, bits, mant, exp, 0, mant, 2 ** (exp - 1) - 1)
            layout = struct.pack("<BBQQ", 3, 1, addr, a.nbytes)
        else:
            dtype = struct.pack("<BBxxIHH", 0x10, 0x08 if a.dtype.kind == "i" else 0, a.itemsize, 0, bits)
            layout = struct.pack("<BBB5xQ", 1, a.ndim + 1, 1, addr) + struct.pack(f"<{a.ndim + 1}I", *a.shape, a.itemsize)
        return object_header([(0x1, space(a.shape)), (0x3, dtype)], [(0x8, layout)])

    def group(children):
        heap, entries = bytearray(8), []                  # heap offset 0: the empty name
        for name in sorted(k for k in children if not k.startswith("@")):
            child = children[name]
            entries.append((len(heap), group(child) if isinstance(child, dict) else dataset(child)))
            heap += name.encode() + bytes(8 - len(name) % 8)
        local_heap = put(b"HEAP" + struct.pack("<B3xQQQ", 0, len(heap), undef, put(bytes(heap))))

        def leaf(es):
            snod = put(b"SNOD" + struct.pack("<BxH", 1, len(es)) + b"".join(struct.pack("<QQII16x", o, a, 0, 0) for o, a in es))
            return put(b"TREE" + struct.pack("<BBHQQQQQ", 0, 0, 1, undef, undef, 0, snod, es[-1][0]))
        btree = leaf(entries)
        if len(entries) > 2:                              # a level-1 node over two leaves
            h = len(entries) // 2
            btree = put(b"TREE" + struct.pack("<BBHQQ5Q", 0, 1, 2, undef, undef, 0, leaf(entries[:h]), entries[h - 1][0],
                                              leaf(entries[h:]), entries[-1][0]))
        attrs = [(0xC, attribute(k[1:], v)) for k, v in children.items() if k.startswith("@")]
        return object_header([(0x11, struct.pack("<QQ", btree, local_heap))] + attrs)

    root = group(tree)
    struct.pack_into("<8s8BHHIQQQQ", buf, 0, b"\x89HDF\r\n\x1a\n", 0, 0, 0, 0, 0, 8, 8, 0, 4, 16, 0, 0, undef, len(buf), undef)
    struct.pack_into("<QQII16x", buf, 56, 0, root, 0, 0)
    return bytes(buf)


def test_fixture_readers_round_trip(femur, tmp_path):
    """fixtures_io on files this test writes in the formats of the reference's data files (those files are not part of the
    repository): a statismo model file holding the committed GPMM-100 fixture, and binary STLs of the femur mesh with the
    facets in cell order and shuffled. The readers return the arrays written, pass over what they do not use (attributes,
    string datasets) and merge STL corners into vertices in the order of first appearance."""
    ref32, cells = femur["ref"].astype(np.float32), femur["cells"]
    basis32, var32 = femur["gpmm_100"]["basis"].astype(np.float32), femur["gpmm_100"]["variance"].astype(np.float32)
    path = str(tmp_path / "model.h5")
    with open(path, "wb") as f:
        f.write(_hdf5_file({
            "@name": b"femur",
            "version": {"majorVersion": np.array(0, np.int32), "minorVersion": np.array(9, np.int32)},
            "modelinfo": {"build-time": b"2020-01-01 00:00:00"},
            "representer": {"@datasetType": b"POLYGON_MESH", "points": np.ascontiguousarray(ref32.T), "cells": np.ascontiguousarray(cells.T)},
            "model": {"mean": ref32.ravel(), "noiseVariance": np.array(0.0, np.float32), "pcaBasis": basis32, "pcaVariance": var32}}))
    found = fx.read_hdf5_datasets(path)
    assert sorted(found) == ["/model/mean", "/model/noiseVariance", "/model/pcaBasis", "/model/pcaVariance", "/representer/cells",
                             "/representer/points", "/version/majorVersion", "/version/minorVersion"]
    assert found["/version/minorVersion"] == 9 and found["/model/noiseVariance"] == 0.0
    m = fx.load_gpmm_h5(path)
    assert m["basis"].shape == (4866, 101) and np.abs(m["mean_def"]).max() == 0.0
    assert np.array_equal(m["basis"], basis32) and np.array_equal(m["variance"], var32)
    assert np.array_equal(m["ref"], ref32) and np.array_equal(m["cells"], cells)
    with open(tmp_path / "mesh.stl", "wb") as f:
        f.write(_binary_stl(ref32, cells))
    v, c = fx.read_binary_stl(str(tmp_path / "mesh.stl"))
    assert np.array_equal(v, m["ref"]) and np.array_equal(c, m["cells"])
    shuffled = cells[np.random.default_rng(0).permutation(len(cells))][:, [1, 2, 0]]
    with open(tmp_path / "shuffled.stl", "wb") as f:
        f.write(_binary_stl(ref32, shuffled))
    v, c = fx.read_binary_stl(str(tmp_path / "shuffled.stl"))
    corners = shuffled.ravel()
    assert np.array_equal(v, ref32[corners[np.sort(np.unique(corners, return_index=True)[1])]])
    assert np.array_equal(v[c], ref32[shuffled])


def test_chain_oracle_closed_form_tracks_reference_structure(twin31):
    """The MH chain through the closed forms accepts/rejects like the chain in the reference's structure."""
    om, ot, _ = _objs(twin31)
    K = 31
    rng = np.random.default_rng(11)
    ids, eids = np.arange(62), np.arange(124)
    tp = twin31["target"][::26][:62]
    pm = orc.IcpProposal(om, ot, 0.1, 10.0, 5.0, 0, True, ids, tp)
    pt = orc.IcpProposal(om, ot, 0.1, 10.0, 5.0, 1, True, ids, tp)
    comps = [dict(kind=orc.PROP_ICP, weight=0.45, icp=pt), dict(kind=orc.PROP_ICP, weight=0.45, icp=pm),
             dict(kind=orc.PROP_RANDOM_SHAPE, weight=0.1, sd=0.1)]
    n = 12
    theta0 = random_theta(twin31, rng, 1)[0]
    u_comp = rng.random(n); u_acc = rng.random(n)
    # z = 0: both factorizations give the same proposal, so the two chains see identical states
    z = np.zeros((n, K))
    a = orc.chain_run(om, ot, comps, True, orc.EVAL_INDEPENDENT, 0, (0.0, 2.0), eids, tp, theta0, n, u_comp, z, u_acc, closed_form=False)
    b = orc.chain_run(om, ot, comps, True, orc.EVAL_INDEPENDENT, 0, (0.0, 2.0), eids, tp, theta0, n, u_comp, z, u_acc, closed_form=True)
    assert np.array_equal(a["comp"], b["comp"]) and np.array_equal(a["accepted"], b["accepted"])
    np.testing.assert_allclose(a["logv"], b["logv"], rtol=1e-6)
    np.testing.assert_allclose(a["theta"], b["theta"], rtol=0, atol=1e-6)
    assert a["accepted"].any()


def test_philox_known_answer():
    """Philox4x32-10 known-answer vectors (Random123 kat_vectors)."""
    assert orc.philox4x32_10([0, 0, 0, 0], [0, 0]).tolist() == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    assert orc.philox4x32_10([0xffffffff] * 4, [0xffffffff] * 2).tolist() == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    assert orc.philox4x32_10([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0]).tolist() == \
        [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]


def test_posterior_variability_oracle_against_closed_forms(twin31):
    """The loop-for-loop restatement of PosteriorVariability.scala against vectorised sample statistics, a known
    answer (rigidly translated copies: all variance along the translation), and LogHelper's index walk."""
    m = twin31
    om = npo.Model(m["ref"], m["cells"], m["basis"], m["variance"])
    rng = np.random.default_rng(3)
    thetas = np.zeros((9, 10 + om.K)); thetas[:, 0] = 1.0
    thetas[:, 10:] = rng.normal(0, 0.5, (9, om.K))
    X = np.stack([om.transformed_mesh(t) for t in thetas])
    mean, cov, total, along = npo.posterior_variability(list(X), m["cells"], sum_normals=True)
    np.testing.assert_allclose(mean, X.mean(0), rtol=1e-13)
    np.testing.assert_allclose(total, X.var(0, ddof=1).sum(1), rtol=1e-12)
    d = X - X.mean(0)
    np.testing.assert_allclose(cov, np.einsum("sni,snj->nij", d, d) / 8, rtol=1e-12, atol=1e-14)
    nbar = np.stack([npo.vertex_normals(x, m["cells"]) for x in X]).mean(0)
    np.testing.assert_allclose(along, (np.einsum("ni,sni->sn", nbar, d) ** 2).sum(0) / 8, rtol=1e-12)
    assert (along <= total * (1 + 1e-12)).all()           # |n| <= 1: the normal part never exceeds the trace
    # known answer: copies translated along e_z by 0, 1, 2 -> cov = diag(0, 0, 1), normal variance = n_z^2
    shifted = [m["ref"] + np.array([0, 0, k], float) for k in range(3)]
    mean, cov, total, along = npo.posterior_variability(shifted, m["cells"], ref_verts=m["ref"], sum_normals=False)
    np.testing.assert_allclose(total, 1.0, rtol=1e-12)
    np.testing.assert_allclose(along, npo.vertex_normals(m["ref"], m["cells"])[:, 2] ** 2, rtol=1e-12, atol=1e-15)
    # a single sample: 0 * (1 / 0) = NaN, as on the JVM
    assert np.isnan(npo.posterior_variability(shifted[:1], m["cells"], sum_normals=True)[2]).all()
    # LogHelper.samplesFromLog
    status = [True, False, False, True, False, True, True, False, False, True]
    assert npo.samples_from_log(status, take_every_n=2, total=7, burn_in=1) == [0, 3, 5]
    assert npo.samples_from_log(status, take_every_n=3, total=100, burn_in=0) == [0, 3, 6, 9]
    assert npo.samples_from_log(status, take_every_n=1, total=3, burn_in=0) == [0, 0, 0]
    with pytest.raises(IndexError):
        npo.samples_from_log([False, True], 1, 2, 0)


def test_nystrom_oracle_reproduces_the_kernel_on_the_nystrom_points():
    """The pair-by-pair kernel restatement against a vectorised evaluation, and the defining property of the Nystrom
    extension: with all 3m eigenpairs, basis diag(variance) basis^T restricted to the Nystrom points is their kernel matrix."""
    rng = np.random.default_rng(5)
    pts = rng.normal(0, 30, (40, 3))
    a = rng.normal(size=(3, 3)); a = a @ a.T
    terms = [(10.0, 90.0, a), (5.0, 40.0, None), (3.0, 10.0, None)]
    nys = pts[:12]
    k = npo.gauss_mixture_kernel(pts, nys, terms)
    d2 = ((pts[:, None] - nys[None]) ** 2).sum(-1)
    want = sum(s * np.exp(-d2 / sg ** 2)[:, None, :, None] * (np.eye(3) if m is None else m)[None, :, None, :] for s, sg, m in terms)
    np.testing.assert_allclose(k, want.reshape(120, 36), rtol=1e-14, atol=1e-300)
    kmm = npo.gauss_mixture_kernel(nys, nys, terms)
    w, v = np.linalg.eigh(kmm)
    assert w.min() > 0
    basis, var = npo.nystrom_extend(k, v, w)
    q = basis * np.sqrt(var)
    np.testing.assert_allclose((q @ q.T)[:36, :36], kmm, rtol=1e-9, atol=1e-9)
    # orthonormality of the discretised eigenfunctions on the Nystrom points: (1/m) sum_x phi_i(x) phi_j(x) = delta_ij
    np.testing.assert_allclose(basis[:36].T @ basis[:36] / 12, np.eye(36), atol=1e-7)


def test_golden_variability_and_femur_kernel(femur):
    """The oracle restatements of the SURVEY 8f rows reproduce their committed golden values on the reference's femur
    fixtures (tests/golden/make_golden.py)."""
    g = femur["golden"]["variability_gpmm_50"]
    m = femur["gpmm_50"]
    om = orc.Model(femur["ref"], femur["cells"], m["basis"], m["variance"])
    meshes = [om.transformed_mesh(np.array(t)) for t in g["thetas"]]
    mean, cov, total, along = npo.posterior_variability(meshes, femur["cells"], sum_normals=True)
    np.testing.assert_allclose([mean.sum(), np.abs(mean).sum()], g["mean_checksum"], rtol=1e-12)
    np.testing.assert_allclose(total[:8], g["total_first8"], rtol=1e-9)
    np.testing.assert_allclose(along[:8], g["normal_first8"], rtol=1e-9)
    np.testing.assert_allclose([total.sum(), along.sum()], [g["total_sum"], g["normal_sum"]], rtol=1e-9)
    k = femur["golden"]["femur_kernel"]
    base = np.array(k["base_matrix"])
    terms = [(10.0, 90.0, base), (5.0, 40.0, None), (3.0, 10.0, None)]
    kk = npo.gauss_mixture_kernel(femur["ref"][:12], femur["ref"][:12], terms)
    np.testing.assert_allclose([kk.sum(), np.abs(kk).sum()], k["k_checksum"], rtol=1e-12)
    np.testing.assert_allclose(kk[0, :9], k["k_row0_first9"], rtol=1e-12)
    np.testing.assert_allclose(np.linalg.eigvalsh(kk)[::-1][:6], k["eigenvalues_first6"], rtol=1e-9)
    # the host mirror builds the same base matrix from the reference points (up to the sign-free product d diag d^T)
    from icp_proposal_b200 import api
    np.testing.assert_allclose(api.femurKernel(femur["ref"]).terms[0][2], base, rtol=1e-9, atol=1e-12)


def test_face_kernel_oracle_known_answers():
    """apps/bfm/FaceKernel.scala restated (np_oracle.face_kernel): analytic known answers of the order-3 B-spline kernel, the
    symmetrisation about x = 0 and positive semi-definiteness of the resulting kernel matrix."""
    from oracle import np_oracle as npo
    rng = np.random.default_rng(5)
    # the cardinal cubic B-spline: partition of unity, unit integral, known values
    assert npo.bspline3(0.0) == pytest.approx(2.0 / 3.0) and npo.bspline3(1.0) == pytest.approx(1.0 / 6.0) and npo.bspline3(2.0) == 0.0
    for t in rng.uniform(-3, 3, 20):
        assert sum(npo.bspline3(t - k) for k in range(-6, 7)) == pytest.approx(1.0, abs=1e-14)
    # the lattice-sum kernel is symmetric, shift invariant by integers and vanishes beyond the joint support (|a - b| >= 4)
    a, b = rng.uniform(-5, 5, 3), rng.uniform(-5, 5, 3)
    assert npo.bspline_kernel3d(a, b) == pytest.approx(npo.bspline_kernel3d(b, a), rel=1e-14)
    assert npo.bspline_kernel3d(a + 3.0, b + 3.0) == pytest.approx(npo.bspline_kernel3d(a, b), rel=1e-12)
    assert npo.bspline_kernel3d(a, a + np.array([4.0, 0.0, 0.0])) == 0.0
    # 1-D closed form at lattice points: sum_k beta(0 - k) beta(0 - k) = (2/3)^2 + 2 (1/6)^2
    one_d = (2.0 / 3.0) ** 2 + 2.0 / 36.0
    assert npo.bspline_kernel3d(np.zeros(3), np.zeros(3)) == pytest.approx(one_d ** 3, rel=1e-14)
    # symmetrised kernel: mirrored point pairs are perfectly (anti-)correlated per axis: k_face(x, xbar) = diag(-1, 1, 1) k_face(x, x)
    levels, scales = [-6, -5, -4, -3, -2], [128.0, 64.0, 32.0, 10.0, 4.0]
    x = rng.uniform(-80, 80, (6, 3))
    xbar = x * np.array([-1.0, 1.0, 1.0])
    kxx = npo.face_kernel(x, x, levels, scales, 1.0, 0.0)
    kxb = npo.face_kernel(x, xbar, levels, scales, 1.0, 0.0)
    for i in range(len(x)):
        np.testing.assert_allclose(kxb[3 * i:3 * i + 3, 3 * i:3 * i + 3], np.diag([-1.0, 1.0, 1.0]) @ kxx[3 * i:3 * i + 3, 3 * i:3 * i + 3], rtol=1e-12)
    # the face kernel (0.7 symmetric + 0.3 plain) with region weights is a symmetric positive semi-definite matrix
    pts = rng.uniform(-60, 60, (14, 3))
    w = rng.uniform(0.2, 1.0, (5, 14))
    wm = rng.uniform(0.2, 1.0, (5, 14))
    plain = npo.face_kernel(pts, pts, levels, scales, 0.0, 1.0, w, w, None)
    np.testing.assert_allclose(plain, plain.T, rtol=1e-13)
    assert np.linalg.eigvalsh(plain).min() > -1e-9 * np.abs(plain).max()
    # with mirror-consistent weights (w(ybar) = w(y)) the symmetrised kernel is symmetric PSD too
    full = npo.face_kernel(pts, pts, levels, scales, 0.7, 0.3, w, w, w)
    np.testing.assert_allclose(full, full.T, rtol=1e-12, atol=1e-12)
    assert np.linalg.eigvalsh(full).min() > -1e-9 * np.abs(full).max()
    assert np.abs(npo.face_kernel(pts, pts, levels, scales, 0.7, 0.3, w, w, wm) - full).max() > 0     # the mirrored weights matter
