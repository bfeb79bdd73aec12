"""CPU: host-side pieces of the T-LESS / VSD evaluation -- PLY reader, the ray-cast oracle against the
reference vsd_obj's stored errors, the score formulas of model.py:530-537, the batch adapter and the
tless_<cat> routing of test_step."""
import os

import numpy as np
import pytest
import torch


def _quad_cube():
    v = np.array([[x, y, z] for x in (0, 1) for y in (0, 1) for z in (0, 1)], dtype=np.float64) * 1.25 + 1 / 3
    q = [(0, 1, 3, 2), (4, 6, 7, 5), (0, 4, 5, 1), (2, 3, 7, 6), (0, 2, 6, 4), (1, 5, 7, 3)]
    return v, q


def _fan(q):
    return np.array([(p[0], p[i], p[i + 1]) for p in q for i in range(1, len(p) - 1)])


def test_read_ply_ascii_and_binary_round_trip(tmp_path):
    from nope_b200.vsd import read_ply
    v, q = _quad_cube()
    # ascii, double vertices, an extra property and an extra element
    with open(tmp_path / "a.ply", "w") as f:
        f.write(f"ply\nformat ascii 1.0\ncomment t\nelement vertex {len(v)}\nproperty double x\nproperty double y\n"
                f"property double z\nproperty uchar red\nelement face {len(q)}\nproperty list uchar int vertex_indices\n"
                "element edge 1\nproperty int a\nproperty int b\nend_header\n")
        for r in v:
            f.write(" ".join(repr(float(c)) for c in r) + " 7\n")
        for p in q:
            f.write(f"{len(p)} " + " ".join(map(str, p)) + "\n")
        f.write("0 1\n")
    va, fa = read_ply(tmp_path / "a.ply")
    assert np.array_equal(va, v) and np.array_equal(fa, _fan(q))
    # binary little endian: float vertices with a trailing normal, uint indices with an int count, one triangle
    tris = [(0, 1, 3)]
    with open(tmp_path / "b.ply", "wb") as f:
        f.write(f"ply\nformat binary_little_endian 1.0\nelement vertex {len(v)}\nproperty float x\nproperty float y\n"
                f"property float z\nproperty float nx\nelement face {len(q) + 1}\n"
                "property list int uint vertex_indices\nend_header\n".encode())
        for r in v:
            f.write(np.array(list(r) + [0.5], dtype="<f4").tobytes())
        for p in list(q) + tris:
            f.write(np.array([len(p)], "<i4").tobytes() + np.array(p, "<u4").tobytes())
    vb, fb = read_ply(tmp_path / "b.ply")
    assert np.array_equal(vb, v.astype(np.float32).astype(np.float64))
    assert np.array_equal(fb, np.concatenate([_fan(q), tris]))


def test_raycaster_plane_depth_and_cube_silhouette():
    from oracle.vsd_oracle import box, pose44, raycast_depth
    K = np.array([[100.0, 0, 32.0], [0, 100.0, 24.0], [0, 0, 1]])
    plane_v = np.array([[-1e3, -1e3, 0], [1e3, -1e3, 0], [1e3, 1e3, 0], [-1e3, 1e3, 0]], np.float32)
    plane_f = np.array([[0, 1, 2], [0, 2, 3]])
    d, _ = raycast_depth(plane_v, plane_f, pose44(np.eye(3), [0, 0, 500.0]), K, 48, 64)
    assert np.all(d == 500.0)
    # an axis-aligned cube face at z = 480 spanning x, y in [-20, 20]: pixel (x, y) is covered iff its sample
    # (x + 0.5, y + 0.5) projects inside [32 - 100*20/480, 32 + 100*20/480] (and the same in y)
    bv, bf = box(half=(20.0, 20.0, 20.0))
    d, amb = raycast_depth(bv, bf, pose44(np.eye(3), [0, 0, 500.0]), K, 48, 64)
    xs, ys = np.meshgrid(np.arange(64) + 0.5, np.arange(48) + 0.5)
    h = 100 * 20 / 480
    inside = (np.abs(xs - 32) < h) & (np.abs(ys - 24) < h)
    assert np.array_equal(d > 0, inside) and np.all(d[inside] == 480.0)
    # the only samples within 1e-3 px of a projected edge lie on the front face's diagonals (x - y = 8 or
    # x + y = 55 with a sample exactly on them)
    ys_, xs_ = np.nonzero(amb)
    assert amb.any() and np.all((xs_ - ys_ == 8) | (xs_ + ys_ == 55))


def test_oracle_vsd_matches_reference_vsd_obj_on_fixture(golden_dir):
    """The fixture's errors come from the unmodified reference vsd_obj (renderer swapped for the ray
    caster); the restated arithmetic must reproduce them exactly, and the ray caster its depths."""
    from oracle.vsd_oracle import error_from_counts, raycast_depth, vsd_counts
    g = np.load(os.path.join(golden_dir, "vsd_fixture.npz"))
    F, k = g["err_reference"].shape
    assert (F, k) == (2, 5) and (g["err_reference"] == 0).any() and (g["err_reference"] == 1).any()
    for f in range(F):
        d, a = raycast_depth(g["verts"], g["faces"], g["gt_poses"][f], g["K"], 120, 160)
        assert np.array_equal(d.astype(np.float32), g["depth_gt"][f]) and np.array_equal(a, g["amb_gt"][f])
        for j in range(k):
            c = vsd_counts(g["depth_raw"][f] / 10.0, g["K"], g["depth_gt"][f], g["depth_est"][f, j])
            assert c == tuple(g["counts"][f, j])
            assert error_from_counts(c) == g["err_reference"][f, j]
    # the fixture exercises bop19's d_test == 0 branch
    assert (g["depth_raw"] == 0).any()


def test_vsd_scores_formulas():
    from nope_b200.vsd import vsd_scores
    err = np.array([[0.5, 0.2, 0.9, 0.1, 0.4], [0.1, 0.8, 0.8, 0.8, 0.8], [1.0, 1.0, 0.31, 0.3, 1.0],
                    [0.35, 0.36, 0.37, 0.38, 0.29]])
    s = vsd_scores(torch.from_numpy(err))
    assert set(s) == {f"top {k}, {n}" for k in (1, 3, 5) for n in ("vsd_median", "vsd_scores 0.3")}
    assert s["top 1, vsd_median"] == np.median([0.5, 0.1, 1.0, 0.35])
    assert s["top 1, vsd_scores 0.3"] == 25.0
    assert s["top 3, vsd_median"] == np.median([0.2, 0.1, 0.31, 0.35]) and s["top 3, vsd_scores 0.3"] == 50.0
    assert s["top 5, vsd_median"] == np.median([0.1, 0.1, 0.3, 0.29]) and s["top 5, vsd_scores 0.3"] == 100.0


def _batch(tmp_path, B=2, N=4):
    import cv2
    paths = []
    for i in range(B):
        p = str(tmp_path / f"d{i}.png")
        cv2.imwrite(p, np.full((6, 8), 1000 + i, np.uint16))
        paths.append(p)
    return {"query": torch.zeros(B, 3, 256, 256), "reference": torch.zeros(B, 3, 256, 256),
            "gt_relativeR": torch.zeros(B, 6), "all_relativeR": torch.zeros(B, N, 6),
            "template_poses": torch.eye(3).expand(B, N, 3, 3), "query_pose": torch.eye(3).expand(B, 3, 3),
            "query_translation": torch.zeros(B, 3, 1), "intrinsic": torch.eye(3).expand(B, 3, 3),
            "depth_path": paths, "obj_id": torch.tensor([1, 2][:B])}


def test_tless_adapter_validates_and_reads_depth(tmp_path):
    from nope_b200.tless import TLessBatchAdapter, keyed_batches
    ad = TLessBatchAdapter(device="cpu")
    b = ad(_batch(tmp_path))
    assert b["depth_raw"].dtype == torch.uint16 and tuple(b["depth_raw"].shape) == (2, 6, 8)
    assert int(b["depth_raw"][1, 0, 0]) == 1001 and b["intrinsic"].dtype == torch.float64
    for key, bad in (("template_poses", torch.zeros(2, 4, 3)), ("query_translation", torch.zeros(2, 3)),
                     ("intrinsic", torch.zeros(2, 4, 4)), ("all_relativeR", torch.zeros(2, 4, 5))):
        x = _batch(tmp_path)
        x[key] = bad
        with pytest.raises(ValueError, match=key):
            ad(x)
    x = _batch(tmp_path)
    x["depth_path"] = x["depth_path"][:1]
    with pytest.raises(ValueError, match="depth_path"):
        ad(x)
    x = _batch(tmp_path)
    del x["obj_id"]
    with pytest.raises(KeyError, match="obj_id"):
        ad(x)
    steps = list(keyed_batches({"seen": [1, 2], "unseen": [3]}))
    assert steps == [{"tless_seen": 1, "tless_unseen": 3}, {"tless_seen": 2}]


def test_test_step_routes_tless_to_eval_vsd(tmp_path, monkeypatch):
    from nope_b200.model import PoseConditional
    m = PoseConditional(u_net=None, save_dir=str(tmp_path))
    calls = []
    monkeypatch.setattr(m, "eval_vsd", lambda b, name, save_path=None: calls.append(("vsd", b, name, save_path)) or "v")
    monkeypatch.setattr(m, "eval_geodesic", lambda b, name, **kw: calls.append(("geo", b, name, kw)) or "g")
    m.global_rank = 3
    out = m.test_step({"tless_seen": "B1", "shapeNet_mug": "B2"}, 7)
    assert out == {"tless_seen": "v", "shapeNet_mug": "g"}
    assert calls[0] == ("vsd", "B1", "seen", os.path.join(str(tmp_path), "predictions", "vsd_seen_batch7_rank_3.npy"))
    assert calls[1] == ("geo", "B2", "mug", {"visualize": True, "save_prediction": True})
