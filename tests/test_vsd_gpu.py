"""GPU: the T-LESS / VSD evaluation -- CUDA rasterizer against the float64 ray caster, determinism, the
fused VSD kernel against the reference vsd_obj's counts, and eval_vsd / test_step end to end."""
import os

import numpy as np
import pytest
import torch

from _util import log

pytestmark = pytest.mark.gpu

KT = np.array([[1075.65, 0.0, 360.0], [0.0, 1073.90, 270.0], [0.0, 0.0, 1.0]])    # T-LESS Primesense, 720x540


def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _render(meshes, ids, poses, K, H, W, **kw):
    from nope_b200.vsd import MeshTable, render_depth
    table = MeshTable(meshes)
    P = torch.tensor(np.stack(poses)[:, :3, :4], dtype=torch.float32, device="cuda:0")
    return render_depth(table, ids, P, torch.tensor(K), H, W, **kw).cpu().numpy()


def _compare(depth, mesh, pose, K, H, W, name, closed=True):
    """Coverage identical on every non-ambiguous pixel, |dz| <= 1e-4 z where both cover, and (closed
    meshes) no hole strictly inside the silhouette."""
    from oracle.vsd_oracle import raycast_depth
    d_o, amb = raycast_depth(mesh[0], mesh[1], pose, K, H, W)
    cov, cov_o = depth > 0, d_o > 0
    bad = (cov != cov_o) & ~amb
    both = cov & cov_o
    dz = np.abs(depth[both] - d_o[both]) / d_o[both] if both.any() else np.zeros(1)
    log("vsd_raster", case=name, covered=int(cov.sum()), ambiguous=int(amb.sum()), mismatched=int(bad.sum()),
        max_rel_dz=float(dz.max()))
    assert not bad.any(), (name, np.argwhere(bad)[:10])
    assert dz.max() <= 1e-4, name
    if closed and cov_o.any():
        import scipy.ndimage as ndi
        inner = ndi.binary_erosion(cov_o, iterations=1) & ~ndi.binary_dilation(amb, iterations=1)
        assert cov[inner].all(), (name, np.argwhere(inner & ~cov)[:10])


def test_raster_matches_raycaster_on_fixture(golden_dir):
    _cuda()
    g = np.load(os.path.join(golden_dir, "vsd_fixture.npz"))
    mesh = (g["verts"], g["faces"])
    for f in range(2):
        poses = [g["gt_poses"][f]]
        for p in g["pred_poses"][f]:
            p = p.copy()
            p[:3, 3] = g["gt_poses"][f][:3, 3]
            poses.append(p)
        d = _render([mesh], [0] * 6, poses, g["K"], 120, 160)
        ref = np.concatenate([g["depth_gt"][f][None], g["depth_est"][f]])
        amb = np.concatenate([g["amb_gt"][f][None], g["amb_est"][f]])
        for j in range(6):
            bad = ((d[j] > 0) != (ref[j] > 0)) & ~amb[j]
            assert not bad.any(), (f, j, np.argwhere(bad)[:10])
            both = (d[j] > 0) & (ref[j] > 0)
            assert np.all(np.abs(d[j][both] - ref[j][both]) <= 1e-4 * ref[j][both])


def test_raster_live_cases():
    _cuda()
    from oracle.vsd_oracle import box, bumpy_sphere, pose44, rotation
    from nope_b200.tless import procedural_mesh
    H, W = 540, 720
    sphere = bumpy_sphere(n_lat=30, n_lon=60, radius=40.0, seed=1)
    blob = procedural_mesh(5, n_lat=40, n_lon=80)
    cube = box(half=(30.0, 20.0, 25.0))
    quad = (np.array([[-500, -400, 0], [500, -400, 0], [500, 400, 0], [-500, 400, 0]], np.float32),
            np.array([[0, 1, 2], [0, 2, 3]]))
    cases = [("sphere", sphere, pose44(rotation((1, 2, 0), 30), [20, -10, 500])),
             ("blob", blob, pose44(rotation((0, 1, 1), -50), [-30, 25, 700])),
             ("cube_close", cube, pose44(rotation((1, 1, 1), 40), [0, 0, 120])),
             ("frame_filling_quad", quad, pose44(rotation((1, 0.3, 0), 25), [3, -2, 300]))]
    for name, mesh, pose in cases:
        d = _render([mesh], [0], [pose], KT, H, W)[0]
        _compare(d, mesh, pose, KT, H, W, name, closed=name != "frame_filling_quad")
    assert (d > 0).all()       # the quad fills the frame through the one-CTA-per-face path
    # a mesh crossing the near plane (camera inside the cube), then poses behind the camera / off-screen
    near = pose44(rotation((0, 1, 0), 10), [5, 3, 0.03])
    d = _render([cube], [0], [near], KT, H, W)[0]
    _compare(d, cube, near, KT, H, W, "near_plane_clip", closed=False)
    assert (d > 0).any()
    empty = [pose44(np.eye(3), [0, 0, -200]), pose44(np.eye(3), [5000, 0, 500]), pose44(np.eye(3), [0, 0, 2e5])]
    assert not _render([sphere], [0, 0, 0], empty, KT, H, W).any()


def test_raster_is_deterministic_across_groupings():
    _cuda()
    from oracle.vsd_oracle import bumpy_sphere, pose44, rotation
    from nope_b200.tless import procedural_mesh
    meshes = [bumpy_sphere(n_lat=20, n_lon=40, seed=2), procedural_mesh(3, n_lat=30, n_lon=60),
              procedural_mesh(4, n_lat=12, n_lon=24, radius=90)]
    rng = np.random.default_rng(0)
    poses = [pose44(rotation(rng.normal(size=3), rng.uniform(0, 360)),
                    [rng.uniform(-80, 80), rng.uniform(-60, 60), rng.uniform(150, 900)]) for _ in range(48)]
    ids = [int(i) for i in rng.integers(0, 3, 48)]
    a = _render(meshes, ids, poses, KT, 540, 720)
    b = _render(meshes, ids, poses, KT, 540, 720)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    for p in (0, 17, 47):
        one = _render(meshes, [ids[p]], [poses[p]], KT, 540, 720)[0]
        assert np.array_equal(one.view(np.uint32), a[p].view(np.uint32)), p


def test_vsd_kernel_counts_equal_reference_on_oracle_depths(golden_dir):
    _cuda()
    from nope_b200.vsd import vsd_error
    g = np.load(os.path.join(golden_dir, "vsd_fixture.npz"))
    dev = "cuda:0"
    err, counts = vsd_error(torch.from_numpy(g["depth_raw"]).to(dev), torch.from_numpy(g["K"]),
                            torch.from_numpy(g["depth_gt"]).to(dev), torch.from_numpy(g["depth_est"]).to(dev),
                            return_counts=True)
    assert np.array_equal(counts.cpu().numpy(), g["counts"])
    assert np.array_equal(err.cpu().numpy(), g["err_reference"])
    # empty union: nothing rendered in either pose -> 1.0
    z = torch.zeros(1, 120, 160, device=dev)
    e = vsd_error(torch.from_numpy(g["depth_raw"][:1]).to(dev), torch.from_numpy(g["K"]), z, z[:, None])
    assert float(e) == 1.0


def test_vsd_errors_on_live_720x540_scene():
    _cuda()
    from oracle.vsd_oracle import error_from_counts, pose44, rotation, scene_depth_raw, vsd_counts
    from nope_b200.tless import procedural_mesh
    from nope_b200.vsd import vsd_error
    mesh = procedural_mesh(7, n_lat=30, n_lon=60)
    gt = pose44(rotation((1, 0, 1), 30), [10, -20, 600])
    raw = scene_depth_raw(mesh[0], mesh[1], gt, KT, 540, 720, seed=4)
    poses = [gt] + [pose44(rotation((1, 0, 1), 30) @ rotation((0, 1, 0), a), [10, -20, 600]) for a in (0, 5, 20, 90)]
    d = _render([mesh], [0] * 5, poses, KT, 540, 720)
    dev = "cuda:0"
    err, counts = vsd_error(torch.from_numpy(raw[None]).to(dev), torch.from_numpy(KT),
                            torch.from_numpy(d[:1]).to(dev), torch.from_numpy(d[None, 1:]).to(dev), return_counts=True)
    ref = [vsd_counts(raw / 10.0, KT, d[0], d[j]) for j in range(1, 5)]
    assert [tuple(c) for c in counts[0].tolist()] == ref
    assert err[0].tolist() == [error_from_counts(c) for c in ref]
    assert err[0, 0] == 0.0 and 0 < err[0, 3] <= 1


def _oracle_frame_errors(batch, topi, meshes, H, W):
    """vsd_obj on the oracle's renders for the model's own top-5 poses, plus the per-entry slack
    (ambiguous pixels of either render + 1) / |union|."""
    from oracle.vsd_oracle import error_from_counts, raycast_depth, vsd_counts
    errs, slack = [], []
    for b in range(topi.shape[0]):
        mesh = meshes[int(batch["obj_id"][b]) - 1]
        K = batch["intrinsic"][b].numpy()
        t = batch["query_translation"][b].numpy().reshape(3)
        gt = np.eye(4)
        gt[:3, :3], gt[:3, 3] = batch["query_pose"][b].numpy(), t
        dg, ag = raycast_depth(mesh[0], mesh[1], gt.astype(np.float32), K, H, W)
        raw = __import__("cv2").imread(batch["depth_path"][b], -1)
        row, srow = [], []
        for j in topi[b]:
            p = np.eye(4)
            p[:3, :3], p[:3, 3] = batch["template_poses"][b][j].numpy(), t
            de, ae = raycast_depth(mesh[0], mesh[1], p.astype(np.float32), K, H, W)
            c = vsd_counts(raw / 10.0, K, dg.astype(np.float32), de.astype(np.float32))
            row.append(error_from_counts(c))
            srow.append((int((ag | ae).sum()) + 1) / max(c[0], 1))
        errs.append(row)
        slack.append(srow)
    return np.array(errs), np.array(slack)


@pytest.fixture
def vsd_model(gpu_model, tmp_path):
    """The session model with a save_dir and CAD models for this test only."""
    saved = gpu_model.save_dir
    gpu_model.save_dir = str(tmp_path / "out")
    yield gpu_model
    gpu_model.save_dir, gpu_model.tless_cad = saved, None


def test_eval_vsd_end_to_end(vsd_model, tmp_path):
    gpu_model = vsd_model
    from nope_b200.tless import SyntheticTLess, TLessBatchAdapter, keyed_batches
    from nope_b200.vsd import read_ply
    ds = SyntheticTLess(tmp_path / "tless", n_items=4, n_meshes=2, grid=26, seed=0)
    loader = torch.utils.data.DataLoader(ds, batch_size=4)
    batch = next(iter(loader))
    gpu_model.load_mesh(str(tmp_path / "tless" / "models"), obj_ids=[1, 2])
    ad = TLessBatchAdapter(device="cuda:0")
    step = next(keyed_batches({"seen": [ad(batch)]}))
    out = gpu_model.test_step(step, 0)
    scores = out["tless_seen"]
    assert set(scores) == {f"top {k}, {n}" for k in (1, 3, 5) for n in ("vsd_median", "vsd_scores 0.3")}
    for key in scores:
        assert f"{key}/val_seen" in gpu_model.logged
    assert "loss/val_seen" in gpu_model.logged
    err = gpu_model.last_vsd_error
    saved = np.load(tmp_path / "out" / "predictions" / "vsd_seen_batch0_rank_0.npy")
    assert np.array_equal(saved, err[:, 0])
    _, topi, _ = gpu_model.predict_pose(ad(batch)["query"], ad(batch)["reference"], ad(batch)["all_relativeR"], k=5)
    meshes = [read_ply(tmp_path / "tless" / "models" / f"obj_{i:06d}.ply") for i in (1, 2)]
    ref, slack = _oracle_frame_errors(batch, topi.cpu().numpy(), meshes, ds.H, ds.W)
    log("eval_vsd", err=err.tolist(), oracle=ref.tolist(), max_abs_diff=float(np.abs(err - ref).max()))
    assert np.all(np.abs(err - ref) <= slack)
    # the same frames in two batches give the same errors
    halves = []
    for sl in (slice(0, 2), slice(2, 4)):
        half = {k: (v[sl] if not isinstance(v, list) else v[sl]) for k, v in batch.items()}
        gpu_model.eval_vsd(ad(half), "seen")
        halves.append(gpu_model.last_vsd_error)
    assert np.array_equal(np.concatenate(halves), err)


def test_cpu_tensors_and_bad_arguments_raise():
    _cuda()
    import ctypes as C
    from nope_b200 import NopeError, _lib
    from nope_b200.vsd import MeshTable, render_depth, vsd_error
    from oracle.vsd_oracle import box
    with pytest.raises(NopeError):
        MeshTable([box()], device="cpu")
    table = MeshTable([box()])
    with pytest.raises(NopeError):
        render_depth(table, [0], torch.zeros(1, 3, 4), torch.eye(3), 8, 8)
    z = torch.zeros(1, 8, 8)
    with pytest.raises(NopeError):
        vsd_error(torch.zeros(1, 8, 8, dtype=torch.uint16), torch.eye(3), z, z[:, None])
    with pytest.raises(NopeError, match="mesh id 3"):
        render_depth(table, [3], torch.zeros(1, 3, 4, device="cuda:0"), torch.eye(3), 8, 8)
    with pytest.raises(NopeError, match="image size"):
        render_depth(table, [0], torch.zeros(1, 3, 4, device="cuda:0"), torch.eye(3), 0, 8)
    lib = _lib.load()
    d = torch.zeros(1, 8, 8, device="cuda:0")
    rc = lib.nope_vsd_error(_lib.ptr(torch.zeros(1, 8, 8, dtype=torch.uint16, device="cuda:0")), 10.0,
                            _lib.ptr(torch.ones(1, 4, dtype=torch.float64, device="cuda:0")), _lib.ptr(d), _lib.ptr(d),
                            1, 0, 8, 8, 15.0, 20.0, _lib.ptr(torch.zeros(3, dtype=torch.int64, device="cuda:0")),
                            _lib.ptr(torch.zeros(1, dtype=torch.float64, device="cuda:0")), C.c_void_p(0))
    assert rc != 0 and b"F*k" in lib.nope_last_error()
