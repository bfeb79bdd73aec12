"""TEST INFRASTRUCTURE ONLY -- never imported by the product path.

The host-side restatement of the VSD evaluation (src/poses/vsd.py, vsd_utils.py) the CUDA path is
checked against:

* `raycast_depth`: a float64 ray caster.  Pixel (x, y) casts the ray through the image point
  (x + 0.5, y + 0.5) of K (OpenCV camera) and keeps the nearest triangle hit with znear <= z <= zfar.
  It also reports *ambiguous* pixels, whose sample point lies within 1e-3 px of a projected triangle
  edge (or whose hit lies on the near / far plane): there any fill rule may legitimately differ.
* `vsd_counts`: the arithmetic of vsd_obj (bop19 masks, step cost) in float64 numpy, returning the
  integer counts the error is a ratio of.
* `reference_vsd_obj`: the UNMODIFIED reference `src.poses.vsd.vsd_obj` (through oracle/ref_import.py)
  with its module-global `pyrenderer` swapped for the ray caster: the VSD arithmetic is the reference's
  own code and only the renderer is restated.  Needs the reference tree (build container only).
* `python -m oracle.vsd_oracle --write-golden` writes tests/golden/vsd_fixture.npz.
"""
import os
import sys
import tempfile

import numpy as np

from .inputs import GOLDEN_DIR

ZNEAR, ZFAR = 0.05, 100000.0
AMBIGUOUS_PX = 1e-3


def _pose34(pose):
    pose = np.asarray(pose, dtype=np.float64)
    return pose[:3, :3], pose[:3, 3]


def raycast_depth(verts, faces, pose, K, H, W, znear=ZNEAR, zfar=ZFAR):
    """-> (depth [H,W] float64, ambiguous [H,W] bool).  verts [V,3], faces [F,3], pose [3,4] or [4,4]."""
    R, t = _pose34(pose)
    V = np.asarray(verts, dtype=np.float64) @ R.T + t
    K = np.asarray(K, dtype=np.float64)
    fx, fy, cx, cy = K[0, 0], K[1, 1], K[0, 2], K[1, 2]
    depth = np.full((H, W), np.inf)
    amb = np.zeros((H, W), dtype=bool)
    for f in np.asarray(faces, dtype=np.int64):
        A, B, Cv = V[f[0]], V[f[1]], V[f[2]]
        zs = np.array([A[2], B[2], Cv[2]])
        if (zs < znear).all() or (zs > zfar).all():
            continue
        if (zs > 0).all():
            us = fx * np.array([A[0], B[0], Cv[0]]) / zs + cx
            vs = fy * np.array([A[1], B[1], Cv[1]]) / zs + cy
            x0, x1 = int(max(np.floor(us.min() - 1.5), 0)), int(min(np.ceil(us.max() + 0.5), W - 1))
            y0, y1 = int(max(np.floor(vs.min() - 1.5), 0)), int(min(np.ceil(vs.max() + 0.5), H - 1))
        else:                                   # a vertex behind the eye: the projection is unbounded
            x0, x1, y0, y1 = 0, W - 1, 0, H - 1
        if x0 > x1 or y0 > y1:
            continue
        px, py = np.meshgrid(np.arange(x0, x1 + 1), np.arange(y0, y1 + 1))
        su, sv = px + 0.5, py + 0.5
        d = np.stack([(su - cx) / fx, (sv - cy) / fy, np.ones_like(su)], -1)
        e1, e2 = B - A, Cv - A
        pvec = np.cross(d, e2)
        det = pvec @ e1
        with np.errstate(divide="ignore", invalid="ignore"):
            inv = 1.0 / det
            tvec = -A
            u = (pvec @ tvec) * inv
            qvec = np.cross(tvec, e1)
            v = (d @ qvec) * inv
            z = (qvec @ e2) * inv
        ok = np.isfinite(inv)
        hit = ok & (u >= 0) & (v >= 0) & (u + v <= 1) & (z >= znear) & (z <= zfar)
        near = ok & (u >= -1e-2) & (v >= -1e-2) & (u + v <= 1 + 1e-2) & (z >= znear * (1 - 1e-6)) & \
            (z <= zfar * (1 + 1e-6))
        # distance (px) of the sample to each edge's projection: the plane through the eye and the edge
        edge_close = np.zeros_like(hit)
        for P0, P1 in ((A, B), (B, Cv), (Cv, A)):
            n = np.cross(P0, P1)
            a, b = n[0] / fx, n[1] / fy
            c = n[2] - n[0] * cx / fx - n[1] * cy / fy
            nrm = np.hypot(a, b)
            if nrm > 0:
                edge_close |= np.abs(a * su + b * sv + c) / nrm <= AMBIGUOUS_PX
        plane_close = (np.abs(z - znear) <= 1e-6 * znear) | (np.abs(z - zfar) <= 1e-6 * zfar)
        amb[y0:y1 + 1, x0:x1 + 1] |= near & (edge_close | plane_close)
        cur = depth[y0:y1 + 1, x0:x1 + 1]
        np.copyto(cur, np.where(hit & (z < cur), z, cur))
    depth[np.isinf(depth)] = 0.0
    return depth, amb


def dist_im(depth, K):
    """depth_im_to_dist_im_fast (vsd_utils.py:40-62)."""
    K = np.asarray(K, dtype=np.float64)
    xs, ys = np.meshgrid(np.arange(depth.shape[1]), np.arange(depth.shape[0]))
    pre_x = (xs - K[0, 2]) / np.float64(K[0, 0])
    pre_y = (ys - K[1, 2]) / np.float64(K[1, 1])
    return np.sqrt(np.multiply(pre_x, depth) ** 2 + np.multiply(pre_y, depth) ** 2 + depth.astype(np.float64) ** 2)


def vsd_counts(depth_test, K, depth_gt, depth_est, delta=15, tau=20):
    """(|union|, |intersection|, costly pixels) of vsd_obj's inner loop (vsd.py:96-127, bop19, step).
    depth_test in mm (float64), renders as float32 arrays."""
    dt, dg, de = dist_im(depth_test, K), dist_im(depth_gt, K), dist_im(depth_est, K)
    vis_gt = np.logical_and(np.logical_or(dg.astype(np.float32) - dt.astype(np.float32) <= delta, dt == 0), dg > 0)
    vis_est = np.logical_and(np.logical_or(de.astype(np.float32) - dt.astype(np.float32) <= delta, dt == 0), de > 0)
    vis_est = np.logical_or(vis_est, np.logical_and(vis_gt, de > 0))
    inter = np.logical_and(vis_gt, vis_est)
    union = np.logical_or(vis_gt, vis_est)
    costs = np.abs(dg[inter] - de[inter]) >= tau
    return int(union.sum()), int(inter.sum()), int(costs.sum())


def error_from_counts(c):
    u, i, n = c
    return 1.0 if u == 0 else (n + (u - i)) / float(u)


def reference_vsd_obj(verts, faces, K, depth_raw_u16, pred_poses, gt_pose, delta=15, tau=20):
    """The reference's vsd_obj on one frame, its renderer replaced by `raycast_depth` (float32 depth,
    as pyrender returns).  Returns the float64 errors [k]."""
    import cv2
    from .ref_import import REFERENCE_ROOT, _install_stubs, reference_available
    if not reference_available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT}")
    _install_stubs()
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    from src.poses import vsd as ref_vsd

    def raycast_renderer(obj_poses, BOP_cad_trimesh, intrinsic, img_size):
        v, f = BOP_cad_trimesh
        if len(obj_poses.shape) == 2:
            obj_poses = obj_poses[None, ...]
        return [raycast_depth(v, f, p, intrinsic, img_size[0], img_size[1])[0].astype(np.float32)
                for p in obj_poses]

    saved = ref_vsd.pyrenderer
    ref_vsd.pyrenderer = raycast_renderer
    try:
        with tempfile.TemporaryDirectory() as d:
            path = os.path.join(d, "depth.png")
            cv2.imwrite(path, np.asarray(depth_raw_u16, dtype=np.uint16))
            frame = {"mesh": (verts, faces), "intrinsic": np.asarray(K), "depth_path": path,
                     "pred_poses": np.asarray(pred_poses, dtype=np.float64).copy(),
                     "query_pose": np.asarray(gt_pose, dtype=np.float64)}
            return ref_vsd.vsd_obj(0, [frame], delta_vsd=delta, tau_vsd=tau)
    finally:
        ref_vsd.pyrenderer = saved


# ------------------------------------------------------------------------------------------------
# procedural geometry (also used by the GPU tests and tools/vsd_bench.py)
# ------------------------------------------------------------------------------------------------
def bumpy_sphere(n_lat=12, n_lon=24, radius=30.0, center=(0.0, 0.0, 0.0), seed=0, bump=0.15):
    """Closed UV sphere with seeded radial bumps: verts float32 [V,3] (mm), faces int64 [F,3]."""
    rng = np.random.default_rng(seed)
    th = np.linspace(0, np.pi, n_lat + 1)[1:-1]
    ph = np.linspace(0, 2 * np.pi, n_lon, endpoint=False)
    T, Pp = np.meshgrid(th, ph, indexing="ij")
    r = radius * (1 + bump * rng.uniform(-1, 1, T.shape))
    ring = np.stack([r * np.sin(T) * np.cos(Pp), r * np.sin(T) * np.sin(Pp), r * np.cos(T)], -1).reshape(-1, 3)
    verts = np.concatenate([[[0, 0, radius]], ring, [[0, 0, -radius]]]) + np.asarray(center)
    faces = []
    idx = lambda i, j: 1 + i * n_lon + (j % n_lon)  # noqa: E731
    for j in range(n_lon):
        faces.append((0, idx(0, j), idx(0, j + 1)))
        faces.append((len(verts) - 1, idx(n_lat - 2, j + 1), idx(n_lat - 2, j)))
    for i in range(n_lat - 2):
        for j in range(n_lon):
            faces.append((idx(i, j), idx(i + 1, j), idx(i + 1, j + 1)))
            faces.append((idx(i, j), idx(i + 1, j + 1), idx(i, j + 1)))
    return verts.astype(np.float32), np.array(faces, dtype=np.int64)


def box(half=(20.0, 20.0, 20.0), center=(0.0, 0.0, 0.0)):
    hx, hy, hz = half
    v = np.array([[sx * hx, sy * hy, sz * hz] for sx in (-1, 1) for sy in (-1, 1) for sz in (-1, 1)]) + np.asarray(center)
    f = [(0, 1, 3), (0, 3, 2), (4, 6, 7), (4, 7, 5), (0, 4, 5), (0, 5, 1), (2, 3, 7), (2, 7, 6),
         (0, 2, 6), (0, 6, 4), (1, 5, 7), (1, 7, 3)]
    return v.astype(np.float32), np.array(f, dtype=np.int64)


def rotation(axis, deg):
    a = np.asarray(axis, dtype=np.float64)
    a = a / np.linalg.norm(a)
    th = np.deg2rad(deg)
    Kx = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    return np.eye(3) + np.sin(th) * Kx + (1 - np.cos(th)) * Kx @ Kx


def pose44(R, t):
    P = np.eye(4)
    P[:3, :3], P[:3, 3] = R, t
    return P.astype(np.float32).astype(np.float64)    # the fp32 values the device sees


def scene_depth_raw(verts, faces, gt_pose, K, H, W, seed=0, occluder=True, holes=0.03):
    """A sensor-like uint16 depth (0.1 mm units) of the object in its GT pose: an occluding box in front
    of part of it, a background plane, seeded noise and zero-depth holes."""
    rng = np.random.default_rng(seed)
    d_obj, _ = raycast_depth(verts, faces, gt_pose, K, H, W)
    R, t = _pose34(gt_pose)
    z_bg = t[2] + 150.0
    scene = np.where(d_obj > 0, d_obj, z_bg)
    if occluder:
        c = (np.asarray(verts, dtype=np.float64) @ R.T + t).mean(0)       # object centre, camera frame
        bv, bf = box(half=(25.0, 60.0, 5.0))
        d_occ, _ = raycast_depth(bv, bf, pose44(np.eye(3), 0.7 * c + np.array([-20.0, 0.0, 0.0])), K, H, W)
        scene = np.where((d_occ > 0) & (d_occ < scene), d_occ, scene)
    scene = scene + rng.normal(0, 1.0, scene.shape)
    raw = np.round(scene * 10.0).clip(0, 65535).astype(np.uint16)
    raw[rng.random(raw.shape) < holes] = 0
    return raw


def fixture_frames():
    """Two frames (160x120, K of a T-LESS Primesense frame scaled by 2/9): one procedural mesh whose
    body sits 250 mm from its origin, so a half-turn rotation about the GT translation puts it behind the
    camera (an empty render: error 1.0)."""
    s = 160.0 / 720.0
    K = np.array([[1075.65 * s, 0, 360.0 * s], [0, 1073.90 * s, 270.0 * s], [0, 0, 1]])
    verts, faces = bumpy_sphere(n_lat=10, n_lon=20, radius=30.0, center=(0.0, 0.0, 250.0), seed=3)
    frames = []
    for fi, (axis, deg) in enumerate((((0.3, 1.0, 0.2), 20.0), ((1.0, -0.4, 0.5), -35.0))):
        Rg = rotation(axis, deg)
        t = np.array([8.0 * fi, -5.0, 150.0])
        gt = pose44(Rg, t)
        cands = [Rg @ rotation((1, 2, 3), 12.0), Rg, Rg @ rotation((0, 1, 0), 40.0),
                 rotation((1, 0, 0), 180.0) @ Rg, Rg @ rotation((1, 0, 1), -7.0)]
        if fi == 1:
            cands = cands[1:] + cands[:1]
        pred = np.stack([pose44(R, t + 100.0) for R in cands])   # translations are replaced by the GT one
        frames.append(dict(K=K, gt_pose=gt, pred_poses=pred,
                           depth_raw=scene_depth_raw(verts, faces, gt, K, 120, 160, seed=fi)))
    return verts, faces, frames


def write_golden():
    verts, faces, frames = fixture_frames()
    H, W = 120, 160
    out = dict(verts=verts, faces=faces, K=frames[0]["K"],
               depth_raw=np.stack([f["depth_raw"] for f in frames]),
               gt_poses=np.stack([f["gt_pose"] for f in frames]),
               pred_poses=np.stack([f["pred_poses"] for f in frames]))
    gt_d, gt_a, est_d, est_a, counts, errs_ref = [], [], [], [], [], []
    for f in frames:
        d, a = raycast_depth(verts, faces, f["gt_pose"], f["K"], H, W)
        gt_d.append(d.astype(np.float32))
        gt_a.append(a)
        ed, ea, cs = [], [], []
        for p in f["pred_poses"]:
            p = p.copy()
            p[:3, 3] = f["gt_pose"][:3, 3]
            d2, a2 = raycast_depth(verts, faces, p, f["K"], H, W)
            ed.append(d2.astype(np.float32))
            ea.append(a2)
            cs.append(vsd_counts(f["depth_raw"] / 10.0, f["K"], gt_d[-1], ed[-1]))
        est_d.append(np.stack(ed))
        est_a.append(np.stack(ea))
        counts.append(cs)
        errs_ref.append(reference_vsd_obj(verts, faces, f["K"], f["depth_raw"], f["pred_poses"], f["gt_pose"]))
    out.update(depth_gt=np.stack(gt_d), amb_gt=np.stack(gt_a), depth_est=np.stack(est_d), amb_est=np.stack(est_a),
               counts=np.array(counts, dtype=np.int64), err_reference=np.stack(errs_ref))
    errs_oracle = np.array([[error_from_counts(c) for c in cs] for cs in counts])
    assert np.array_equal(errs_oracle, out["err_reference"]), (errs_oracle, out["err_reference"])
    path = os.path.join(GOLDEN_DIR, "vsd_fixture.npz")
    np.savez_compressed(path, **out)
    print(path, os.path.getsize(path), "bytes; reference errors:\n", out["err_reference"])


if __name__ == "__main__":
    if "--write-golden" in sys.argv:
        write_golden()
