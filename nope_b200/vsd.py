"""VSD (Visible Surface Discrepancy, the BOP pose-error metric) on the GPU: the T-LESS branch of the
reference's evaluation (src/poses/vsd.py, src/poses/vsd_utils.py, model.py:391-541).

* `read_ply`: the CAD models (obj_0000NN.ply, mm); ascii and binary_little_endian, polygons fan-triangulated.
* `MeshTable`: meshes packed on the device once.
* `render_depth`: depth renders of many (mesh, pose) pairs in one call (CUDA z-buffer rasterizer).
* `vsd_error`: the fused per-hypothesis VSD error (bop19 visibility, step cost), exact integer counts.
* `vsd_scores`: the score dict of model.py:530-537.

The port follows the per-frame contract of `vsd_obj` (vsd.py:58-136): a mesh, the 3x3 intrinsics, the
frame's raw depth, k predicted 4x4 poses and one GT pose, errors returned in frame order.  The reference's
`eval_vsd` cannot run as written (it indexes a dict of batched arrays with frame numbers, stores
"gt_poses" where `vsd_obj` reads "query_pose", and collects rows in completion order); those quirks are
not reproduced.  The GT pose is rendered once per frame instead of k times (the k renders are identical).

Renderer convention (what pyrender's IntrinsicsCamera with the OpenCV flip of vsd.py:31-45 computes):
OpenCV camera, pixel (x, y) samples the image point (x + 0.5, y + 0.5), depth = camera z of the nearest
surface, 0 where nothing is hit, znear = 0.05, zfar = 1e5.  pyrender reads depth back through a
non-linear depth buffer; this rasterizer computes it exactly (float64 geometry, fp32 output).
"""
import ctypes as C
import os

import numpy as np
import torch

from . import _lib

DEPTH_SCALE_TLESS = 10.0      # cv2.imread(depth_path, -1) / 10.0 (vsd.py:74): 0.1 mm units -> mm
ZNEAR, ZFAR = 0.05, 100000.0  # vsd.py:42-44

_PLY_TYPES = {"char": "i1", "int8": "i1", "uchar": "u1", "uint8": "u1", "short": "i2", "int16": "i2",
              "ushort": "u2", "uint16": "u2", "int": "i4", "int32": "i4", "uint": "u4", "uint32": "u4",
              "float": "f4", "float32": "f4", "double": "f8", "float64": "f8"}


def read_ply(path):
    """-> (vertices [V,3] float64, faces [F,3] int64).  Reads the `vertex` x/y/z and the `face` vertex
    index list of an ascii or binary_little_endian PLY; other elements and properties are skipped and
    polygons with more than three corners are fan-triangulated."""
    with open(path, "rb") as f:
        data = f.read()
    end = data.find(b"end_header")
    if not data.startswith(b"ply") or end < 0:
        raise ValueError(f"{path}: not a PLY file")
    body = data[data.index(b"\n", end) + 1:]
    fmt, elements = None, []
    for line in data[:end].decode("ascii", "replace").splitlines():
        tok = line.split()
        if not tok:
            continue
        if tok[0] == "format":
            fmt = tok[1]
        elif tok[0] == "element":
            elements.append((tok[1], int(tok[2]), []))
        elif tok[0] == "property" and elements:
            if tok[1] == "list":
                elements[-1][2].append((tok[4], "list", _PLY_TYPES[tok[2]], _PLY_TYPES[tok[3]]))
            else:
                elements[-1][2].append((tok[2], _PLY_TYPES[tok[1]]))
    if fmt not in ("ascii", "binary_little_endian"):
        raise ValueError(f"{path}: PLY format {fmt!r} is not supported (ascii, binary_little_endian)")
    verts, faces = None, []
    if fmt == "ascii":
        words = body.split()
        pos = 0
        for name, count, props in elements:
            rows = []
            for _ in range(count):
                row = {}
                for pr in props:
                    if pr[1] == "list":
                        n = int(words[pos])
                        row[pr[0]] = [int(w) for w in words[pos + 1:pos + 1 + n]]
                        pos += 1 + n
                    else:
                        row[pr[0]] = float(words[pos])
                        pos += 1
                rows.append(row)
            if name == "vertex":
                verts = np.array([[r["x"], r["y"], r["z"]] for r in rows], dtype=np.float64).reshape(-1, 3)
            elif name == "face":
                key = next(pr[0] for pr in props if pr[1] == "list")
                faces = [r[key] for r in rows]
    else:
        pos = 0
        for name, count, props in elements:
            if all(pr[1] != "list" for pr in props):
                dt = np.dtype([(pr[0], "<" + pr[1]) for pr in props])
                arr = np.frombuffer(body, dtype=dt, count=count, offset=pos)
                pos += dt.itemsize * count
                if name == "vertex":
                    verts = np.stack([arr["x"], arr["y"], arr["z"]], 1).astype(np.float64)
                continue
            rows = []
            for _ in range(count):
                for pr in props:
                    if pr[1] == "list":
                        ct, it = np.dtype("<" + pr[2]), np.dtype("<" + pr[3])
                        n = int(np.frombuffer(body, ct, 1, pos)[0])
                        pos += ct.itemsize
                        idx = np.frombuffer(body, it, n, pos)
                        pos += it.itemsize * n
                        if name == "face" and pr[0] in ("vertex_indices", "vertex_index"):
                            rows.append(idx.tolist())
                    else:
                        pos += np.dtype(pr[1]).itemsize
            if name == "face":
                faces = rows
    if verts is None:
        raise ValueError(f"{path}: no vertex element")
    tris = [(p[0], p[i], p[i + 1]) for p in faces for i in range(1, len(p) - 1)]
    return verts, np.array(tris, dtype=np.int64).reshape(-1, 3)


class MeshTable:
    """Meshes packed on one device: vertices [sum V,3] fp32, faces [sum F,3] int32 (indices local to the
    mesh) and host offsets.  Each entry of `meshes` is a PLY path, a (vertices, faces) pair, or an object
    with `.vertices` / `.faces` (a trimesh.Trimesh, say)."""

    def __init__(self, meshes, device="cuda:0"):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.NopeError("MeshTable needs a CUDA device (no CPU fallback)")
        vs, fs = [], []
        for m in meshes:
            if isinstance(m, (str, os.PathLike)):
                v, f = read_ply(m)
            elif hasattr(m, "vertices") and hasattr(m, "faces"):
                v, f = m.vertices, m.faces
            else:
                v, f = m
            v = np.asarray(v.cpu() if torch.is_tensor(v) else v, dtype=np.float64).reshape(-1, 3)
            f = np.asarray(f.cpu() if torch.is_tensor(f) else f, dtype=np.int64).reshape(-1, 3)
            if len(v) == 0 or len(f) == 0:
                raise ValueError(f"mesh {len(vs)} has no vertices or no faces")
            if f.min() < 0 or f.max() >= len(v):
                raise ValueError(f"mesh {len(vs)}: face index outside [0, {len(v)})")
            vs.append(v)
            fs.append(f)
        self.n_vertices = np.array([len(v) for v in vs], dtype=np.int64)
        self.n_faces = np.array([len(f) for f in fs], dtype=np.int64)
        self.voff = np.concatenate([[0], np.cumsum(self.n_vertices)]).astype(np.int64)
        self.foff = np.concatenate([[0], np.cumsum(self.n_faces)]).astype(np.int64)
        self.verts = torch.from_numpy(np.concatenate(vs).astype(np.float32)).to(self.device)
        self.faces = torch.from_numpy(np.concatenate(fs).astype(np.int32)).to(self.device)

    def __len__(self):
        return len(self.n_vertices)


def _host_i64(a):
    return C.c_void_p(a.ctypes.data)


def render_depth(table, mesh_ids, poses, K, H, W, znear=ZNEAR, zfar=ZFAR):
    """Depth renders [P,H,W] fp32 of mesh `mesh_ids[p]` under `poses[p]` ([P,3,4] or [P,4,4], object ->
    OpenCV camera, mm) with intrinsics K ([3,3] shared or [P,3,3], used in float64); 0 = background."""
    lib = _lib.load()
    dev = table.device
    if not torch.is_tensor(poses) or poses.device.type != "cuda":
        raise _lib.NopeError("render_depth needs CUDA pose tensors (no CPU fallback)")
    ids = np.ascontiguousarray(np.asarray(torch.as_tensor(mesh_ids).cpu(), dtype=np.int32).reshape(-1))
    P = len(ids)
    if poses.shape[0] != P or tuple(poses.shape[1:]) not in ((3, 4), (4, 4)):
        raise ValueError(f"poses: expected [{P},3,4] or [{P},4,4], got {tuple(poses.shape)}")
    pose = poses[:, :3, :4].to(dev, torch.float32).contiguous()
    K = torch.as_tensor(K).to(dev, torch.float64)
    K = K.expand(P, 3, 3) if K.dim() == 2 else K
    if tuple(K.shape) != (P, 3, 3):
        raise ValueError(f"K: expected [3,3] or [{P},3,3], got {tuple(K.shape)}")
    intr = torch.stack([K[:, 0, 0], K[:, 1, 1], K[:, 0, 2], K[:, 1, 2]], 1).contiguous()
    depth = torch.empty((P, H, W), device=dev, dtype=torch.float32)
    ws_bytes = lib.nope_vsd_workspace_bytes(_host_i64(table.voff), _host_i64(table.foff), len(table),
                                            C.c_void_p(ids.ctypes.data), P)
    if ws_bytes < 0:
        _lib.check(-1)
    ws = torch.empty(int(ws_bytes), device=dev, dtype=torch.uint8)
    with torch.cuda.device(dev):
        _lib.check(lib.nope_vsd_render(_lib.ptr(table.verts), _lib.ptr(table.faces), _host_i64(table.voff),
                                       _host_i64(table.foff), len(table), C.c_void_p(ids.ctypes.data),
                                       _lib.ptr(pose), _lib.ptr(intr), P, int(H), int(W), float(znear), float(zfar),
                                       _lib.ptr(ws), int(ws_bytes), _lib.ptr(depth),
                                       C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
    return depth


def vsd_error(depth_raw, K, depth_gt, depth_est, delta=15, tau=20, depth_scale=DEPTH_SCALE_TLESS,
              return_counts=False):
    """VSD errors [F,k] float64 of vsd_obj (vsd.py:93-135, bop19, step cost).
    depth_raw [F,H,W] uint16 sensor depth (divided by depth_scale in float64 on the device), K [F,3,3]
    (or [3,3]), depth_gt [F,H,W] and depth_est [F,k,H,W] fp32 renders.  With return_counts also the
    int64 [F,k,3] (|union|, |intersection|, costly pixels) the errors are exact ratios of."""
    lib = _lib.load()
    for name, t in (("depth_raw", depth_raw), ("depth_gt", depth_gt), ("depth_est", depth_est)):
        if not torch.is_tensor(t) or t.device.type != "cuda":
            raise _lib.NopeError(f"vsd_error needs CUDA tensors ({name} is not; no CPU fallback)")
    dev = depth_gt.device
    F_, H, W = depth_gt.shape
    if depth_est.dim() != 4 or depth_est.shape[0] != F_ or tuple(depth_est.shape[2:]) != (H, W):
        raise ValueError(f"depth_est: expected [{F_},k,{H},{W}], got {tuple(depth_est.shape)}")
    if tuple(depth_raw.shape) != (F_, H, W) or depth_raw.dtype != torch.uint16:
        raise ValueError(f"depth_raw: expected uint16 [{F_},{H},{W}], got {depth_raw.dtype} {tuple(depth_raw.shape)}")
    k = depth_est.shape[1]
    K = torch.as_tensor(K).to(dev, torch.float64)
    K = K.expand(F_, 3, 3) if K.dim() == 2 else K
    intr = torch.stack([K[:, 0, 0], K[:, 1, 1], K[:, 0, 2], K[:, 1, 2]], 1).contiguous()
    # contiguous copies are bound to names: a temporary freed before the call could be reused by the next one
    raw = depth_raw.to(dev).contiguous()
    dgt = depth_gt.float().contiguous()
    dest = depth_est.float().contiguous()
    counts = torch.empty((F_, k, 3), device=dev, dtype=torch.int64)
    err = torch.empty((F_, k), device=dev, dtype=torch.float64)
    with torch.cuda.device(dev):
        _lib.check(lib.nope_vsd_error(_lib.ptr(raw), float(depth_scale), _lib.ptr(intr), _lib.ptr(dgt), _lib.ptr(dest),
                                      F_, k, H, W, float(delta), float(tau), _lib.ptr(counts), _lib.ptr(err),
                                      C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
    return (err, counts) if return_counts else err


def vsd_scores(err):
    """model.py:530-537: for k in (1, 3, 5), the median over frames of the best of the first k errors and
    the percentage of frames whose best is <= 0.3."""
    e = np.asarray(err.cpu() if torch.is_tensor(err) else err, dtype=np.float64)
    out = {}
    for k in (1, 3, 5):
        best = np.min(e[:, :k], 1)
        out[f"top {k}, vsd_median"] = np.median(best)
        for threshold in (0.3,):
            out[f"top {k}, vsd_scores {threshold}"] = np.mean((best <= threshold) * 100.0)
    return out
