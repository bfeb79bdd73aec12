"""Input side of the T-LESS evaluation (the `tless_<cat>` branch of model.py:550-565, eval_vsd model.py:391-541).

The reference's BOP loader has no test split (src/dataloader/bop.py:298-299 raises), so the batch schema is
what eval_vsd reads:
  query, reference [B,3,256,256]; gt_relativeR [B,6]; all_relativeR [B,N,6]; template_poses [B,N,3,3]
  (per batch element); query_pose [B,3,3]; query_translation [B,3,1] (mm); intrinsic [B,3,3];
  depth_path (B strings, uint16 PNGs in 0.1 mm); obj_id [B]; gt_templates optional.
* `TLessBatchAdapter` validates that schema, reads the depth PNGs into pinned memory (`depth_raw`
  uint16 [B,H,W]) and moves the tensors to the device.
* `keyed_batches`: {"tless_<cat>": batch} per step, as `trainer.test` hands them to `test_step`.
* `SyntheticTLess`: seeded procedural meshes written as PLY plus depth PNGs of rendered scenes (an
  occluder, sensor noise, zero-depth holes): plumbing and throughput, not accuracy.
"""
import os

import numpy as np
import torch

BATCH_KEYS = ("query", "reference", "gt_relativeR", "all_relativeR", "template_poses", "query_pose",
              "query_translation", "intrinsic", "depth_path", "obj_id")


def read_depth(paths):
    """uint16 depth PNGs -> pinned uint16 tensor [B,H,W] (cv2.imread(path, -1), vsd.py:74)."""
    import cv2
    ims = []
    for p in paths:
        im = cv2.imread(str(p), -1)
        if im is None or im.dtype != np.uint16 or im.ndim != 2:
            raise ValueError(f"depth_path {p!r}: not a single-channel uint16 image")
        ims.append(im)
    if len({im.shape for im in ims}) != 1:
        raise ValueError(f"depth images differ in size: {sorted({im.shape for im in ims})}")
    out = torch.from_numpy(np.stack(ims))
    return out.pin_memory() if torch.cuda.is_available() else out


class TLessBatchAdapter:
    """Validates a collated T-LESS test batch and puts it on `device` (depth read from depth_path)."""

    def __init__(self, device="cuda:0", image_size=256):
        self.device = torch.device(device)
        self.image_size = image_size

    def __call__(self, batch):
        missing = [k for k in BATCH_KEYS if k not in batch]
        if missing:
            raise KeyError(f"T-LESS test batch misses {missing}")
        q = batch["query"]
        B = q.shape[0]
        N = batch["all_relativeR"].shape[1] if batch["all_relativeR"].dim() == 3 else -1
        S = self.image_size
        shapes = {"query": (B, 3, S, S), "reference": (B, 3, S, S), "gt_relativeR": (B, 6),
                  "all_relativeR": (B, N, 6), "template_poses": (B, N, 3, 3), "query_pose": (B, 3, 3),
                  "query_translation": (B, 3, 1), "intrinsic": (B, 3, 3)}
        out = {}
        for name, shape in shapes.items():
            t = torch.as_tensor(batch[name])
            if tuple(t.shape) != shape:
                raise ValueError(f"{name}: expected {list(shape)}, got {list(t.shape)}")
            out[name] = t.to(self.device, torch.float64 if name == "intrinsic" else torch.float32)
        obj = torch.as_tensor(batch["obj_id"]).reshape(-1)
        if obj.shape[0] != B:
            raise ValueError(f"obj_id: expected {B} ids, got {obj.shape[0]}")
        out["obj_id"] = obj.to(torch.int64)
        paths = list(batch["depth_path"])
        if len(paths) != B:
            raise ValueError(f"depth_path: expected {B} paths, got {len(paths)}")
        out["depth_path"] = paths
        out["depth_raw"] = read_depth(paths).to(self.device, non_blocking=True)
        if batch.get("gt_templates") is not None:
            out["gt_templates"] = batch["gt_templates"]      # stays on the host: visualisation only
        return out


def keyed_batches(loaders):
    """loaders: {category: iterable of batches} -> yields {"tless_<category>": batch} per step."""
    its = {c: iter(l) for c, l in loaders.items()}
    while its:
        step = {}
        for c in list(its):
            try:
                step[f"tless_{c}"] = next(its[c])
            except StopIteration:
                del its[c]
        if step:
            yield step


def _write_ply(path, verts, faces):
    with open(path, "wb") as f:
        f.write(f"ply\nformat binary_little_endian 1.0\nelement vertex {len(verts)}\nproperty float x\n"
                f"property float y\nproperty float z\nelement face {len(faces)}\n"
                "property list uchar int vertex_indices\nend_header\n".encode())
        f.write(np.asarray(verts, dtype="<f4").tobytes())
        rec = np.zeros(len(faces), dtype=[("n", "u1"), ("i", "<i4", 3)])
        rec["n"], rec["i"] = 3, faces
        f.write(rec.tobytes())


def procedural_mesh(seed, n_lat=24, n_lon=48, radius=40.0):
    """A closed, seeded 'bumpy sphere' mesh (mm): verts [V,3] float32, faces [F,3] int64."""
    rng = np.random.default_rng(seed)
    th = np.linspace(0, np.pi, n_lat + 1)[1:-1]
    ph = np.linspace(0, 2 * np.pi, n_lon, endpoint=False)
    T, P = np.meshgrid(th, ph, indexing="ij")
    r = radius * (1 + 0.2 * rng.uniform(-1, 1) * np.sin(3 * T) * np.cos(2 * P + rng.uniform(0, 6)))
    ring = np.stack([r * np.sin(T) * np.cos(P), r * np.sin(T) * np.sin(P), 1.3 * r * np.cos(T)], -1).reshape(-1, 3)
    verts = np.concatenate([[[0, 0, 1.3 * radius]], ring, [[0, 0, -1.3 * radius]]])
    idx = lambda i, j: 1 + i * n_lon + (j % n_lon)  # noqa: E731
    faces = []
    for j in range(n_lon):
        faces += [(0, idx(0, j), idx(0, j + 1)), (len(verts) - 1, idx(n_lat - 2, j + 1), idx(n_lat - 2, j))]
    for i in range(n_lat - 2):
        for j in range(n_lon):
            faces += [(idx(i, j), idx(i + 1, j), idx(i + 1, j + 1)), (idx(i, j), idx(i + 1, j + 1), idx(i, j + 1))]
    return verts.astype(np.float32), np.array(faces, dtype=np.int64)


class SyntheticTLess(torch.utils.data.Dataset):
    """Items of the T-LESS test schema over `n_meshes` procedural objects.  __init__ writes
    `root`/models/obj_0000NN.ply and one depth PNG per item (rendered on `device` with the package's
    rasterizer: the object in its GT pose, an occluding slab, a background plane, noise and holes)."""

    H, W = 540, 720
    K = np.array([[1075.65, 0.0, 360.0], [0.0, 1073.90, 270.0], [0.0, 0.0, 1.0]])     # T-LESS Primesense

    def __init__(self, root, category="test", n_items=4, n_meshes=2, grid=26, seed=0, device="cuda:0"):
        from .poses import synthetic_pose_batch
        from .vsd import MeshTable, render_depth
        self.root, self.category, self.n = str(root), category, n_items
        os.makedirs(os.path.join(self.root, "models"), exist_ok=True)
        os.makedirs(os.path.join(self.root, "depth"), exist_ok=True)
        meshes = [procedural_mesh(seed * 100 + m) for m in range(n_meshes)]
        for m, (v, f) in enumerate(meshes):
            _write_ply(os.path.join(self.root, "models", f"obj_{m + 1:06d}.ply"), v, f)
        _, R = synthetic_pose_batch(grid, 1)
        self.R = R.numpy().astype(np.float32)
        rng = np.random.default_rng(seed)
        self.items = []
        slab = (np.array([[x, y, 0.0] for x in (-30, 30) for y in (-200, 200)], np.float32),
                np.array([[0, 1, 3], [0, 3, 2]], np.int64))
        table = MeshTable(meshes + [slab], device=device)
        for i in range(n_items):
            qi, ri = int(rng.integers(len(self.R))), int(rng.integers(len(self.R)))
            t = np.array([rng.uniform(-60, 60), rng.uniform(-40, 40), rng.uniform(600, 900)], np.float32)
            m = int(rng.integers(n_meshes))
            pose = np.concatenate([self.R[qi], t[:, None]], 1)
            occ = np.concatenate([np.eye(3, dtype=np.float32), (t * 0.8 + [-45.0, 0, 0])[:, None].astype(np.float32)], 1)
            d = render_depth(table, [m, n_meshes], torch.tensor(np.stack([pose, occ]), device=device),
                             torch.tensor(self.K), self.H, self.W).cpu().numpy().astype(np.float64)
            scene = np.full((self.H, self.W), t[2] + 200.0)
            for layer in d[::-1]:
                scene = np.where((layer > 0) & (layer < scene), layer, scene)
            scene += rng.normal(0, 1.0, scene.shape)
            raw = np.round(scene * 10.0).clip(0, 65535).astype(np.uint16)
            raw[rng.random(raw.shape) < 0.02] = 0
            path = os.path.join(self.root, "depth", f"{category}_{i:06d}.png")
            import cv2
            cv2.imwrite(path, raw)
            self.items.append((qi, ri, t, m, path))

    def __len__(self):
        return self.n

    def __getitem__(self, index):
        from .poses import relative_rotation_6d
        qi, ri, t, m, path = self.items[index]
        g = torch.Generator().manual_seed(index)
        return {
            "query": torch.rand(3, 256, 256, generator=g) * 2 - 1,
            "reference": torch.rand(3, 256, 256, generator=g) * 2 - 1,
            "gt_relativeR": relative_rotation_6d(self.R[qi][None], self.R[ri])[0],
            "all_relativeR": relative_rotation_6d(self.R, self.R[ri]),
            "template_poses": torch.from_numpy(self.R.copy()),
            "query_pose": torch.from_numpy(self.R[qi].copy()),
            "query_translation": torch.from_numpy(t.reshape(3, 1).copy()),
            "intrinsic": torch.from_numpy(self.K.copy()),
            "depth_path": path,
            "obj_id": m + 1,
        }
