"""Host-side mirror of the reference task module `PoseConditional`
(src/model/model.py:32-565), inference surface only: forward (loss), sample,
generate_templates, retrieval, plus predict_pose (= eval_geodesic lines 313-357 without
logging, SURVEY.md F2), and the T-LESS evaluation eval_vsd (model.py:378-541) on the GPU renderer and
VSD kernel of nope_b200.vsd.  Training, wandb/video logging are out of scope (SURVEY.md section 8).

Differences that are deliberate and documented:
  * generate_templates batches the whole pose grid through one engine sweep instead of a
    Python loop that re-encodes the reference per pose (model.py:212-222, 115).
  * retrieval raises ValueError for an unknown metric instead of returning None
    (model.py:256 falls through); "cosine" is an extension (SURVEY.md F3).
  * ranking is deterministic: descending score, ties -> lowest index.
  * eval_vsd follows vsd_obj's per-frame contract (vsd.py:58-136); the reference's eval_vsd cannot run as
    written (see nope_b200/vsd.py).  Errors come back in frame order, the GT pose is rendered once per frame.
"""
import ctypes as C
import os
import types

import torch
import torch.nn.functional as F

from . import _lib

_METRICS = {"l2": 0, "cosine": 1, "cosine_occlusion": 2}     # NOPE_METRIC_* of include/nope_b200.h


def _ns(d):
    return d if not isinstance(d, dict) else types.SimpleNamespace(**d)


class PoseConditional:
    def __init__(self, u_net, optim_config=None, testing_config=None, save_dir=None, **kwargs):
        self.u_net = u_net
        self.save_dir = save_dir
        self.optim_config = _ns(optim_config) if optim_config is not None else \
            types.SimpleNamespace(loss_type="l1")
        self.testing_config = _ns(testing_config) if testing_config is not None else \
            types.SimpleNamespace(similarity_metric="l2")
        loss_type = getattr(self.optim_config, "loss_type", "l1")
        self.loss = F.l1_loss if loss_type == "l1" else F.mse_loss
        self.dist = None     # optional nope_b200.dist.ShardedSweep for multi-GPU
        from .metrics import GeodesicError
        self.metric = GeodesicError()              # model.py:56
        self.logged = {}                           # what Lightning's self.log would have received
        self.global_step, self.global_rank = 0, 0

    @property
    def device(self):
        return self.u_net.device

    def eval(self):
        self.u_net.eval()
        return self

    def load_state_dict(self, state_dict, strict=True):
        """Accepts a Lightning checkpoint's `state_dict` (keys prefixed `u_net.`) or a bare
        UNet state_dict."""
        if any(k.startswith("u_net.") for k in state_dict):
            state_dict = {k[len("u_net."):]: v for k, v in state_dict.items()
                          if k.startswith("u_net.")}
        self.u_net.load_state_dict(state_dict, strict=strict)
        return self

    def state_dict(self):
        """Lightning-style keys: every UNet / encoder entry under `u_net.` (model.py:33-40)."""
        return {"u_net." + k: v for k, v in self.u_net.state_dict().items()}

    # ------------------------------------------------------------------ model.py:96-111
    def compute_loss(self, pred, gt):
        loss = self.loss(pred, gt, reduction="none")
        return loss.flatten(1).mean(dim=1).mean()

    @torch.no_grad()
    def forward(self, query, reference, relativeR):
        query_feat = self.u_net.encoder.encode_image(query)
        reference_feat = self.u_net.encoder.encode_image(reference, mode="mode")
        pred = self.u_net(reference_feat, relativeR)
        return self.compute_loss(pred, query_feat)

    __call__ = forward

    # ------------------------------------------------------------------ model.py:113-124
    @torch.no_grad()
    def sample(self, reference, relativeR):
        reference_feat = self.u_net.encoder.encode_image(reference, mode="mode")
        return self.u_net(reference_feat, relativeR), None   # template encoder: no decoder

    # ------------------------------------------------------------------ model.py:193-252
    @torch.no_grad()
    def generate_templates(self, reference, all_relativeR, gt_templates=None, visualize=False):
        reference_feat = self.u_net.encoder.encode_image(reference, mode="mode")
        emb = self.u_net.sweep(reference_feat, all_relativeR, want_emb=True)["emb"]
        return emb, None, None

    # ------------------------------------------------------------------ model.py:254-266
    @torch.no_grad()
    def retrieval(self, query, template_feat, k=5):
        metric = getattr(self.testing_config, "similarity_metric", "l2")
        if metric not in _METRICS:
            raise ValueError(f"unknown similarity_metric {metric!r} (supported: {sorted(_METRICS)})")
        query_feat = self.u_net.encoder.encode_image(query, mode="mode")
        return score_topk(query_feat, template_feat, k=k, metric=metric, threshold=self._occlusion_threshold())

    def _occlusion_threshold(self):
        """`threshold` of the template encoder (OcclusionAwareSimilarity, base_template.py:67-75;
        configs/model/template_base.yaml: 0.2)."""
        return float(getattr(self.u_net.encoder, "threshold", 0.2))

    # ------------------------------------------------------------------ model.py:313-357
    @torch.no_grad()
    def predict_pose(self, query, reference, all_relativeR, template_poses=None, k=5,
                     return_templates=False):
        """-> (R [B,k,3,3] | None, nearest_idx [B,k] int64, similarity [B,N]).  The scores and
        the ranking come out of the sweep's fused last layer; the [B,N,C,32,32] templates are
        only materialised when asked for."""
        metric = getattr(self.testing_config, "similarity_metric", "l2")
        if metric not in _METRICS:
            raise ValueError(f"unknown similarity_metric {metric!r} (supported: {sorted(_METRICS)})")
        enc = self.u_net.encoder
        self.u_net.set_metric(metric, self._occlusion_threshold())     # scored in the sweep's last layer
        B = query.shape[0]
        feats = enc.encode_image(torch.cat([query.to(self.device), reference.to(self.device)]))
        query_feat, reference_feat = feats[:B], feats[B:]
        N = all_relativeR.shape[1]
        k = min(k, N)
        if self.dist is not None:
            sim, topi, emb = self.dist.sweep(self.u_net, reference_feat, all_relativeR, query_feat,
                                             k=k, metric=metric, want_emb=return_templates,
                                             threshold=self._occlusion_threshold())
        else:
            out = self.u_net.sweep(reference_feat, all_relativeR, query_feat=query_feat,
                                   want_emb=return_templates, k=k)
            sim, topi, emb = out["sim"], out["topi"], out["emb"]
        R = None
        if template_poses is not None:
            tp = template_poses[0] if template_poses.dim() == 4 else template_poses
            R = tp.to(topi.device)[topi]          # model.py:352-354
        if return_templates:
            # under sharding `emb` is (local templates, lo, hi): each rank keeps only its slice
            return R, topi, sim, emb
        return R, topi, sim


    # ------------------------------------------------------------------ model.py:185-191, 268-376, 550-565
    def log(self, name, value, **kwargs):
        self.logged.setdefault(name, []).append(float(value))

    def log_score(self, dict_scores, split_name):
        for key, value in dict_scores.items():
            self.log(f"{key}/{split_name}", value, sync_dist=True)

    @torch.no_grad()
    def eval_geodesic(self, batch, data_name, visualize=False, save_prediction=False):
        """`eval_geodesic` of the reference without the wandb / image logging (the template encoder has
        no decoder, so the reference itself sets visualize=False on this path, model.py:269-274):
        validation loss under the ground-truth pose, template sweep + retrieval, geodesic accuracy."""
        query, reference = batch["query"], batch["reference"]
        loss = self.forward(query=query, relativeR=batch["gt_relativeR"], reference=reference)
        self.log(f"loss/val_{data_name}", loss)
        template_poses = batch["template_poses"][0]
        predR, nearest_idx, similarity = self.predict_pose(query, reference, batch["all_relativeR"],
                                                           template_poses, k=5)
        error, acc = self.metric(predR=predR, gtR=batch["query_pose"].to(predR.device),
                                 symmetry=batch["symmetry"].reshape(-1).to(predR.device))
        self.log_score(acc, split_name=f"val_{data_name}")
        if save_prediction and self.save_dir is not None:
            import os
            import numpy as np
            os.makedirs(os.path.join(self.save_dir, "predictions"), exist_ok=True)
            np.savez(os.path.join(self.save_dir, "predictions",
                                  f"pred_{data_name}_step{self.global_step}_rank{self.global_rank}"),
                     query_pose=batch["query_pose"].cpu().numpy(), similarity=similarity.cpu().numpy(),
                     nearest_idx=nearest_idx.cpu().numpy())
        return error, nearest_idx, similarity

    # ------------------------------------------------------------------ model.py:378-389
    def load_mesh(self, cad_dir, obj_ids=range(1, 31)):
        """The T-LESS CAD models obj_000001.ply ... obj_000030.ply (mm), packed on the model's device."""
        from .vsd import MeshTable
        self.tless_obj_ids = list(obj_ids)
        self.tless_cad = MeshTable([os.path.join(cad_dir, f"obj_{i:06d}.ply") for i in self.tless_obj_ids],
                                   device=self.device)
        return self

    # ------------------------------------------------------------------ model.py:391-541
    @torch.no_grad()
    def eval_vsd(self, batch, data_name, save_path=None):
        """`eval_vsd` of the reference without the wandb / image logging and the process pool: validation
        loss, top-5 retrieval (through ShardedSweep when set; every rank then computes the same VSD),
        predicted poses = retrieved rotations with the GT translation, 1 + k depth renders per frame, VSD
        errors [B,k] (float64), the scores of model.py:530-537.  Saves vsd_error[:, 0] to `save_path`."""
        import numpy as np
        from .vsd import render_depth, vsd_error, vsd_scores
        if getattr(self, "tless_cad", None) is None:
            raise RuntimeError("eval_vsd needs the CAD models: call load_mesh(cad_dir) first")
        query, reference = batch["query"], batch["reference"]
        loss = self.forward(query=query, relativeR=batch["gt_relativeR"], reference=reference)
        self.log(f"loss/val_{data_name}", loss)
        _, nearest_idx, _ = self.predict_pose(query, reference, batch["all_relativeR"], None, k=5)
        dev = nearest_idx.device
        B, k = nearest_idx.shape
        tp = batch["template_poses"].to(dev)
        retrieved_R = tp[torch.arange(B, device=dev)[:, None].expand(B, k), nearest_idx]   # model.py:469-475
        t = batch["query_translation"].to(dev, torch.float32).reshape(B, 3, 1)
        gt = torch.cat([batch["query_pose"].to(dev, torch.float32), t], dim=2)           # [B,3,4]
        pred = torch.cat([retrieved_R.to(torch.float32), t[:, None].expand(B, k, 3, 1)], dim=3)
        obj_ids = [int(i) for i in torch.as_tensor(batch["obj_id"]).reshape(-1).tolist()]
        try:
            mesh_idx = [self.tless_obj_ids.index(i) for i in obj_ids]
        except ValueError:
            raise ValueError(f"obj_id {obj_ids} not among the loaded meshes {self.tless_obj_ids}") from None
        if "depth_raw" in batch:
            depth_raw = batch["depth_raw"].to(dev)
        else:
            from .tless import read_depth
            depth_raw = read_depth(batch["depth_path"]).to(dev)
        H, W = depth_raw.shape[-2:]
        K = batch["intrinsic"].to(dev)
        poses = torch.cat([gt[:, None], pred], dim=1).reshape(B * (1 + k), 3, 4)
        ids = [m for m in mesh_idx for _ in range(1 + k)]
        depth = render_depth(self.tless_cad, ids, poses, K.double().repeat_interleave(1 + k, 0), H, W)
        depth = depth.view(B, 1 + k, H, W)
        err = vsd_error(depth_raw, K.double(), depth[:, 0], depth[:, 1:])
        scores = vsd_scores(err)
        self.log_score(scores, split_name=f"val_{data_name}")
        err = err.cpu().numpy()
        if save_path is not None:
            os.makedirs(os.path.dirname(os.path.abspath(save_path)), exist_ok=True)
            np.save(save_path, err[:, 0])
        self.last_vsd_error = err
        return scores

    def test_step(self, batch, idx_batch):
        """model.py:550-565: one entry per dataloader, keyed "<dataset>_<category>"."""
        out = {}
        for dataloader_name in batch.keys():
            data_name, category = dataloader_name.split("_")
            if data_name in ["tless"]:
                save_path = None if self.save_dir is None else os.path.join(
                    self.save_dir, "predictions", f"vsd_{category}_batch{idx_batch}_rank_{self.global_rank}.npy")
                out[dataloader_name] = self.eval_vsd(batch[dataloader_name], category, save_path=save_path)
                continue
            out[dataloader_name] = self.eval_geodesic(batch[dataloader_name], category, visualize=True,
                                                      save_prediction=True)
        self.global_step += 1
        return out


def score_topk(query_feat, template_feat, k=5, metric="l2", idx_base=0, threshold=0.2):
    """similarity [B,N] and nearest_idx [B,k] of materialised templates
    (the arithmetic of model.py:260-265) on the GPU."""
    if metric not in _METRICS:
        raise ValueError(f"unknown similarity_metric {metric!r} (supported: {sorted(_METRICS)})")
    lib = _lib.load()
    dev = template_feat.device
    if dev.type != "cuda":
        raise _lib.NopeError("score_topk needs CUDA tensors (no CPU fallback)")
    q = query_feat.to(dev, torch.float32).contiguous()
    t = template_feat.to(torch.float32).contiguous()
    B, N, Cc = t.shape[0], t.shape[1], t.shape[2]
    hw = t.shape[3] * t.shape[4]
    if k > N:
        raise RuntimeError(f"selected index k out of range (k={k}, N={N})")  # torch.topk's error
    sim = torch.empty((B, N), device=dev, dtype=torch.float32)
    topv = torch.empty((B, k), device=dev, dtype=torch.float32)
    topi = torch.empty((B, k), device=dev, dtype=torch.int64)
    with torch.cuda.device(dev):
        _lib.check(lib.nope_score_topk(_lib.ptr(q), _lib.ptr(t), B, N, Cc, hw, _METRICS[metric], float(threshold), k,
                                       _lib.ptr(sim), _lib.ptr(topv), _lib.ptr(topi), idx_base,
                                       C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
    return sim, topi


def topk(sim, k, idx_base=0):
    """Deterministic top-k of sim [B,N] on the GPU (descending, ties -> lowest index)."""
    lib = _lib.load()
    sim = sim.contiguous()
    B, N = sim.shape
    topv = torch.empty((B, k), device=sim.device, dtype=torch.float32)
    topi = torch.empty((B, k), device=sim.device, dtype=torch.int64)
    with torch.cuda.device(sim.device):
        _lib.check(lib.nope_topk(_lib.ptr(sim), B, N, k, _lib.ptr(topv), _lib.ptr(topi), idx_base,
                                 C.c_void_p(torch.cuda.current_stream(sim.device).cuda_stream)))
    return topv, topi


def build_model(u_net_dim=192, descriptor_size=8, device="cuda:0", chunk=642,
                similarity_metric="l2", precision="fp16"):
    """The one configuration the reference resolves: configs/model/template_base.yaml.
    precision: "fp16" (fast), "fp16_w2" (exact weights), "parity" (split precision, meets the
    1e-3 embedding tolerance of the fp32 reference with margin: 2.2e-4), "parity_fast" (the same with single-fp16
    tensors inside the ResnetBlocks: ~5e-4, 15 % faster) or "bf16" (BASELINE configs[2]: bf16 storage, ~1e-2)."""
    from .encoder import FeatureExtractor
    from .unet import UNet
    enc = FeatureExtractor(descriptor_size=descriptor_size, threshold=0.2, normalize=False)
    unet = UNet(u_net_dim=u_net_dim, rot_representation_dim=6, encoder=enc,
                pose_mlp_name="single_layer", device=device, chunk=chunk, precision=precision)
    return PoseConditional(unet, optim_config={"loss_type": "l1"},
                           testing_config={"similarity_metric": similarity_metric}, save_dir=None)
