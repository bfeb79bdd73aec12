"""CPU experiment (test tooling, uses the oracle): where does the embedding error of a 16-bit
pipeline come from, and which precision option closes the gap to the 1e-3 bar?

The oracle's UNet.forward is restated with a rounding hook at every point where the CUDA path
stores a 16-bit tensor, matching the FUSED schedule of round 2 (GroupNorm + SiLU + pose bias +
residual applied in the convolution epilogue on the fp32 accumulator, so block convolutions never
round their raw output):

  w      conv / linear weights                (off = "weights exact": fp16 hi + lo K-segments)
  h1     block1 output  SiLU(GN(conv1)) + pose bias
  out    resnet-block output, attention-block output (the residual stream)
  aux    res_conv / down / up-sample conv outputs, GN(1) pre-norm output, qkv, attention core
  pose   SiLU(pose_mlp) and the pose projections

usage: python tools/precision_sim.py [n_hyp] [bf16]
"""
import os
import sys

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import unet_oracle as orc, weights  # noqa: E402

torch.set_num_threads(8)
HEADS, DH = 4, 32


def make_round(dtype):
    return lambda t: t.to(dtype).float()


def forward(sd, x, pose, R, on):
    """on: set of rounding points that are active; R: rounding function."""
    r = lambda key, t: R(t) if key in on else t

    def block(p, x, extra=None, res=None, key="h1"):
        x = F.conv2d(r("cin", x) if key == "h1" else x, sd[f"{p}.proj.weight"], sd[f"{p}.proj.bias"], padding=1)
        x = F.silu(F.group_norm(x, 8, sd[f"{p}.norm.weight"], sd[f"{p}.norm.bias"], eps=1e-5))
        if extra is not None:
            x = x + extra
        if res is not None:
            x = x + res
        return r(key, x)

    def resblock(p, x, c):
        pb = None
        if c is not None and f"{p}.mlp.1.weight" in sd:
            pb = r("pose", F.linear(c, sd[f"{p}.mlp.1.weight"], sd[f"{p}.mlp.1.bias"]))[:, :, None, None]
        h = block(f"{p}.block1", x, extra=pb, key="h1")
        res = x
        if f"{p}.res_conv.weight" in sd:
            res = r("aux", F.conv2d(r("cin", x), sd[f"{p}.res_conv.weight"], sd[f"{p}.res_conv.bias"]))
        return block(f"{p}.block2", h, res=res, key="out")

    def linattn(p, x):
        b, ch, h, w = x.shape
        n = h * w
        y = r("attn", F.group_norm(r("cin", x), 1, sd[f"{p}.fn.norm.weight"], sd[f"{p}.fn.norm.bias"], eps=1e-5))
        qkv = r("attn", F.conv2d(y, sd[f"{p}.fn.fn.to_qkv.weight"]))
        q, k, v = [t.reshape(b, HEADS, DH, n) for t in qkv.chunk(3, dim=1)]
        q = q.softmax(dim=-2) * DH ** -0.5
        k = k.softmax(dim=-1)
        ctx = torch.einsum("bhdn,bhen->bhde", k, v)
        o = r("attn", torch.einsum("bhde,bhdn->bhen", ctx, q).reshape(b, HEADS * DH, h, w))
        o = F.conv2d(o, sd[f"{p}.fn.fn.to_out.0.weight"], sd[f"{p}.fn.fn.to_out.0.bias"])
        o = F.group_norm(o, 1, sd[f"{p}.fn.fn.to_out.1.weight"], sd[f"{p}.fn.fn.to_out.1.bias"], eps=1e-5)
        return r("out", o + x)

    def attn(p, x):
        b, ch, h, w = x.shape
        n = h * w
        y = r("attn", F.group_norm(r("cin", x), 1, sd[f"{p}.fn.norm.weight"], sd[f"{p}.fn.norm.bias"], eps=1e-5))
        qkv = r("attn", F.conv2d(y, sd[f"{p}.fn.fn.to_qkv.weight"]))
        q, k, v = [t.reshape(b, HEADS, DH, n) for t in qkv.chunk(3, dim=1)]
        sim = torch.einsum("bhdi,bhdj->bhij", q * DH ** -0.5, k)
        a = (sim - sim.amax(dim=-1, keepdim=True)).softmax(dim=-1)
        o = torch.einsum("bhij,bhdj->bhid", a, v).permute(0, 1, 3, 2).reshape(b, HEADS * DH, h, w)
        o = F.conv2d(r("attn", o), sd[f"{p}.fn.fn.to_out.weight"], sd[f"{p}.fn.fn.to_out.bias"])
        return r("out", o + x)

    x = r("out", F.conv2d(x, sd["init_conv.weight"], sd["init_conv.bias"], padding=1))
    rr = x
    c = r("pose", F.silu(F.linear(pose, sd["pose_mlp.0.weight"], sd["pose_mlp.0.bias"])))
    hs = []
    for i in range(4):
        x = resblock(f"downs.{i}.0", x, c); hs.append(x)
        x = resblock(f"downs.{i}.1", x, c)
        x = linattn(f"downs.{i}.2", x); hs.append(x)
        if f"downs.{i}.3.1.weight" in sd:
            x = r("aux", orc.hard_downsample(sd, f"downs.{i}.3", r("cin", x)))
        else:
            x = r("aux", F.conv2d(r("cin", x), sd[f"downs.{i}.3.weight"], sd[f"downs.{i}.3.bias"], padding=1))
    for _ in range(2):
        x = resblock("mid_block1", x, c)
        x = attn("mid_attn", x)
        x = resblock("mid_block2", x, c)
    for i in range(4):
        x = resblock(f"ups.{i}.0", torch.cat((x, hs.pop()), 1), c)
        x = resblock(f"ups.{i}.1", torch.cat((x, hs.pop()), 1), c)
        x = linattn(f"ups.{i}.2", x)
        if f"ups.{i}.3.1.weight" in sd:
            x = r("aux", orc.hard_upsample(sd, f"ups.{i}.3", r("cin", x)))
        else:
            x = r("aux", F.conv2d(r("cin", x), sd[f"ups.{i}.3.weight"], sd[f"ups.{i}.3.bias"], padding=1))
    x = resblock("final_res_block", torch.cat((x, rr), 1), c)
    x = resblock("final_conv.0", x, None)
    return F.conv2d(x, sd["final_conv.1.weight"], sd["final_conv.1.bias"])


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 4
    dtype = torch.bfloat16 if "bf16" in sys.argv else torch.float16
    R = make_round(dtype)
    sd = weights.make_unet_state_dict(0)
    g = np.load(os.path.join(ROOT, "tests", "golden", "level2_642_b1.npz"))
    rf = torch.from_numpy(g["ref_feat"])
    poses = torch.from_numpy(g["all_relativeR"])[0]
    pick = torch.linspace(0, 641, n).long()
    x = rf.expand(n, -1, -1, -1)
    big = lambda k, v: v.dim() >= 2 and "final_conv.1" not in k and "init_conv" not in k and "pose_mlp" not in k
    sdq = {k: (R(v) if big(k, v) else v) for k, v in sd.items()}
    with torch.no_grad():
        ref = orc.unet_forward(sd, x, poses[pick])
        chk = forward(sd, x, poses[pick], R, set())
        print("restatement vs oracle:", float((chk - ref).norm() / ref.norm()))

        def err(s, on):
            o = forward(s, x, poses[pick], R, on)
            e = (o - ref).flatten(1).norm(dim=1) / ref.flatten(1).norm(dim=1)
            return float(e.mean()), float(e.max())
        allp = {"h1", "out", "aux", "attn", "pose"}
        rows = [
            ("weights only", sdq, set()),
            ("activations only (all points)", sd, allp),
            ("weights + all activations  [fp16 mode, fused]", sdq, allp),
            ("exact weights + all acts   [hi+lo weights]", sd, allp),
            ("  ... minus out (residual stream exact)", sd, allp - {"out"}),
            ("  ... minus h1", sd, allp - {"h1"}),
            ("  ... minus aux", sd, allp - {"aux"}),
            ("  ... minus pose", sd, allp - {"pose"}),
            ("exact w, skip paths exact (out rounded at conv inputs only)", sd, (allp - {"out"}) | {"cin"}),
            ("fp16 w, skip paths exact", sdq, (allp - {"out"}) | {"cin"}),
            ("exact w, skip exact, aux exact", sd, {"h1", "pose", "cin"}),
            ("exact w, skip exact, h1 exact", sd, {"aux", "pose", "cin"}),
            ("exact w, only attn-internal rounded", sd, {"attn"}),
            ("exact w, attn + pose rounded", sd, {"attn", "pose"}),
            ("exact w, attn + pose + aux(conv) rounded", sd, {"attn", "pose", "aux"}),
            ("exact w, attn + pose + h1 rounded  [parity_fast]", sd, {"attn", "pose", "h1"}),
            ("fp16 w (attn layers only exact?) n/a", sd, set()),
            ("only cin", sd, {"cin"}),
            ("only h1", sd, {"h1"}), ("only out", sd, {"out"}), ("only aux", sd, {"aux"}), ("only pose", sd, {"pose"}),
        ]
        for name, s, on in rows:
            m, mx = err(s, on)
            print(f"{name:50s} mean {m:.3e}  max {mx:.3e}")


if __name__ == "__main__":
    main()
