"""CPU experiment: which fp16 roundings make up the embedding error of the fp16 pipeline?
Runs the oracle with .half().float() inserted at the points where the CUDA path stores fp16
(weights, conv outputs, GroupNorm outputs, residual stream).  Result (2 hypotheses, seed 0):
weights only 9.1e-4, +conv out 1.20e-3, +gn out 1.28e-3, +residual stream 1.43e-3 (the GPU
measures 1.41e-3): fp16 WEIGHT rounding alone is ~0.9e-3 rel-L2, so an fp16 tensor-core UNet
cannot reach 1e-3 on embeddings; scores stay < 1e-3 and the ranking is unchanged."""
import os, sys, torch, numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch.nn.functional as F
from oracle import unet_oracle as orc, weights
torch.set_num_threads(8)
sd = weights.make_unet_state_dict(0)
g=np.load(os.path.join(ROOT, 'tests', 'golden', 'cfg1_b1_n6.npz'))
rf=torch.from_numpy(g['ref_feat']); poses=torch.from_numpy(g['all_relativeR'])[0,:2]
x=rf.expand(2,-1,-1,-1)
ref=orc.unet_forward(sd,x,poses)
h=lambda t:t.half().float()
def run(rw, rconv, rgn, rres, rattn):
    sdq={k:(h(v) if (rw and v.dim()>=2 and 'final_conv.1' not in k and 'init_conv' not in k and 'pose_mlp' not in k) else v) for k,v in sd.items()}
    # monkeypatch oracle pieces
    def block(sd_,p,x,groups=8):
        x=F.conv2d(x,sd_[f"{p}.proj.weight"],sd_[f"{p}.proj.bias"],padding=1)
        if rconv: x=h(x)
        x=F.group_norm(x,groups,sd_[f"{p}.norm.weight"],sd_[f"{p}.norm.bias"],eps=1e-5)
        return F.silu(x)
    def resnet_block(sd_,p,x,emb=None):
        hh=block(sd_,f"{p}.block1",x)
        if emb is not None and f"{p}.mlp.1.weight" in sd_:
            t=F.linear(F.silu(emb),sd_[f"{p}.mlp.1.weight"],sd_[f"{p}.mlp.1.bias"])
            hh=t[:,:,None,None]+hh
        if rgn: hh=h(hh)
        hh=block(sd_,f"{p}.block2",hh)
        if f"{p}.res_conv.weight" in sd_:
            x=F.conv2d(x,sd_[f"{p}.res_conv.weight"],sd_[f"{p}.res_conv.bias"])
            if rconv: x=h(x)
        out=hh+x
        return h(out) if rres else out
    o_block, o_res, o_lin, o_att = orc.block, orc.resnet_block, orc.linear_attention, orc.attention
    def lin(sd_,p,x):
        y=o_lin(sd_,p,x)
        return h(y) if rres else y
    def att(sd_,p,x):
        y=o_att(sd_,p,x)
        return h(y) if rres else y
    orc.block, orc.resnet_block, orc.linear_attention, orc.attention = block, resnet_block, lin, att
    try:
        out=orc.unet_forward(sdq,x,poses)
    finally:
        orc.block, orc.resnet_block, orc.linear_attention, orc.attention = o_block,o_res,o_lin,o_att
    return float((out-ref).norm()/ref.norm())
with torch.no_grad():
    print('weights only        ', run(1,0,0,0,0))
    print('+conv out           ', run(1,1,0,0,0))
    print('+gn out             ', run(1,1,1,0,0))
    print('+residual stream    ', run(1,1,1,1,0))
    print('residual only       ', run(0,0,0,1,0))
    print('conv out only       ', run(0,1,0,0,0))
    print('gn out only         ', run(0,0,1,0,0))
