"""How sensitive are the layer-golden gradients to bf16 rounding?  Runs the fp32 oracle with the
block boundaries (and the 2-D weights) rounded to bf16 and prints the deviation from the reference
golden per quantity.  CPU only."""
import os, sys, numpy as np, torch
ROOT=os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0,ROOT)
from oracle import swin_oracle as so, make_goldens as mg
c=mg.LAYER_CASE; H,W=c["res"]
g=np.load(os.path.join(ROOT,'tests','golden','swin_layer.npz'))
params=so.make_layer_params(c["dim"],c["res"],c["heads"],c["seed"])
def rnd(x): return x + (x.bfloat16().float()-x).detach()
orig_block=so.swin_block
def noisy_block(x,p,*a,**k):
    return rnd(orig_block(rnd(x),p,*a,**k))
so.swin_block=noisy_block
leaf={k:(v.clone().requires_grad_(True) if v.is_floating_point() and not k.endswith("attn_mask") else v) for k,v in params.items()}
# also round weights to bf16 like the kernels do
leafr={k:(rnd(v) if (v.is_floating_point() and v.dim()==2 and 'table' not in k and v.requires_grad) else v) for k,v in leaf.items()}
x=so.make_features(61,c["B"],4,c["dim"],H,W).requires_grad_(True)
w1=so.make_features(62,c["B"],4,c["dim"],H,W)-0.4
w2=so.make_features(63,c["B"],4,2*c["dim"],H//2,W//2)-0.4
y1,y2=so.swin_layer_v5(x,leafr,c["dim"],c["res"],c["heads"])
((y1*w1).sum()+(y2*w2).sum()).backward()
def err(a,b):
    a=a.detach().double(); b=torch.as_tensor(b).double(); return float((a-b).abs().max()/b.abs().max())
print('y1',err(y1,g['y1']),'dx',err(x.grad,g['dx']))
for n in ["layers.0.0.attn.relative_position_bias_table","layers.1.1.attn.relative_position_bias_table","layers.4.1.attn.relative_position_bias_table","layers.2.1.norm1.weight","downsample.norm.weight"]:
    print(n, err(leaf[n].grad, g['d_'+n]))
