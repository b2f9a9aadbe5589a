"""CPU study behind the tensor-core training kernel's numerics (csrc/train_tc.cuh): the reference's training step
(oracle/restatement.py, autograd) with feature_nn's GEMMs replaced by emulations of what the tensor core computes --
3xTF32 row GEMMs, and four candidates for the weight-gradient GEMMs dW = g^T h:
  3term   hi/lo split of both operands (three tf32 passes)
  2term   g split, h rounded to nearest tf32
  1term   ONE pass, both operands rounded to nearest (what the kernel does: operands stored as bits + 0x1000)
  trunc2  g split, h truncated (what the hardware does to a raw fp32 operand: biased)
Prints max |grad - reference| / max |reference| on the three golden steps (B = 64) and on a B = 2000 batch.
Test infrastructure only (imports oracle/).  Run:  python tools/dw_precision.py"""
import sys, json, numpy as np, torch
sys.path.insert(0, __import__('os').path.dirname(__import__('os').path.dirname(__import__('os').path.abspath(__file__))))
from oracle import restatement as R
from bnn_chaos_model_b200 import synth
torch.set_num_threads(8)

def rn_tf32(x):
    b = x.contiguous().view(torch.int32)
    return ((b + 0x1000) & ~0x1FFF).view(torch.float32)
def trunc_tf32(x):
    return (x.contiguous().view(torch.int32) & ~0x1FFF).view(torch.float32)
def split(x):
    hi = rn_tf32(x); lo = trunc_tf32(x - hi)   # hardware truncates the lo operand
    return hi, lo
def mm3(a, b):  # a[M,K] @ b[K,N], 3xTF32
    ah, al = split(a); bh, bl = split(b)
    return (al.double()@bh.double() + ah.double()@bl.double() + ah.double()@bh.double()).float()

def mm2(a, b):  # a rounded to nearest tf32 (single), b split: a_hi b_lo + a_hi b_hi
    ah = rn_tf32(a); bh, bl = split(b)
    return (ah.double()@bl.double() + ah.double()@bh.double()).float()

MODE = {'dw': '2term', 'bwd': '3term'}
class TCLinear(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, W, b):
        ctx.save_for_backward(x, W)
        shp = x.shape
        y = mm3(x.reshape(-1, shp[-1]), W.t().contiguous()) + b
        return y.reshape(*shp[:-1], W.shape[0])
    @staticmethod
    def backward(ctx, g):
        x, W = ctx.saved_tensors
        g2 = g.reshape(-1, g.shape[-1]); x2 = x.reshape(-1, x.shape[-1])
        gx = (mm2(g2, W) if MODE.get('bwd') == '2term' else mm3(g2, W)).reshape(x.shape)
        gh, gl = split(g2)
        if MODE['dw'] == '2term':
            xh = rn_tf32(x2)
            dW = (gh.double().t()@xh.double() + gl.double().t()@xh.double()).float()
        elif MODE['dw'] == '1term':
            dW = (gh.double().t()@rn_tf32(x2).double()).float()
        elif MODE['dw'] == '3term':
            xh, xl = split(x2)
            dW = (gl.double().t()@xh.double() + gh.double().t()@xl.double() + gh.double().t()@xh.double()).float()
        elif MODE['dw'] == 'trunc2':
            xh = trunc_tf32(x2)
            dW = ((gh+gl).double().t()@xh.double()).float()
        db = g2.sum(0)
        return gx, dW, db

def feature_nn_tc(spec, p, x):
    for i in range(3):
        x = TCLinear.apply(x, p[f"feature_nn.{2*i}.weight"], p[f"feature_nn.{2*i}.bias"])
        if i < 2: x = torch.relu(x)
    return x

def grad_with(spec, theta, x, y, e_in, e1, e2, es, tc):
    th = theta.clone().requires_grad_(True)
    orig = R.feature_nn
    if tc: R.feature_nn = feature_nn_tc
    try:
        total, logs = R.training_loss(spec, th, x, y, e_in, e1, e2, es)
        (g,) = torch.autograd.grad(total, th)
    finally:
        R.feature_nn = orig
    return float(total), g

z = np.load(__import__('os').path.join(__import__('os').path.dirname(__import__('os').path.dirname(__import__('os').path.abspath(__file__))), 'tests', 'golden', 'train_v50.npz'))
st = np.load(__import__('os').path.join(__import__('os').path.dirname(__import__('os').path.dirname(__import__('os').path.abspath(__file__))), 'tests', 'golden', 'swag_v50_seed0.npz'))
hp = json.loads(str(st['hparams']))
spec = R.ModelSpec.from_hparams(hp)
B = int(z['B'])
x = torch.from_numpy(synth.make_systems(B, seed=int(z['x_seed'])))
y = torch.from_numpy(z['y'])
theta = torch.from_numpy(z['theta0'])
for step in range(3):
    e_in = torch.from_numpy(np.load(__import__('os').path.join(__import__('os').path.dirname(__import__('os').path.dirname(__import__('os').path.abspath(__file__))), 'tests', 'golden', f'train_v50_eps_in{step}.npz'))['eps_in'].astype(np.float32))
    e12 = torch.from_numpy(z['eps12'][step]); es = torch.from_numpy(z['eps_sum'][step])
    th = theta if step == 0 else torch.from_numpy(z[f'theta_ref_{step-1}'])
    gref = torch.from_numpy(z[f'grad_ref_{step}'])
    l0, g0 = grad_with(spec, th, x, y, e_in, e12[:, :20], e12[:, 20:], es, False)
    print(f"step {step}: fp32 restatement vs golden: {float((g0-gref).abs().max()/gref.abs().max()):.2e}  loss {l0} vs {float(z[f'loss_ref_{step}'])}")
    for mode in ('3term', '2term', 'trunc2', '1term', '1term+bwd2'):
        MODE['dw'] = mode.split('+')[0]; MODE['bwd'] = '2term' if '+' in mode else '3term'
        l1, g1 = grad_with(spec, th, x, y, e_in, e12[:, :20], e12[:, 20:], es, True)
        print(f"   {mode}: grad err/max {float((g1-gref).abs().max()/gref.abs().max()):.2e}  loss rel {abs(l1-l0)/abs(l0):.2e}")
# B = 2000
B = 2000
x = torch.from_numpy(synth.make_systems(B, seed=5)); y = torch.from_numpy(synth.make_labels(B, seed=5))
g = torch.Generator().manual_seed(1)
e_in = torch.randn(x.shape, generator=g); e12 = torch.randn((B, 40), generator=g); es = torch.randn((B, 40), generator=g)
theta = torch.from_numpy(st['w_avg'])
l0, g0 = grad_with(spec, theta.double() if False else theta, x, y, e_in, e12[:, :20], e12[:, 20:], es, False)
for mode in ('3term', '2term', 'trunc2', '1term', '1term+bwd2'):
    MODE['dw'] = mode.split('+')[0]; MODE['bwd'] = '2term' if '+' in mode else '3term'
    l1, g1 = grad_with(spec, theta, x, y, e_in, e12[:, :20], e12[:, 20:], es, True)
    print(f"B=2000 {mode}: grad err/max {float((g1-g0).abs().max()/g0.abs().max()):.2e}  loss rel {abs(l1-l0)/abs(l0):.2e}")
