"""Per-block attribution of the end-to-end fp16 error (test infrastructure: drives the CPU oracle; ~15 min on 8 cores).

    python tools/precision_attribution.py [out.json]

Same rounding model as tests/precision_study.py (fp32 arithmetic, fp16 ROUNDING where the CUDA path stores or feeds fp16),
but the roundings are switched on for ONE block of ONE network at a time (control_model.input_blocks.i, middle_block,
model.diffusion_model.{input_blocks.i, middle_block, output_blocks.i, out}), everything else staying fp32.  Independent
rounding errors add in variance, so err_g^2 is block g's share of the end-to-end error^2; the table says where a
two-term (hi + lo) fp16 split of the tensor-core operands buys the most per GEMM flop.
"""
import json, os, sys, time
import torch, torch.nn.functional as F
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ctrlora_oracle as O, synth
torch.set_num_threads(8)
g = torch.load(os.path.join(ROOT, 'tests', 'golden', 'sd15_rank128_golden.pt'), weights_only=False)
seed = g['seed']
s = synth.synth_state_dict(g['control_shapes'], seed, 'control_model.')
u = synth.synth_state_dict(g['unet_shapes'], seed, 'model.diffusion_model.')
sd = {'control_model.' + k: v for k, v in s.items()}
sd.update({'model.diffusion_model.' + k: v for k, v in u.items()})
x = synth.synth_input('x', (1, 4, 64, 64), seed); hint = synth.synth_input('hint', (1, 4, 64, 64), seed)
ctx = synth.synth_input('ctx', (1, 77, 768), seed); t = g['t']
rel = lambda a, b: ((a.float() - b.float()).norm() / b.float().norm()).item()
q = lambda z: z.half().float()

ACTIVE = {'pred': lambda net, p: False, 'w': True, 'a': True, 'res': True}
FLOPS = {}


def net_of(sd_):
    return 'cn' if 'zero_convs.0.0.weight' in sd_ else 'unet'


def group_of(net, p):
    parts = p.split('.')
    if parts[0] in ('input_blocks', 'output_blocks'):
        return f'{net}.{parts[0]}.{parts[1]}'
    return f'{net}.{parts[0]}'


def on(sd_, p):
    return ACTIVE['pred'](net_of(sd_), p)


def qw(z, a): return q(z) if (a and ACTIVE['w']) else z
def qa(z, a): return q(z) if (a and ACTIVE['a']) else z
def rq(z, a): return q(z) if (a and ACTIVE['res']) else z


RESID_OUT = ('.out_layers.3', '.skip_connection', '.to_out.0', '.net.2', '.proj_out')


def count(sd_, p, flops):
    k = group_of(net_of(sd_), p)
    FLOPS[k] = FLOPS.get(k, 0.0) + flops


def linear(sd_, p, x_, lora_scale=1.0):
    a = on(sd_, p)
    W = sd_[p + '.weight']
    dk = p + '.lora_layer.down.weight'
    if dk in sd_:
        W = W + lora_scale * sd_[p + '.lora_layer.up.weight'] @ sd_[dk]
    count(sd_, p, 2.0 * x_.numel() / x_.shape[-1] * W.numel())
    y = F.linear(qa(x_, a), qw(W, a), sd_.get(p + '.bias'))
    return y if p.endswith(RESID_OUT) else qa(y, a)


def conv(sd_, p, x_, stride=1, padding=0):
    a = on(sd_, p)
    y = F.conv2d(qa(x_, a), qw(sd_[p + '.weight'], a), sd_.get(p + '.bias'), stride=stride, padding=padding)
    count(sd_, p, 2.0 * y.numel() / y.shape[1] * sd_[p + '.weight'].numel())
    return y if p.endswith(RESID_OUT) else qa(y, a)


def group_norm(sd_, p, x_, eps):
    return F.group_norm(qa(x_, on(sd_, p)).float(), 32, sd_[p + '.weight'], sd_[p + '.bias'], eps)


def layer_norm(sd_, p, x_):
    return F.layer_norm(qa(x_, on(sd_, p)), (x_.shape[-1],), sd_[p + '.weight'], sd_[p + '.bias'], 1e-5)


def res_block(sd_, p, x_, emb):
    a = on(sd_, p)
    h = conv(sd_, p + '.in_layers.2', F.silu(group_norm(sd_, p + '.in_layers.0', x_, 1e-5)), padding=1)
    We = sd_[p + '.emb_layers.1.weight']
    if (p + '.emb_layers.1.lora_layer.down.weight') in sd_:
        We = We + sd_[p + '.emb_layers.1.lora_layer.up.weight'] @ sd_[p + '.emb_layers.1.lora_layer.down.weight']
    emb_out = F.linear(F.silu(emb), We, sd_[p + '.emb_layers.1.bias'])
    h = h + emb_out[:, :, None, None]
    h = conv(sd_, p + '.out_layers.3', F.silu(group_norm(sd_, p + '.out_layers.0', h, 1e-5)), padding=1)
    skip = conv(sd_, p + '.skip_connection', x_) if (p + '.skip_connection.weight') in sd_ else x_
    return rq(skip + h, a)


def cross_attention(sd_, p, x_, context, heads):
    a = on(sd_, p)
    c_ = x_ if context is None else context
    qq, k, v = linear(sd_, p + '.to_q', x_), linear(sd_, p + '.to_k', c_), linear(sd_, p + '.to_v', c_)
    b, n, c = qq.shape; d = c // heads
    split = lambda t_: t_.view(b, t_.shape[1], heads, d).permute(0, 2, 1, 3)
    qq, k, v = split(qq), split(k), split(v)
    sim = torch.einsum('bhid,bhjd->bhij', qq, k) * (d ** -0.5)
    pr = qa(sim.softmax(dim=-1), a)
    out = torch.einsum('bhij,bhjd->bhid', pr, v)
    out = qa(out.permute(0, 2, 1, 3).reshape(b, n, c), a)
    return linear(sd_, p + '.to_out.0', out)


def feed_forward(sd_, p, x_):
    a = on(sd_, p)
    W = sd_[p + '.net.0.proj.weight']; bb = sd_[p + '.net.0.proj.bias']
    dk = p + '.net.0.proj.lora_layer.down.weight'
    if dk in sd_:
        W = W + sd_[p + '.net.0.proj.lora_layer.up.weight'] @ sd_[dk]
    count(sd_, p, 2.0 * x_.numel() / x_.shape[-1] * W.numel())
    y = F.linear(qa(x_, a), qw(W, a), bb)
    v, gate = y.chunk(2, dim=-1)
    return linear(sd_, p + '.net.2', qa(v * F.gelu(gate), a))


def transformer_block(sd_, p, x_, context, heads):
    a = on(sd_, p)
    x_ = rq(cross_attention(sd_, p + '.attn1', layer_norm(sd_, p + '.norm1', x_), None, heads) + x_, a)
    x_ = rq(cross_attention(sd_, p + '.attn2', layer_norm(sd_, p + '.norm2', x_), context, heads) + x_, a)
    return rq(feed_forward(sd_, p + '.ff', layer_norm(sd_, p + '.norm3', x_)) + x_, a)


def spatial_transformer(sd_, p, x_, context, heads):
    b, c, h, w = x_.shape
    x_in = x_
    y = conv(sd_, p + '.proj_in', group_norm(sd_, p + '.norm', x_, 1e-6))
    y = y.permute(0, 2, 3, 1).reshape(b, h * w, -1)
    i = 0
    while (p + f'.transformer_blocks.{i}.norm1.weight') in sd_:
        y = transformer_block(sd_, p + f'.transformer_blocks.{i}', y, context, heads); i += 1
    y = y.reshape(b, h, w, -1).permute(0, 3, 1, 2)
    return rq(conv(sd_, p + '.proj_out', y) + x_in, on(sd_, p))


for name in ('linear', 'conv', 'group_norm', 'layer_norm', 'res_block', 'cross_attention', 'feed_forward',
             'transformer_block', 'spatial_transformer'):
    setattr(O, name, globals()[name])


def run():
    with torch.no_grad():
        return O.apply_model(sd, x, t, ctx, hint, 8, 320)


if __name__ == '__main__':
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, 'profiles', 'r2_precision_attribution.json')
    t0 = time.time()
    ref = run()
    flops = dict(FLOPS)
    groups = sorted(flops)
    print('fp32 vs golden', rel(ref, g['eps']), f'{time.time() - t0:.0f}s', len(groups), 'groups', flush=True)
    res = {'groups': {}, 'flops': flops}
    ACTIVE['pred'] = lambda net, p: True
    res['all'] = rel(run(), ref)
    print('all roundings', res['all'], flush=True)
    for kind in ('w', 'a', 'res'):
        ACTIVE.update(w=kind == 'w', a=kind == 'a', res=kind == 'res')
        res['only_' + kind] = rel(run(), ref)
        print('only', kind, res['only_' + kind], flush=True)
    ACTIVE.update(w=True, a=True, res=True)
    for grp in groups:
        ACTIVE['pred'] = lambda net, p, grp=grp: group_of(net, p) == grp
        e = rel(run(), ref)
        res['groups'][grp] = e
        print(f'{grp:40s} err {e:.3e}  var share {e * e / res["all"] ** 2:6.3f}  gemm GF {flops[grp] / 1e9:7.1f}', flush=True)
        json.dump(res, open(out_path, 'w'), indent=1)
    tot = sum(v * v for v in res['groups'].values()) ** 0.5
    print('sqrt(sum var)', tot, 'vs all', res['all'], f'{time.time() - t0:.0f}s')
    res['sqrt_sum_var'] = tot
    json.dump(res, open(out_path, 'w'), indent=1)
