"""Float64 references of the single layers of the CascadedNet forward, and the per-layer gates they are held to.

Each function computes ONE operation of the reference model (lib/layers.py, lib/nets.py) in float64 from the
state_dict as the checkpoint stores it: BatchNorm is applied unfolded (eval mode) after a bias-free convolution, as in
oracle/net_oracle.py, never through the folded weights the native library packs at load time.  The tensors may live
on any torch device; tests/test_gpu_layers.py feeds each function the native forward's own read-back input of the
layer (teacher forcing), tests/test_layer_reference.py chains them on their own outputs and calibrates the gates.
"""
import numpy as np
import torch
import torch.nn.functional as F

from oracle import net_oracle

NETS = ('stg1_low_band_net.0', 'stg1_high_band_net', 'stg2_low_band_net.0', 'stg2_high_band_net', 'stg3_full_band_net')
SHORT = ('stg1_low', 'stg1_high', 'stg2_low', 'stg2_high', 'stg3')
ASPP_DILATIONS = ((4, 2), (8, 4), (12, 6))   # lib/nets.py:10

# Gates, as max|got - ref| / max|ref| unless stated otherwise.  Split-bf16 storage alone is 2^-17 ~ 7.6e-6 relative;
# a convolution that drops one of its three bf16 products is off by ~2^-9 ~ 2e-3, 40x above GATE_CONV.
GATE_CONV = 5e-5      # every convolution / decoder output and every materialised upsample / pool slice
GATE_LSTM = 1e-5      # fp32 LSTM planes; absolute on the hidden states (tanh outputs)
GATE_L0 = 3e-5        # LSTM 1x1 input convolution, per pixel, relative to sum_c |w_c| |d2_c|
GATE_MASK = 4e-6      # sigmoid mask, absolute: the fp32 sum of nout products for a logit up to |z| ~ 20 alone reaches 1e-6


def state_dict64(sd, device='cpu'):
    """{key: float64 tensor on device} (int64 BatchNorm counters are dropped: nothing reads them)."""
    out = {}
    for k, v in sd.items():
        t = v if torch.is_tensor(v) else torch.from_numpy(np.asarray(v))
        if t.is_floating_point():
            out[k] = t.to(device=device, dtype=torch.float64)
    return out


def rel_err(got, ref):
    """max|got - ref| / max|ref| (max|ref| floored at 1e-30)."""
    got, ref = got.to(torch.float64), ref.to(torch.float64)
    return ((got - ref).abs().max() / ref.abs().max().clamp_min(1e-30)).item()


def abs_err(got, ref):
    return (got.to(torch.float64) - ref.to(torch.float64)).abs().max().item()


def conv(sd, p, x, stride=1, pad=1, dil=1, act='relu'):
    """Conv2DBNActiv (lib/layers.py:8-26) at state_dict prefix p."""
    return net_oracle.conv_bn_act(sd, p, x, stride=stride, pad=pad, dil=dil, act=act)


def upsample(x):
    """lib/layers.py:52: bilinear x2, align_corners=True."""
    return F.interpolate(x, scale_factor=2, mode='bilinear', align_corners=True)


def enc_conv1(sd, p, x):
    return conv(sd, p, x, stride=2, act='leaky')


def enc_conv2(sd, p, x):
    return conv(sd, p, x, act='leaky')


def aspp_pool(x):
    """AdaptiveAvgPool2d((1, None)) (lib/layers.py:71)."""
    return x.mean(dim=2, keepdim=True)


def aspp_branch(sd, p, i, x):
    """Branch i (1 = pooled 1x1, 2 = 1x1, 3..5 = dilated 3x3) of ASPPModule at prefix p (lib/layers.py:92-105)."""
    if i == 1:
        return conv(sd, p + '.conv1.1', x, pad=0)
    if i == 2:
        return conv(sd, p + '.conv2', x, pad=0)
    d = ASPP_DILATIONS[i - 3]
    return conv(sd, '%s.conv%d' % (p, i), x, pad=d, dil=d)


def decoder(sd, p, low, skip):
    """Decoder (lib/layers.py:51-64): conv(cat[up(low), skip]); the widths of this net always match (no crop)."""
    return conv(sd, p + '.conv1', torch.cat([upsample(low), skip], 1))


# ---- LSTM branch (lib/layers.py:108-133) in the layouts of the native planes ----------------------------------------
def lstm_conv_weight(sd, p):
    """BatchNorm-folded weight [C] and bias of the branch's 1x1 input convolution (2n -> 1)."""
    scale = sd[p + '.conv.conv.1.weight'] / torch.sqrt(sd[p + '.conv.conv.1.running_var'] + net_oracle.BN_EPS)
    w = sd[p + '.conv.conv.0.weight'].reshape(-1) * scale
    b = sd[p + '.conv.conv.1.bias'] - sd[p + '.conv.conv.1.running_mean'] * scale
    return w, b


def lstm_l0(sd, p, h):
    """Pre-activation sums of the 1x1 convolution, [N, bins, T] from h [N, 2n, bins, T]; also sum_c |w_c| |h_c|."""
    w, _ = lstm_conv_weight(sd, p)
    return torch.einsum('c,nchw->nhw', w, h), torch.einsum('c,nchw->nhw', w.abs(), h.abs())


def lstm_xp(sd, p, l0):
    """Gate pre-activations [N, T, 8*hid] (forward direction's i, f, g, o, then the reverse direction's) of
    relu(l0 + folded BN bias) [N, bins, T]."""
    _, b = lstm_conv_weight(sd, p)
    a = torch.relu(l0 + b).transpose(1, 2)
    outs = []
    for sfx in ('', '_reverse'):
        w = sd['%s.lstm.weight_ih_l0%s' % (p, sfx)]
        outs.append(a @ w.t() + sd['%s.lstm.bias_ih_l0%s' % (p, sfx)] + sd['%s.lstm.bias_hh_l0%s' % (p, sfx)])
    return torch.cat(outs, 2)


def lstm_direction(xp, whh, reverse):
    """One direction of nn.LSTM over xp [N, T, 4*hid] (gate order i, f, g, o) from zero state: h [N, T, hid]."""
    N, T, g4 = xp.shape
    hid = g4 // 4
    h = xp.new_zeros(N, hid)
    c = xp.new_zeros(N, hid)
    out = xp.new_empty(N, T, hid)
    for t in (range(T - 1, -1, -1) if reverse else range(T)):
        g = xp[:, t] + h @ whh.t()
        i, f, gg, o = torch.sigmoid(g[:, :hid]), torch.sigmoid(g[:, hid:2 * hid]), torch.tanh(g[:, 2 * hid:3 * hid]), \
            torch.sigmoid(g[:, 3 * hid:])
        c = f * c + i * gg
        h = o * torch.tanh(c)
        out[:, t] = h
    return out


def lstm_hs(sd, p, xp):
    """Hidden states [N, T, 2*hid] (forward, then reverse) from the gate pre-activations xp [N, T, 8*hid]."""
    g4 = xp.shape[2] // 2
    return torch.cat([lstm_direction(xp[:, :, :g4], sd[p + '.lstm.weight_hh_l0'], False),
                      lstm_direction(xp[:, :, g4:], sd[p + '.lstm.weight_hh_l0_reverse'], True)], 2)


def lstm_y(sd, p, hs):
    """Linear + BatchNorm1d(eval) + ReLU of hs [N, T, 2*hid] -> the branch output plane [bins, N, T]."""
    y = hs @ sd[p + '.dense.0.weight'].t() + sd[p + '.dense.0.bias']
    y = (y - sd[p + '.dense.1.running_mean']) / torch.sqrt(sd[p + '.dense.1.running_var'] + net_oracle.BN_EPS)
    y = torch.relu(y * sd[p + '.dense.1.weight'] + sd[p + '.dense.1.bias'])
    return y.permute(2, 0, 1)


def mask_out(sd, f3):
    """lib/nets.py:79,109-115: sigmoid(out(f3)), the last frequency row replicated once (bins = max_bin + 1)."""
    m = torch.sigmoid(torch.einsum('oc,nchw->nohw', sd['out.weight'][:, :, 0, 0], f3))
    return torch.cat([m, m[:, :, -1:]], 2)


# ---- the whole net chained on its own outputs ------------------------------------------------------------------------
def basenet(sd, p, x):
    """BaseNet (lib/nets.py:26-41) from the single-layer references above."""
    e = [conv(sd, p + '.enc1', x)]
    for k in (2, 3, 4, 5):
        e.append(enc_conv2(sd, '%s.enc%d.conv2' % (p, k), enc_conv1(sd, '%s.enc%d.conv1' % (p, k), e[-1])))
    e5 = e[-1]
    f1 = aspp_branch(sd, p + '.aspp', 1, aspp_pool(e5)).expand(-1, -1, e5.shape[2], -1)
    feats = [f1] + [aspp_branch(sd, p + '.aspp', i, e5) for i in (2, 3, 4, 5)]
    h = conv(sd, p + '.aspp.bottleneck', torch.cat(feats, 1), pad=0)
    h = decoder(sd, p + '.dec4', h, e[3])
    h = decoder(sd, p + '.dec3', h, e[2])
    h = decoder(sd, p + '.dec2', h, e[1])
    lp = p + '.lstm_dec2'
    y = lstm_y(sd, lp, lstm_hs(sd, lp, lstm_xp(sd, lp, lstm_l0(sd, lp, h)[0])))
    return decoder(sd, p + '.dec1', torch.cat([h, y.permute(1, 0, 2)[:, None]], 1), e[0])


def forward_stages(sd, x):
    """lib/nets.py:82-117 on x [N, 2, bins, W]: the stage activations l1, h1, l2, h2, f3 and the mask."""
    x = x[:, :, :x.shape[2] - 1]
    hb = x.shape[2] // 2
    l1_in, h1_in = x[:, :, :hb], x[:, :, hb:]
    l1 = conv(sd, 'stg1_low_band_net.1', basenet(sd, NETS[0], l1_in), pad=0)
    h1 = basenet(sd, NETS[1], h1_in)
    l2 = conv(sd, 'stg2_low_band_net.1', basenet(sd, NETS[2], torch.cat([l1_in, l1], 1)), pad=0)
    h2 = basenet(sd, NETS[3], torch.cat([h1_in, h1], 1))
    f3 = basenet(sd, NETS[4], torch.cat([x, torch.cat([l1, h1], 2), torch.cat([l2, h2], 2)], 1))
    return dict(l1=l1, h1=h1, l2=l2, h2=h2, f3=f3, mask=mask_out(sd, f3))
