"""fp64 value and per-element forward-error scale of one spatio-temporal block.

Test infrastructure only.  ``block(x, sd, key, spec, pad)`` returns ``(value, mag)`` for the block that
``regular.st_block`` computes: ``value`` is that function evaluated in float64, ``mag`` the same graph of
operations evaluated on magnitudes -- every BatchNorm folded into its conv in float64, then ``|W|``, ``|bias|``,
``|mixing coefficients|`` and ``|x|``, with no ReLU (ReLU is 1-Lipschitz, so it never enlarges an error).  A
kernel result ``got`` of the block is accepted element by element when

    |got - value| <= EPS * mag + TINY

Derivation of EPS (split-bf16 arithmetic of the kernels, per block of two stages: graph conv, temporal conv)
--------------------------------------------------------------------------------------------------------
Every operand a of a tensor-core GEMM is held as hi = bf16(a), lo = bf16(a - hi) (bf16: 8 significant bits).
For a in [2^e, 2^(e+1)) the first rounding leaves |a - hi| <= 2^(e-8); that residual is < 2^(e-8) unless it
is exactly representable, so the second rounding leaves |a - hi - lo| <= 2^(e-17) <= 2^-17 |a|.  Each product
is formed as hi*hi + lo*hi + hi*lo; the dropped lo*lo is at most 2^-8 |w| * 2^-8 |x| per product in the worst
case, and over the K products of one output (independent mantissas) its sum stays below 2^-18 sum |w||x|,
the figure used here.  Per stage, relative to sum |w||x| (the stage's share of ``mag``):

    activation operand split      2^-17   (the store of the previous stage; the input frame for stage 1)
    weight split                  2^-17
    dropped lo*lo                 2^-18
    fp32 accumulation             sqrt(K) * 2^-24, K <= 9 * 256 + 256 = 2560 -> 2^-18.3
    split-bf16 store of the result 2^-17   (becomes the next stage's activation split)

The input split is counted once and each store once, so one block is
    2^-17 * (1 + 2 * (1 + 0.5 + 0.39 + 1)) = 6.78 * 2^-17 = 2^-14.24,
since the graph conv's error enters the temporal conv through |W_t| and is covered by the temporal stage's
``mag``, which is built from the graph conv's ``mag``.  That sum treats every product's rounding error as if they
all had the same sign.  They are independent and of either sign, so over the K >= 64 products of a tensor-core
output their sum concentrates: the probabilistic bound lambda * u * ||t||_2 (Higham & Mary, 2019) with terms of
similar size is lambda / sqrt(K) of the worst case, 1/4 for K = 64 and lambda = 2.  Hence
    EPS = 2^-14.24 / 4 ~= 2^-16.
This is a high-probability bound, not a strict one; tests/test_error_bound_cpu.py checks on an emulation of the
kernels' arithmetic that correct arithmetic stays 4x inside it and that the faults a kernel could have break it.
The SIMT kernels multiply the same split operands in fp32 against fp32 weights, which is no less accurate.

Softmax stages (adaptive graph conv, attention unit).  The attention weights S are computed from GEMM results
whose error moves the softmax argument; that error is not bounded analytically here.  Instead S is taken to
carry a relative error of at most SOFTMAX_REL * EPS, an empirical constant: the mixing (or S @ v) stage then
contributes SOFTMAX_REL * EPS * (|x| @ S) on top of its own terms, i.e. ``mag`` uses (|adj + S| + SOFTMAX_REL * S).

What the bound cannot see
-------------------------
* A small error in one mixing coefficient.  One coefficient off by 2^-10 relative moves the outputs by 0.2-0.5 of the
  bound, because that term is diluted over three partitions, nine taps and the residual.  All coefficients rounded to
  bf16 (2^-9) do break it, by 1.8-2.6x (tests/test_error_bound_cpu.py).
* Precision faults inside the attention unit.  Its ``mag`` is about 50x looser than for a plain block: the
  (1 + SOFTMAX_REL) factor and the cancellation inside the softmax-weighted sum S @ v.  No emulation shows that a
  dropped product in k_tc_sa or k_sa_attn would exceed it.  For attention units the bound is a coarse check: it
  catches wrong rows, heads or tokens, not last-bit arithmetic.
* Chained through a whole stack (``model``), the magnitudes compound from block to block, so that check is coarse as
  well.  A whole model is held tightly by checking each block on the previous block's actual output (``block``) and
  the logits on the last block's actual outputs (``head``), as tests/test_gpu_models.py does.
"""
import torch
import torch.nn.functional as F

from . import regular

EPS = 2.0 ** -16
TINY = 1e-30
SOFTMAX_REL = 4.0


def _folded(sd, conv_key, bn_key):
    """BN folded into the conv in float64: (W (cout, cin, k, 1), b (cout,))."""
    s = sd[bn_key + "weight"].double() / torch.sqrt(sd[bn_key + "running_var"].double() + regular.BN_EPS)
    t = sd[bn_key + "bias"].double() - sd[bn_key + "running_mean"].double() * s
    w = sd[conv_key + "weight"].double() * s[:, None, None, None]
    return w, s * sd[conv_key + "bias"].double() + t, s


def _mconv(xm, w, b, stride=1, pad=0):
    return F.conv2d(xm, w.abs(), b.abs(), stride=(stride, 1), padding=(pad, 0))


def _gcn_skip_mag(xm, sd, key):
    if (key + "gcn_residual.0.weight") in sd:
        w, b, _ = _folded(sd, key + "gcn_residual.0.", key + "gcn_residual.1.")
        return _mconv(xm, w, b)
    return xm


def _plain_gcn_mag(xm, sd, key):
    B, C, T, V = xm.shape
    s = _folded(sd, key + "g_conv.0.", key + "bn.")[2]
    adj = (sd[key + "A"].double() * sd[key + "graph_attn"].double()).abs()
    total = 0
    bias = 0
    for p in range(3):
        mixed = torch.matmul(xm.reshape(B, C * T, V), adj[p]).reshape(B, C, T, V)
        total = total + F.conv2d(mixed, (sd[key + f"g_conv.{p}.weight"].double() * s[:, None, None, None]).abs())
        bias = bias + s * sd[key + f"g_conv.{p}.bias"].double()
    bias = bias + sd[key + "bn.bias"].double() - sd[key + "bn.running_mean"].double() * s
    return total + bias.abs()[None, :, None, None] + _gcn_skip_mag(xm, sd, key)


def _adaptive_gcn_mag(x, xm, sd, key):
    """Per frame (the continual model's T = 1 attention)."""
    B, C, T, V = x.shape
    s = _folded(sd, key + "g_conv.0.", key + "bn.")[2]
    adj = (sd[key + "A"].double() + sd[key + "graph_attn"].double())
    outs = []
    for t in range(T):
        xt, xmt = x[:, :, t: t + 1], xm[:, :, t: t + 1]
        total = 0
        bias = 0
        for p in range(3):
            theta = regular._conv(xt, sd, key + f"a_conv.{p}.")
            phi = regular._conv(xt, sd, key + f"b_conv.{p}.")
            ic = theta.shape[1]
            S = torch.softmax(torch.matmul(theta.permute(0, 3, 1, 2).reshape(B, V, ic), phi.reshape(B, ic, V)) / ic, dim=-2)
            att = (S + adj[p]).abs() + SOFTMAX_REL * S
            mixed = torch.matmul(xmt.reshape(B, C, V), att).reshape(B, C, 1, V)
            total = total + F.conv2d(mixed, (sd[key + f"g_conv.{p}.weight"].double() * s[:, None, None, None]).abs())
            bias = bias + s * sd[key + f"g_conv.{p}.bias"].double()
        bias = bias + sd[key + "bn.bias"].double() - sd[key + "bn.running_mean"].double() * s
        outs.append(total + bias.abs()[None, :, None, None] + _gcn_skip_mag(xmt, sd, key))
    return torch.cat(outs, dim=2)


def _attention_gcn_mag(x, xm, sd, key):
    """GcnUnitAttention on magnitudes; the q/k/v and output convs enter with |W|, the softmax weights as computed."""
    B, C, T, V = x.shape
    s_in = sd[key + "data_bn.weight"].double() / torch.sqrt(sd[key + "data_bn.running_var"].double() + regular.BN_EPS)
    t_in = sd[key + "data_bn.bias"].double() - sd[key + "data_bn.running_mean"].double() * s_in
    s_in, t_in = s_in.reshape(C, V)[None, :, None, :], t_in.reshape(C, V)[None, :, None, :]
    y = x * s_in + t_in
    ym = xm * s_in.abs() + t_in.abs()
    wq, bq = sd[key + "attention_conv.qkv_conv.weight"].double(), sd[key + "attention_conv.qkv_conv.bias"].double()
    wo, bo, s = _folded(sd, key + "attention_conv.attn_out.", key + "bn.")
    dv = wo.shape[0]
    dk = (wq.shape[0] - dv) // 2
    nh = regular.ATTENTION_HEADS
    ya, yma = y.permute(0, 2, 1, 3).reshape(B * T, C, 1, V), ym.permute(0, 2, 1, 3).reshape(B * T, C, 1, V)
    qkv = F.conv2d(ya, wq, bq)
    vm = _mconv(yma, wq, bq)[:, 2 * dk:]
    q, k, _ = torch.split(qkv, [dk, dk, dv], dim=1)
    q = q.reshape(B * T, nh, dk // nh, V) * ((dk // nh) ** -0.5)
    k = k.reshape(B * T, nh, dk // nh, V)
    w = torch.softmax(torch.matmul(q.transpose(2, 3), k), dim=-1)
    om = (1.0 + SOFTMAX_REL) * torch.matmul(w, vm.reshape(B * T, nh, dv // nh, V).transpose(2, 3))
    om = om.reshape(B * T, nh, 1, V, dv // nh).permute(0, 1, 4, 2, 3).reshape(B * T, dv, 1, V)
    om = _mconv(om, wo, bo).reshape(B, T, dv, V).permute(0, 2, 1, 3)
    if C == dv:
        om = om + s.abs()[None, :, None, None] * xm
    return om


def gcn_mag(x, xm, sd, key):
    if (key + "attention_conv.qkv_conv.weight") in sd:
        return _attention_gcn_mag(x, xm, sd, key)
    if (key + "a_conv.0.weight") in sd:
        return _adaptive_gcn_mag(x, xm, sd, key)
    return _plain_gcn_mag(xm, sd, key)


def block(x, sd, key, spec, pad, xm=None):
    """x (B, Cin, T, V) -> (value, mag), both float64 (B, Cout, T_out, V).  ``xm``: magnitude of the input (|x| by
    default; the previous block's ``mag`` when chaining).  Adaptive attention is evaluated per frame, as the
    continual model steps it."""
    x = x.double()
    xm = x.abs() if xm is None else xm.double()
    value = regular.st_block(x, sd, key, spec, pad, per_frame=True)
    gm = gcn_mag(x, xm, sd, key + "gcn.")
    w, b, _ = _folded(sd, key + "tcn.t_conv.", key + "tcn.bn.")
    mag = _mconv(gm, w, b, spec.stride, pad)
    shrink = 4 - pad
    xms = xm[:, :, shrink: xm.shape[2] - shrink] if shrink else xm
    if spec.res_kind == 1:
        mag = mag + xms
    elif spec.res_kind == 2:
        w, b, _ = _folded(sd, key + "residual.t_conv.", key + "residual.bn.")
        mag = mag + _mconv(xms, w, b, spec.stride)
    return value, mag


def data_bn(x, sd):
    """Raw frames (N, C, T, V, M) -> data_bn-normalised (value, mag), both float64 (N*M, C, T, V).  The affine map on
    magnitudes is |scale| * |x| + |shift|."""
    x = x.double()
    N, C, T, V, M = x.shape
    s = sd["data_bn.weight"].double() / torch.sqrt(sd["data_bn.running_var"].double() + regular.BN_EPS)
    t = sd["data_bn.bias"].double() - sd["data_bn.running_mean"].double() * s
    y = x.permute(0, 4, 3, 1, 2).reshape(N, M * V * C, T)
    m = (s.abs()[:, None] * y.abs() + t.abs()[:, None]).view(N, M, V, C, T).permute(0, 1, 3, 4, 2).reshape(N * M, C, T, V)
    return regular.normalise_input(x, sd), m


def head(y_seq, sd, arch, ym=None):
    """Last-block outputs (N*M, C, n, V) in emission order -> fp64 (value, mag) of the logits (N, classes, n_emit), the way
    the continual head computes them: spatial and person mean, the sliding window of ``arch.pool_size`` entries whose
    first ``arch.pool_padding`` positions start as zeros (the sum is always divided by ``pool_size``), then fc.
    ``ym``: magnitude of the input (|y| by default).  The magnitudes go through |fc|."""
    y = y_seq.double()
    ym = y.abs() if ym is None else ym.double()
    P, pp, M = arch.pool_size, arch.pool_padding, arch.persons
    first = P - 1 - pp  # pool inputs before the first emission
    w, b = sd["fc.weight"].double(), sd["fc.bias"].double()
    out = []
    for seq, wt, bt in ((y, w, b), (ym, w.abs(), b.abs())):
        NM, C, n, V = seq.shape
        p = seq.view(NM // M, M, C, n, V).mean(4).mean(1)  # (N, C, n)
        p = F.pad(p, (P - 1, 0))  # the window's zero entries before the first input
        win = p.unfold(2, P, 1)[:, :, first:].sum(3) / P  # (N, C, n_emit): window ending at input first + e
        out.append(torch.einsum("kc,nce->nke", wt, win) + bt[None, :, None])
    return out[0], out[1]


def model(x, sd, arch):
    """Raw frames (N, C, T, V, M) -> fp64 (value, mag) of the logits of every emission (N, classes, n_emit) of a whole
    continual model.  The block bound is chained: each block's ``mag`` is built from its predecessor's, starting from
    ``data_bn`` on |x|, and the head averages and pools the last ``mag`` and passes it through |fc|.  Each block adds at
    most EPS * its own ``mag``, and later blocks carry it no further than their magnitudes do, so the logits are held to
    n_blocks * EPS * mag, a coarse figure next to the single-block bound."""
    h, hm = data_bn(x, sd)
    for name, spec in zip(arch.block_names, arch.blocks):
        h, hm = block(h, sd, name, spec, arch.padding, xm=hm)
    # the regular clip math pads the end of every block: keep the outputs the continual walk has emitted
    n = emitted(x.shape[2], arch)
    return head(h[:, :, :n], sd, arch, ym=hm[:, :, :n])


def emitted(frames, arch):
    """Outputs the last block of a continual stack has emitted after ``frames`` steps from a fresh state."""
    first = arch.receptive_field - 1 - arch.stack_padding
    return max(0, (frames - 1 - first) // arch.stack_stride + 1)


def headroom(got, value, mag):
    """max |got - value| / (EPS * mag + TINY): <= 1 passes the bound, <= 1/4 with 4x margin."""
    d = (got.double() - value).abs()
    return float((d / (EPS * mag + TINY)).max())
