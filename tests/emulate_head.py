"""fp64 references and per-element error bounds for single launches of the head kernels (tests only).

Each reference takes the kernel's own input for that launch, so errors do not compound across launches:
  * tcn_igemm_kernel (csrc/tcn_tc.cu), launch 1: h1 = LReLU(conv1(x) + b1);
    launch 2: y = post(LReLU(LReLU(conv2(h1) + b2) + res)), res = x or Wd x + bd, h1 as the kernel stored it;
  * tcn_block_kernel (csrc/tcn.cu): one whole TemporalBlock in fp32 FMA;
  * fusion_head_kernel (csrc/fusion.cu) and the composed fusion path: the fused features, and the classifier
    on cat(leader features, the kernel's fused features).
A launch passes when |got - ref| <= bound for every element (ratio() <= 1).  The bounds are envelopes
c * (|a| (*) |b|) built from the magnitudes of the operands, never a fraction of max |ref|: an element that
should be small keeps a small bound.

fp32 accumulation over K products: any summation order has |error| <= (K - 1) 2^-24 sum|terms| with round to
nearest.  The tensor core adds each K = 8 MMA group into the fp32 TMEM accumulator, so an output sees K/8
accumulator roundings; each group's own alignment and truncation costs at most a few 2^-23 of sum|terms|.
K 2^-24 covers both (K/8 steps x 4 units of 2^-23) and is also the recursive-summation worst case, so it
is the accumulation constant for every path here (acc_const).
"""
import torch
import torch.nn.functional as F

from oracle import lfan_oracle as O

U = 2.0 ** -24            # unit roundoff of fp32
LEAKY = 0.01


def tf32_truncate(x):
    """fp32 -> TF32 by dropping the low 13 mantissa bits (round toward zero)."""
    return (x.contiguous().view(torch.int32) & ~0x1FFF).view(torch.float32)


# How tcgen05.mma kind::tf32 converts fp32 operands it reads from shared memory: it drops the low 13 bits.
# Measured on an NVIDIA B200 (1000 W) on the benchmark's video stack at B = 8, T = 300: with truncated
# operands the worst ratio to the bound is 0.028, with round-to-nearest operands (O.tf32_round, cvt.rna)
# it is 21 (tests/test_gpu_head_launches.py::test_tf32_operand_convention).
TF32_OPERAND = tf32_truncate
TF32_OTHER = O.tf32_round


def acc_const(K):
    return K * U


def dot_const(n):
    """Error constant of an fp32 dot product of n terms in the fusion head (see fusion_fused)."""
    return 2 * n ** 0.5 * U


def ratio(got, ref, bound):
    """Elementwise |got - ref| / bound (<= 1 passes); a NaN in got counts as inf."""
    r = (got.to(ref.dtype) - ref).abs() / (bound + 1e-300)
    return torch.nan_to_num(r, nan=float("inf"))


def _lrelu(v):
    return torch.where(v >= 0, v, v * LEAKY)


def causal_conv(x, w, d, shifts=None):
    """x [B,T,C], w [C_out, k, C] -> [B,T,C_out]: sum_j x[b, t - (k-1-j) d] w[:, j] with zeros before t = 0
    of each sequence (Conv1d padding (k-1)d + Chomp1d).  `shifts` overrides the per-tap shifts."""
    B, T, _ = x.shape
    k = w.shape[1]
    out = x.new_zeros(B, T, w.shape[0])
    for j in range(k):
        sh = (k - 1 - j) * d if shifts is None else shifts[j]
        xs = F.pad(x, (0, 0, sh, 0))[:, :T] if sh > 0 else x
        out = out + xs @ w[:, j].t()
    return out


# ---------------------------------------------------------------------------------------------------------
# TCN, tensor-core kernel.  blk: K-major block (packing.tcn_block_to_kmajor): w1 [C_out][k C_in],
# w2 [C_out][k C_out (+ C_in)].  In dtype float64 the functions return (ref, bound); in float32 they are the
# stand-in of a correct kernel (TF32 operands, fp32 matmuls) and return (out, None).
# ---------------------------------------------------------------------------------------------------------
def _kt(blk, name, cin, dtype, tf32):
    k = blk["kernel_size"]
    w = blk[name]
    return tf32(w.float()).to(dtype).view(blk["c_out"], -1)[:, :k * cin].reshape(blk["c_out"], k, cin)


def tcn_tc_launch1(blk, x, dtype=torch.float64, tf32=None, shifts=None):
    """h1 = LReLU(conv1(x) + b1); x: the fp32 input the kernel read [B,T,C_in]."""
    tf32 = tf32 or TF32_OPERAND
    cin, d = blk["c_in"], blk["dilation"]
    xt = tf32(x.float()).to(dtype)
    w = _kt(blk, "w1", cin, dtype, tf32)
    b = blk["b1"].to(dtype)
    z = causal_conv(xt, w, d, shifts) + b
    if dtype != torch.float64:
        return _lrelu(z), None
    S = causal_conv(xt.abs(), w.abs(), d, shifts)
    return _lrelu(z), acc_const(blk["kernel_size"] * cin) * S + 2 * U * (S + b.abs())


def tcn_tc_launch2(blk, x, h1, dtype=torch.float64, tf32=None):
    """y = post(LReLU(LReLU(conv2(h1) + b2) + res)); x: the block input, h1: what launch 1 stored."""
    tf32 = tf32 or TF32_OPERAND
    k, d, cin, cout = blk["kernel_size"], blk["dilation"], blk["c_in"], blk["c_out"]
    ht = tf32(h1.float()).to(dtype)
    w2 = _kt(blk, "w2", cout, dtype, tf32)
    b2 = blk["b2"].to(dtype)
    a = causal_conv(ht, w2, d) + b2
    f = _lrelu(a)
    if blk["wd"] is not None:
        wd = tf32(blk["w2"].float()).to(dtype)[:, k * cout:]                 # [C_out][C_in]
        xt = tf32(x.float()).to(dtype)
        res = xt @ wd.t() + blk["bd"].to(dtype)
    else:
        res = x.to(dtype)
    y = _lrelu(f + res)
    s = t = None
    if blk["post_scale"] is not None:
        s, t = blk["post_scale"].to(dtype), blk["post_shift"].to(dtype)
        y = y * s + t
    if dtype != torch.float64:
        return y, None
    S2 = causal_conv(ht.abs(), w2.abs(), d)
    env = acc_const(k * cout) * S2 + 4 * U * (S2 + b2.abs())
    if blk["wd"] is not None:
        Sd = xt.abs() @ wd.abs().t()
        env = env + acc_const(cin) * Sd + 4 * U * (Sd + blk["bd"].to(dtype).abs())
    else:
        env = env + 4 * U * res.abs()
    if s is not None:
        env = env * s.abs()
    return y, env + 2 * U * y.abs()


# ---------------------------------------------------------------------------------------------------------
# TCN, fp32 CUDA-core kernel (one launch per block).  blk: tap-major block (packing.pack_tcn):
# w1 [k][C_in][C_out], w2 [k][C_out][C_out], wd [C_in][C_out].  conv1's output stays in fp32 inside the
# kernel, so its error is carried into conv2 through |w2|.
# ---------------------------------------------------------------------------------------------------------
def tcn_fp32_block(blk, x):
    k, d, cin, cout = blk["kernel_size"], blk["dilation"], blk["c_in"], blk["c_out"]
    xd = x.double()
    w1 = blk["w1"].double().permute(2, 0, 1)                  # [C_out][k][C_in]
    w2 = blk["w2"].double().permute(2, 0, 1)
    b1, b2 = blk["b1"].double(), blk["b2"].double()
    S1 = causal_conv(xd.abs(), w1.abs(), d)
    h1 = _lrelu(causal_conv(xd, w1, d) + b1)
    e1 = acc_const(k * cin) * S1 + 2 * U * (S1 + b1.abs())
    S2 = causal_conv(h1.abs(), w2.abs(), d)
    f = _lrelu(causal_conv(h1, w2, d) + b2)
    env = causal_conv(e1, w2.abs(), d) + acc_const(k * cout) * S2 + 4 * U * (S2 + b2.abs())
    if blk["wd"] is not None:
        wd = blk["wd"].double()
        res = xd @ wd + blk["bd"].double()
        Sd = xd.abs() @ wd.abs()
        env = env + acc_const(cin) * Sd + 4 * U * (Sd + blk["bd"].double().abs())
    else:
        res = xd
        env = env + 4 * U * res.abs()
    y = _lrelu(f + res)
    if blk["post_scale"] is not None:
        s = blk["post_scale"].double()
        y = y * s + blk["post_shift"].double()
        env = env * s.abs()
    return y, env + 2 * U * y.abs()


# ---------------------------------------------------------------------------------------------------------
# Fusion head.  fw: packing.pack_fusion output; feats: list of [R, D_m].  First-order propagation of fp64
# envelopes through QKV linear -> scores -> softmax -> att V + V -> o_proj -> LayerNorm.
#
# The long dot products here (QKV over D_m <= 128, o_proj and the LayerNorm sums over E <= 128, the classifier
# over D_0 + E) use dot_const(n) = 2 sqrt(n) u instead of the worst case n u.  A sum of n terms makes n
# roundings of at most u |partial sum| each; for these operands (inputs and weights of both signs) the partial
# sums stay far below sum|terms| and the roundings do not line up, so the error of a correct kernel stays
# well under 2 sqrt(n) u sum|terms| (the fp32 stand-ins of tests/test_head_parity_guards.py stay below 0.1).  The
# worst-case n u would be loose enough to hide an O(1/E) LayerNorm fault such as the unbiased variance.
# The short sums (head_dim-long scores, the M-long softmax and att V) keep their worst-case constants.
# ---------------------------------------------------------------------------------------------------------
def fusion_fused(fw, feats):
    """-> (fused ref [R,E] fp64, bound [R,E])."""
    M, md, H = fw["n_modals"], fw["modal_dim"], fw["num_heads"]
    hd = md // H
    E = M * md
    f = [t.double() for t in feats]
    R = f[0].shape[0]
    qkv, eq = [], []
    for m in range(M):
        w, b = fw["wqkv"][m].double(), fw["bqkv"][m].double()
        qkv.append((f[m] @ w + b).view(R, H, 3, hd))
        eq.append((dot_const(fw["dim"][m] + 1) * (f[m].abs() @ w.abs() + b.abs())).view(R, H, 3, hd))

    def split(ts, i):
        return torch.stack([t[:, :, i] for t in ts], dim=2)           # [R,H,M,hd]

    q, k, v = split(qkv, 0), split(qkv, 1), split(qkv, 2)
    dq, dk, dv = split(eq, 0), split(eq, 1), split(eq, 2)
    scale = hd ** -0.5
    s = q @ k.transpose(-1, -2) * scale                                # [R,H,M,M]
    qk_abs = q.abs() @ k.abs().transpose(-1, -2)
    ds = scale * (dq @ k.abs().transpose(-1, -2) + q.abs() @ dk.transpose(-1, -2) + hd * U * qk_abs) + 6 * U * s.abs()
    ds = ds + U * (s - s.amax(-1, keepdim=True)).abs() + 4 * U             # max subtraction and expf inside softmax
    p = torch.softmax(s, dim=-1)
    dp = p * (ds + (p * ds).sum(-1, keepdim=True)) + (M + 2) * U * p
    vals = p @ v + v
    dvals = dp @ v.abs() + p @ dv + dv + (M + 1) * U * (p @ v.abs() + v.abs())
    vals, dvals = vals.reshape(R, E), dvals.reshape(R, E)
    wo, bo = fw["wo"].double(), fw["bo"].double()
    o = vals @ wo + bo
    do = dvals @ wo.abs() + dot_const(E + 1) * (vals.abs() @ wo.abs() + bo.abs())
    g, beta = fw["ln_g"].double(), fw["ln_b"].double()
    mu = o.mean(-1, keepdim=True)
    var = (o - mu).pow(2).mean(-1, keepdim=True)
    r = (var + O.LN_EPS).rsqrt()
    yh = (o - mu) * r
    fused = yh * g + beta
    prop = g.abs() * r * (do + do.mean(-1, keepdim=True) + yh.abs() * (yh.abs() * do).mean(-1, keepdim=True))
    own = (g.abs() * r * (1 + yh.abs()) * dot_const(E + 2) * o.abs().mean(-1, keepdim=True)
           + (yh * g).abs() * (dot_const(E + 2) * o.pow(2).mean(-1, keepdim=True) * r * r + 6 * U) + U * beta.abs())
    return fused, prop + own


def fusion_logits(fw, feats0, fused):
    """Classifier on cat(leader features, fused) -> (logits ref fp64, bound).  `fused` is the kernel's."""
    cat = torch.cat([feats0.double(), fused.double()], dim=-1)
    wr, br = fw["wr"].double(), fw["br"].double()
    return cat @ wr + br, dot_const(cat.shape[1] + 2) * (cat.abs() @ wr.abs() + br.abs())
