"""float64 references of the policy forward, one stage at a time, with a per-element error bound -- TEST INFRASTRUCTURE.

Each stage starts from whatever tensor the caller passes (on the GPU tests: the engine's own tap of the stage's input, so that
upstream noise does not accumulate) and is computed in float64 from the Keras-layout weights (BatchNormalization folded in
float64 here, never the engine's folded or packed operands).  Stages and the engine's taps (``PolicyB200.debug_tap``):

    trunk12   bit maps            -> pool2 (tap 1)      conv1 + BN + ReLU + pool, pool1 rounded to bf16, conv2 + BN + ReLU + pool
    conv3     pool2 (tap 1)       -> pool3 (tap 2)
    conv4     pool3 (tap 2)       -> flat (tap 3)       NHWC order, the first 5000 entries of the 5120 pitch
    dense1    flat                -> hflat (tap 4)      flat @ dense1/kernel[8:]  (fp32, before bias and vector slice)
    heads     hflat + vec         -> act, up2 (tap 5)   vector slice + bias, ReLU, dense2, output1; updense1, upconv1, upconv2
    up3       up2 (tap 5)         -> up3 (tap 6)        upsample x2 + conv + BN + ReLU
    up4       up3 (tap 6)         -> ptr                upsample x2 + conv + bias

Bound, per element:   |x - ref| <= alpha * u * B + eps_out (+ extra)
  B        the same stage evaluated on absolute values (|folded weights| on |input|, the absolute value taken before the
           upsampling, |bias| terms included); a pooled cell takes the maximum of B over its 4 conv pixels; on the first and
           last row / column of upconv3 and upconv4 the out-of-range taps count twice, read on the replicate-extended input:
           the engine evaluates those pixels as the replicate-extended fold minus a correction, two separately rounded terms
           that cancel (measured without this: up to 6.4 times the plain bound on the CUDA-core engine's top row);
  u        the rounding unit of the stage's operands: 2^-8 for bf16 weights, 2^-10 for the tf32 upconv2 of the tensor path
           (weights and activations each rounded to nearest, 2^-11 apiece), plus K * 2^-23 for an fp32 sum of K terms;
           stages that run entirely in fp32 get the sum of (K + 2) * 2^-24 over their chained layers;
  eps_out  half a bf16 ulp of the result where the stage stores bf16 (of max(|ref|, |x|), which covers a rounding that crosses
           a power of two);
  extra    trunk12 only: conv2's |weights| applied to one bf16 ulp of pool1 (the engine's fp32 conv1 and this float64 conv1 may
           round pool1 to neighbouring bf16 values) plus conv1's fp32 error.
``ratio`` returns, per element, the alpha that element needs: max(|x - ref| - eps_out - extra, 0) / (u * B).

Nothing under ofighters_b200/ imports this module.
"""
import numpy as np
import torch
import torch.nn.functional as F

from .policy_torch import BN_EPS, upsample2x

U_BF16 = 2.0 ** -8
U_TF32 = 2.0 ** -10
ACC32 = 2.0 ** -23           # per term of a tensor-core fp32 accumulation
U_FP32 = 2.0 ** -24
U_CHAIN = 192 * U_FP32       # heads: (8 + 2) + (100 + 2) + (50 + 2) terms to act, (100 + 2) + (9 + 2) + (18 + 2) to up2, rounded up

REGIONS = ("interior", "top", "bottom", "left", "right", "corner_tl", "corner_tr", "corner_bl", "corner_br")


def _fold(w, conv, bn):
    """-> (kernel OIHW, bias, |bias| bound) in float64 with BatchNormalization folded in."""
    k = w[conv + "/kernel"].double().permute(3, 2, 0, 1).contiguous()
    b = w[conv + "/bias"].double()
    if bn is None:
        return k, b, b.abs()
    s = w[bn + "/gamma"].double() / torch.sqrt(w[bn + "/var"].double() + BN_EPS)
    mean, beta = w[bn + "/mean"].double(), w[bn + "/beta"].double()
    return k * s[:, None, None, None], (b - mean) * s + beta, (b.abs() + mean.abs()) * s.abs() + beta.abs()


def _conv(x, k, b):
    return F.conv2d(x, k, b, padding=1)


def _nchw(t):
    return t.double().permute(0, 3, 1, 2).contiguous()


def _nhwc(t):
    return t.permute(0, 2, 3, 1).contiguous()


def bf16_ulp(v):
    """One bf16 ulp of |v| (0 for 0)."""
    m, e = torch.frexp(v.double().abs())
    return torch.where(m == 0, torch.zeros_like(m), torch.ldexp(torch.ones_like(m), e - 8))


def _stage(ref, B, u, bf16_out, extra=None):
    return {"ref": ref, "B": B, "u": u, "bf16_out": bf16_out, "extra": extra}


def _conv_pool_stage(w, x, i):
    k, b, babs = _fold(w, "conv%d" % i, "norm%d" % i)
    ref = F.max_pool2d(F.relu(_conv(x, k, b)), 2)
    B = F.max_pool2d(_conv(x.abs(), k.abs(), babs), 2)
    return ref, B, k


def trunk12(w, bits):
    """bits [n, 400, 400, 2] (0 / 1) -> pool2 [n, 100, 100, 8]."""
    x = _nchw(bits)
    k1, b1, b1abs = _fold(w, "conv1", "norm1")
    p1 = F.max_pool2d(F.relu(_conv(x, k1, b1)), 2)
    B1 = F.max_pool2d(_conv(x, k1.abs(), b1abs), 2)
    p1r = p1.to(torch.bfloat16).double()                        # the engine stores pool1 in bf16 (round to nearest even)
    ref, B, k2 = _conv_pool_stage(w, p1r, 2)
    extra = F.max_pool2d(F.conv2d(bf16_ulp(p1r) + 2.0 ** -18 * B1, k2.abs(), padding=1), 2)
    return _stage(_nhwc(ref), _nhwc(B), U_BF16 + 72 * ACC32, True, _nhwc(extra))


def conv_level(w, x_nhwc, i):
    """conv3 (i = 3) on pool2 [n, 100, 100, 8] or conv4 (i = 4) on pool3 [n, 50, 50, 8]; conv4's result is flattened NHWC."""
    ref, B, _ = _conv_pool_stage(w, _nchw(x_nhwc), i)
    ref, B = _nhwc(ref), _nhwc(B)
    if i == 4:
        ref, B = ref.reshape(ref.shape[0], -1), B.reshape(B.shape[0], -1)
    return _stage(ref, B, U_BF16 + 72 * ACC32, True)


def dense1_flat(w, flat):
    """flat [n, 5000] -> flat @ dense1/kernel[8:] [n, 100] (the engine keeps it in fp32)."""
    W = w["dense1/kernel"].double()[8:]
    f = flat.double()
    return _stage(f @ W, f.abs() @ W.abs(), U_BF16 + 5000 * ACC32, False)


def heads(w, hflat, vec, P=1, bilinear="tf2", tf32_up2=True):
    """hflat [A, 100] (tap 4), vec [A * P, 8] -> (act stage [A * P, 2], up2 stage [A * P, 100, 100, 4])."""
    d = {k: v.double() for k, v in w.items() if "dense" in k or "output" in k}
    hf = hflat.double().repeat_interleave(P, dim=0)
    v = vec.double()
    Wv = d["dense1/kernel"][:8]
    h = F.relu(v @ Wv + hf + d["dense1/bias"])
    Bh = v.abs() @ Wv.abs() + hf.abs() + d["dense1/bias"].abs()

    def dense(x, Bx, name, relu):
        y = x @ d[name + "/kernel"] + d[name + "/bias"]
        return (F.relu(y) if relu else y), Bx @ d[name + "/kernel"].abs() + d[name + "/bias"].abs()

    d2, Bd2 = dense(h, Bh, "dense2", True)
    act, Bact = dense(d2, Bd2, "output1", False)
    u, Bu = dense(h, Bh, "updense1", True)
    u, Bu = u.reshape(-1, 1, 25, 25), Bu.reshape(-1, 1, 25, 25)
    for i in (1, 2):
        k, b, babs = _fold(w, "upconv%d" % i, "upnorm%d" % i)
        u = F.relu(_conv(upsample2x(u, bilinear), k, b))
        Bu = _conv(upsample2x(Bu, bilinear), k.abs(), babs)
    return (_stage(act, Bact, U_CHAIN, False),
            _stage(_nhwc(u), _nhwc(Bu), (U_TF32 if tf32_up2 else 0.0) + U_CHAIN, True))


def _upconv_B(xa, kabs, babs):
    """B of a convolution on an upsampled map whose border pixels the engine takes as the replicate-extended fold minus a
    correction for the out-of-range taps (each rounded on its own): the in-range taps once, the out-of-range ones -- read on
    the replicate-extended |input| -- twice.  Equal to the plain B away from the border."""
    b_in = _conv(xa, kabs, None)
    b_rep = F.conv2d(F.pad(xa, (1, 1, 1, 1), mode="replicate"), kabs)
    return 2 * b_rep - b_in + babs[None, :, None, None]


def up3(w, up2_nhwc, bilinear="tf2"):
    """up2 [n, 100, 100, 4] -> up3 [n, 200, 200, 8]."""
    x = upsample2x(_nchw(up2_nhwc), bilinear)
    xa = upsample2x(_nchw(up2_nhwc).abs(), bilinear)
    k, b, babs = _fold(w, "upconv3", "upnorm3")
    return _stage(_nhwc(F.relu(_conv(x, k, b))), _nhwc(_upconv_B(xa, k.abs(), babs)), U_BF16 + 36 * ACC32, True)


def up4(w, up3_nhwc, bilinear="tf2"):
    """up3 [n, 200, 200, 8] -> ptr [n, 400, 400]."""
    x = upsample2x(_nchw(up3_nhwc), bilinear)
    xa = upsample2x(_nchw(up3_nhwc).abs(), bilinear)
    k, b, babs = _fold(w, "upconv4", None)
    return _stage(_conv(x, k, b)[:, 0], _upconv_B(xa, k.abs(), babs)[:, 0], U_BF16 + 72 * ACC32, False)


def chain(w, bits, vec, bilinear="tf2"):
    """All stages chained on their own float64 results (no bf16 rounding of pool1): the full forward, for the CPU check against
    policy_torch.forward(dtype=float64)."""
    x = _nchw(bits)
    for i in range(1, 5):
        x, _, _ = _conv_pool_stage(w, x, i)
    flat = _nhwc(x).reshape(x.shape[0], -1)
    hflat = dense1_flat(w, flat)["ref"]
    act, up2 = heads(w, hflat, vec, 1, bilinear)
    u3 = up3(w, up2["ref"], bilinear)
    return act["ref"], up4(w, u3["ref"], bilinear)["ref"]


def ratio(x, st):
    """Per element: the alpha this element needs, max(|x - ref| - eps_out - extra, 0) / (u * B) (inf where B = 0 and x != ref)."""
    x = x.double().cpu()
    ref = st["ref"]
    x = x.reshape(ref.shape)
    err = (x - ref).abs()
    if st["bf16_out"]:
        err = err - 0.5 * bf16_ulp(torch.maximum(ref.abs(), x.abs()))
    if st["extra"] is not None:
        err = err - st["extra"]
    err = err.clamp_min(0.0)
    den = st["u"] * st["B"]
    return torch.where(err == 0, torch.zeros_like(err), err / den)


def region_max(r):
    """r [n, H, W(, C)] -> {region: max}: interior, the four edge rows / columns without their ends, the four corners."""
    H, W = r.shape[1], r.shape[2]
    r = r.reshape(r.shape[0], H, W, -1)
    sl = {"interior": (slice(1, H - 1), slice(1, W - 1)), "top": (0, slice(1, W - 1)), "bottom": (H - 1, slice(1, W - 1)),
          "left": (slice(1, H - 1), 0), "right": (slice(1, H - 1), W - 1), "corner_tl": (0, 0), "corner_tr": (0, W - 1),
          "corner_bl": (H - 1, 0), "corner_br": (H - 1, W - 1)}
    return {k: float(r[:, a, b].max()) for k, (a, b) in sl.items()}


# ---------------------------------------------------------------------------------------------------------- synthetic bit maps
def dirty_counts(img):
    """img [400, 400] or [400, 400, 2] (non-zero = set) -> dirty cells of the sparse trunk (pool1 pixels, pool2 cells, pool3 cells).
    A pool1 pixel (Y, X) is dirty iff a bit is set in rows 2Y-1 .. 2Y+2 and columns 2X-1 .. 2X+2; a cell of the next level is
    dirty iff its window (rows / columns 2Y-1 .. 2Y+2) one level down holds a dirty cell."""
    a = np.asarray(img)
    if a.ndim == 3:
        a = a.any(axis=2)
    x = torch.as_tensor(a != 0, dtype=torch.float32)[None, None]
    out = []
    for _ in range(3):
        x = F.max_pool2d(F.pad(x, (1, 1, 1, 1)), 4, 2)
        out.append(int(x.sum()))
    return tuple(out)


# the sparse trunk's list capacities (ofb_policy_st.cu): ST_CAP1 dirty pool1 pixels, ST_VCAP dirty pool2 / pool3 cells
ST_CAP1, ST_VCAP = 1280, 1024


def _grow(level, target, caps, passes):
    """Bits added pass by pass (each pass a list of positions) while the counts allow: dirty cells of `level` == target, the
    others <= caps."""
    b = np.zeros((400, 400), np.uint8)
    for cands in passes:
        for y, x in cands:
            b[y, x] = 1
            n = dirty_counts(b)
            if n[level] > target or any(n[i] > caps[i] for i in range(3)):
                b[y, x] = 0
            elif n[level] == target:
                return b
    raise AssertionError("no map with %d dirty cells at level %d" % (target, level + 1))


def _lattice(spacing, lo, hi):
    return [(y, x) for y in range(lo, hi, spacing) for x in range(lo, hi, spacing)]


_CORNERS3 = [(0, 0), (0, 399), (399, 0)]          # one dirty cell per level each; (399, 399) is kept for ``plus_one``


def capacity_map(level, plus_one=False):
    """[400, 400, 2] bits whose dirty-cell count at `level` (0: pool1, 1: pool2, 2: pool3) is exactly the sparse trunk's capacity
    (ST_CAP1, ST_VCAP, ST_VCAP) while the other levels stay within theirs; ``plus_one`` adds the corner bit (399, 399), one more
    dirty cell at every level."""
    caps = (ST_CAP1, ST_VCAP, ST_VCAP)
    if level == 0:                                 # a dense block: many pool1 pixels, few cells above
        b = _grow(0, ST_CAP1, caps, [_lattice(2, 150, 300), _CORNERS3])
    elif level == 1:                               # isolated bits every 8 px
        b = _grow(1, ST_VCAP, caps, [_lattice(8, 20, 380), _CORNERS3])
    else:                                          # bits at y, x = 3 (mod 8) dirty 3 x 3 pool3 cells but 2 x 2 pool2 cells
        b = _grow(2, ST_VCAP, caps, [_lattice(24, 3, 397), _lattice(24, 15, 397), _CORNERS3])
    if plus_one:
        b[399, 399] = 1
    return np.stack([b, np.zeros_like(b)], axis=2)


def edge_maps(seed=0):
    """name -> [400, 400, 2] uint8 bit maps at the edges of the trunk and the border classes."""
    m = {}
    z = np.zeros((400, 400, 2), np.uint8)
    m["empty"] = z.copy()
    m["ones"] = np.ones_like(z)
    for d in range(4):                            # corners and edge midpoints, d px in from the edge: every border class
        b = z.copy()
        for (y, x) in [(d, d), (d, 399 - d), (399 - d, d), (399 - d, 399 - d), (d, 200), (399 - d, 200), (200, d), (200, 399 - d)]:
            b[y, x, d % 2] = 1
        m["border%d" % d] = b
    b = z.copy()
    b[399, 0, 1] = 1
    m["corner_bl"] = b
    yy, xx = np.mgrid[0:400, 0:400]
    b = z.copy(); b[..., 0] = (yy + xx) % 2; m["checker"] = b
    b = z.copy(); b[..., 1] = ((yy // 2) + (xx // 2)) % 2; m["checker2"] = b
    b = z.copy(); b[..., 0] = yy % 4 == 0; m["stripes_h"] = b
    b = z.copy(); b[..., 1] = xx % 3 == 0; m["stripes_v"] = b
    rng = np.random.default_rng(seed)
    for p in (0.005, 0.02, 0.1, 0.5):
        m["random%g" % p] = (rng.random((400, 400, 2)) < p * np.array([1.0, 0.5])).astype(np.uint8)
    for level, name in enumerate(("cap1", "vcap2", "vcap3")):
        m[name] = capacity_map(level)
        m[name + "+1"] = capacity_map(level, plus_one=True)
    return m


def pack_bits(imgs):
    """[A, 400, 400, 2] (non-zero = set) -> int32 [A, 2, 5000] bit maps (bit y * 400 + x, little-endian words)."""
    a = (np.asarray(imgs) != 0).transpose(0, 3, 1, 2).reshape(len(imgs), 2, 160000)
    return torch.from_numpy(np.packbits(a, axis=2, bitorder="little").view(np.int32).copy())


# ---------------------------------------------------------------------------------------------------------- edge weight sets
def edge_weights(kind, seed=5):
    """Weight sets at the edges of the folding (from policy_torch.init_weights(seed, randomize_bn=True)):
    neg_gamma   a negative BN gamma on some channels of every BN layer
    dead        a tiny var with a large |beta| on some channels of every BN layer: whole channels are ReLU-dead (or saturated
                high), max-pools tie
    bias4       upconv4's bias = 2^17 (the map's values are O(1), fp32's spacing there is 2^-6): pre-bias values that differ
                tie after the bias (at a bias of 64 the maxima of these scenes are further apart than fp32's spacing)
    const_ptr   upnorm3's beta very negative: up3 == 0, ptr == upconv4's bias (0.5)
    zero_ptr    the same with upconv4's bias 0 (the map is all +-0)
    equal_act   output1's kernel 0 and equal biases: both action values equal"""
    from .policy_torch import init_weights
    w = init_weights(seed, randomize_bn=True)
    bns = sorted(k[:-6] for k in w if k.endswith("/gamma"))
    if kind == "neg_gamma":
        for n in bns:
            g = w[n + "/gamma"].clone()
            g[1::3] = -g[1::3]
            w[n + "/gamma"] = g
    elif kind == "dead":
        for n in bns:
            v, be = w[n + "/var"].clone(), w[n + "/beta"].clone()
            v[0::4] = 1e-6
            be[0::4] = -50.0
            be[2::4] = 3.0
            w[n + "/var"], w[n + "/beta"] = v, be
    elif kind == "bias4":
        w["upconv4/bias"] = torch.tensor([131072.0])
    elif kind in ("const_ptr", "zero_ptr"):
        w["upnorm3/beta"] = torch.full((8,), -1e4)
        w["upconv4/bias"] = torch.tensor([0.5 if kind == "const_ptr" else 0.0])
    elif kind == "equal_act":
        w["output1/kernel"] = torch.zeros(50, 2)
        w["output1/bias"] = torch.full((2,), 0.25)
    elif kind != "random_bn":
        raise ValueError(kind)
    return w
