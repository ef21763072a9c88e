"""CPU checks of the per-stage float64 references and error bounds (oracle/policy_layers.py) that the GPU layer tests rely on."""
import numpy as np
import pytest
import torch

from oracle import policy_layers as pl
from oracle import policy_torch as po


def _scene_imgs(n=2, seed=3):
    """Disks and short strokes like the simulator's, plus an all-ones corner patch: [n, 400, 400, 2] float."""
    g = np.random.default_rng(seed)
    img = np.zeros((n, 400, 400, 2), np.float32)
    yy, xx = np.mgrid[0:400, 0:400]
    for b in range(n):
        for _ in range(6):
            cy, cx, r = g.integers(0, 400), g.integers(0, 400), g.integers(3, 9)
            img[b, ..., 0][(yy - cy) ** 2 + (xx - cx) ** 2 <= r * r] = 1
        for _ in range(8):
            y, x = g.integers(0, 400), g.integers(0, 390)
            img[b, y, x:x + 10, 1] = 1
        img[b, :5, :7, :] = 1
    return torch.from_numpy(img)


@pytest.mark.parametrize("bilinear", ["tf2", "tf1"])
def test_chained_stages_equal_float64_forward(bilinear):
    w = po.init_weights(5, randomize_bn=True)
    img = _scene_imgs()
    vec = torch.randn(2, 8, generator=torch.Generator().manual_seed(1))
    act, ptr = pl.chain(w, img, vec, bilinear)
    act_ref, ptr_ref = po.forward(w, img, vec, bilinear=bilinear, dtype=torch.float64)
    assert float((act - act_ref).abs().max()) <= 1e-12 * max(1.0, float(act_ref.abs().max()))
    assert float((ptr - ptr_ref).abs().max()) <= 1e-12 * max(1.0, float(ptr_ref.abs().max()))


@pytest.mark.parametrize("wname", ["keras_default", "random_bn", "neg_gamma", "dead"])
def test_fp32_oracle_within_bounds(wname):
    """The fp32 oracle (policy_torch, fp32 everywhere) stays inside every stage's bound against the float64 references -- a
    bound must hold for arithmetic that is more accurate than the engine's.  Each stage takes the oracle's own input, rounded to
    bf16 where the engine stores bf16 (that rounding is the engine's, and the references start from it)."""
    w = po.init_weights(0) if wname == "keras_default" else pl.edge_weights(wname)
    img = _scene_imgs()
    vec = torch.randn(2, 8, generator=torch.Generator().manual_seed(2))
    act, ptr, inter = po.forward(w, img, vec, return_intermediates=True)

    def bf(t):
        return t.permute(0, 2, 3, 1).to(torch.bfloat16)

    worst = {}
    st = pl.trunk12(w, img)
    worst["trunk12"] = float(pl.ratio(bf(inter["pool2"]).float(), st).max())
    p2 = bf(inter["pool2"])
    x3 = po.F.max_pool2d(po._conv_bn_relu(p2.float().permute(0, 3, 1, 2), w, "conv3", "norm3"), 2)
    worst["conv3"] = float(pl.ratio(bf(x3).float(), pl.conv_level(w, p2, 3)).max())
    p3 = bf(x3)
    x4 = po.F.max_pool2d(po._conv_bn_relu(p3.float().permute(0, 3, 1, 2), w, "conv4", "norm4"), 2)
    flat = bf(x4).reshape(2, -1)
    worst["conv4"] = float(pl.ratio(flat.float(), pl.conv_level(w, p3, 4)).max())
    hflat = flat.float() @ w["dense1/kernel"][8:]
    worst["dense1"] = float(pl.ratio(hflat, pl.dense1_flat(w, flat)).max())
    act_st, up2_st = pl.heads(w, hflat, vec, 1, tf32_up2=False)
    h = torch.relu(vec @ w["dense1/kernel"][:8] + hflat + w["dense1/bias"])
    a = torch.relu(h @ w["dense2/kernel"] + w["dense2/bias"]) @ w["output1/kernel"] + w["output1/bias"]
    worst["act"] = float(pl.ratio(a, act_st).max())
    u = torch.relu(h @ w["updense1/kernel"] + w["updense1/bias"]).reshape(-1, 1, 25, 25)
    for i in (1, 2):
        u = po._conv_bn_relu(po.upsample2x(u), w, "upconv%d" % i, "upnorm%d" % i)
    up2 = bf(u)
    worst["up2"] = float(pl.ratio(up2.float(), up2_st).max())
    u3 = bf(po._conv_bn_relu(po.upsample2x(up2.float().permute(0, 3, 1, 2)), w, "upconv3", "upnorm3"))
    worst["up3"] = float(pl.ratio(u3.float(), pl.up3(w, up2)).max())
    p = po._conv_bn_relu(po.upsample2x(u3.float().permute(0, 3, 1, 2)), w, "upconv4", None)[:, 0]
    worst["ptr"] = float(pl.ratio(p, pl.up4(w, u3)).max())
    print(wname, {k: "%.3f" % v for k, v in worst.items()})
    # fp32 weights: everything but the bf16 / fp32 output rounding is far inside the bf16-operand bound
    assert all(v <= 0.25 for v in worst.values()), worst


def test_ratio_sees_a_single_wrong_pixel():
    """An error of 2 % of max|ref| on one border pixel of the pointer map is outside the bound; the map-wide criterion of the
    end-to-end tests (2.5e-2 * max|ref|) lets it through."""
    w = po.init_weights(5, randomize_bn=True)
    u3 = (torch.rand(1, 200, 200, 8, generator=torch.Generator().manual_seed(0)) * 2).to(torch.bfloat16)
    st = pl.up4(w, u3)
    x = st["ref"].clone()
    assert float(pl.ratio(x, st).max()) == 0.0
    x[0, 0, 137] += 0.02 * float(x.abs().max())
    reg = pl.region_max(pl.ratio(x, st))
    assert reg["top"] > 1.0 and reg["interior"] == 0.0 and reg["corner_tl"] == 0.0, reg


@pytest.mark.parametrize("level", [0, 1, 2])
def test_capacity_maps_have_the_claimed_dirty_counts(level):
    caps = (pl.ST_CAP1, pl.ST_VCAP, pl.ST_VCAP)
    n = pl.dirty_counts(pl.capacity_map(level))
    assert n[level] == caps[level] and all(n[i] <= caps[i] for i in range(3)), n
    n1 = pl.dirty_counts(pl.capacity_map(level, plus_one=True))
    assert n1 == tuple(v + 1 for v in n), (n, n1)           # one over the capacity at `level`
    assert n1[level] == caps[level] + 1


def test_dirty_counts_follow_the_definition():
    """Against a direct loop over the definition (a pool1 pixel (Y, X) is dirty iff a bit is set in rows 2Y-1 .. 2Y+2 and
    columns 2X-1 .. 2X+2; the levels above use the same window on the level below)."""
    g = np.random.default_rng(4)
    b = (g.random((400, 400)) < 0.002).astype(np.uint8)
    b[0, 0] = b[399, 399] = b[0, 250] = 1

    def up(d, n):
        o = np.zeros((n // 2, n // 2), bool)
        for Y in range(n // 2):
            for X in range(n // 2):
                o[Y, X] = d[max(2 * Y - 1, 0):2 * Y + 3, max(2 * X - 1, 0):2 * X + 3].any()
        return o

    d1 = up(b != 0, 400)
    d2 = up(d1, 200)
    d3 = up(d2, 100)
    assert pl.dirty_counts(b) == (int(d1.sum()), int(d2.sum()), int(d3.sum()))
    # a corner bit dirties one cell per level, an isolated interior bit 2 x 2 pool1 pixels
    one = np.zeros((400, 400), np.uint8)
    one[0, 0] = 1
    assert pl.dirty_counts(one) == (1, 1, 1)
    one[0, 0], one[200, 201] = 0, 1
    assert pl.dirty_counts(one)[0] == 4


def test_edge_maps_and_packing():
    m = pl.edge_maps()
    names = list(m)
    bits = pl.pack_bits(np.stack([m[k] for k in names]))
    assert bits.dtype == torch.int32 and tuple(bits.shape) == (len(names), 2, 5000)
    # the packing is the inverse of the tests' unpacking (bit y * 400 + x of channel c, little-endian words)
    d = np.unpackbits(bits.numpy().view(np.uint8).reshape(len(names), 2, -1), axis=2, bitorder="little")
    assert np.array_equal(d.reshape(len(names), 2, 400, 400).transpose(0, 2, 3, 1), np.stack([m[k] for k in names]) != 0)
    assert int(m["ones"].sum()) == 2 * 160000 and int(m["empty"].sum()) == 0
    for d_ in range(4):
        assert int(m["border%d" % d_].sum()) == 8
