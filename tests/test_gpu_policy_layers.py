"""Every kernel of the policy forward against a float64 reference of its own inputs, per element -- B200 box.

Each stage takes the engine's own tap of its input (so upstream noise does not accumulate) and is compared with the float64
stage reference of oracle/policy_layers.py under the per-element bound documented there:
    |x - ref| <= ALPHA[stage] * u * B + eps_out
The analytic value of alpha is 1 (every product rounds its weight once to bf16 -- or each tf32 operand once -- and the fp32
sums add K * 2^-23 on top, which is inside u).  The tests print, per path, stage and region (interior, the four edge rows /
columns, the four corners), the largest alpha an element needed.

Measured on B200 (NVIDIA B200, 1000 W power limit), the largest alpha any element needed over every path, map, weight set and
batch size of this module: trunk12 0.000 (inside eps_out and the pool1 ulp), conv3 0.693, conv4 0.618, dense1 0.450, act 0.000,
up2 0.014, up3 0.819, ptr 0.580 -- interior and border regions alike once the border's out-of-range taps are counted twice
(oracle/policy_layers.py).  A 5 % change of one corner coefficient of the fused tail needs 1.54 at the corner.

Paths: the product path (fused sparse trunk + fused tail), the dense trunk, the three-kernel trunk, the CUDA-core sparse trunk,
the two-kernel tail, the CUDA-core engine, the CTA-pair tail; TF2 and TF1 upsampling; one and seven policy ships per arena.
Maps: synthetic bit maps (``oracle.policy_layers.edge_maps``): empty, all ones, single bits at every border class, checkerboards,
stripes, random densities and maps whose dirty-cell counts sit exactly at the sparse trunk's list capacities and one over.
"""
import numpy as np
import pytest
import torch

from oracle import policy_layers as pl
from oracle import policy_torch as po

pytestmark = pytest.mark.gpu

ALPHA = {"trunk12": 1.0, "conv3": 1.0, "conv4": 1.0, "dense1": 1.0, "act": 1.0, "up2": 1.0, "up3": 1.0, "ptr": 1.0}

# name -> (PolicyB200 keyword arguments, engine, P)
PATHS = {
    "product": ({}, "tensor", 1),
    "product_P7": ({}, "tensor", 7),
    "dense_trunk": ({"dense_trunk": True}, "tensor", 1),
    "three_kernel_trunk": ({"fused_trunk": False}, "tensor", 1),
    "cc_sparse_trunk": ({"cc_sparse_trunk": True}, "tensor", 1),
    "two_kernel_tail": ({"fused_tail": False}, "tensor", 1),
    "pair_tail": ({"tail_pair": True}, "tensor", 1),
    "cuda_core": ({}, "cuda_core", 1),
    "cuda_core_P7": ({}, "cuda_core", 7),
    "tf1_product": ({"bilinear": "tf1"}, "tensor", 1),
    "tf1_two_kernel_tail": ({"bilinear": "tf1", "fused_tail": False}, "tensor", 1),
    "tf1_cuda_core": ({"bilinear": "tf1"}, "cuda_core", 1),
}

_WORST = {}


@pytest.fixture(scope="module")
def maps():
    m = pl.edge_maps()
    names = list(m)
    imgs = np.stack([m[k] for k in names])
    bits = pl.pack_bits(imgs).cuda()
    g = torch.Generator().manual_seed(17)
    vec = (torch.rand((len(names) * 7, 8), generator=g) * 2 - 1)
    return {"names": names, "imgs": torch.from_numpy(imgs.astype(np.float32)), "bits": bits, "vec": vec}


def _policy(w, kw, engine, max_ships):
    from ofighters_b200.policy import PolicyB200
    pol = PolicyB200(w, max_ships=max_ships, **kw)
    pol.set_taps(True)
    pol.set_engine(engine)
    return pol


def _tf32_up2(kw, engine):
    return engine == "tensor" and kw.get("fused_tail", True)


def _stage_ratios(w, pol, bits, imgs, vec, P, bilinear, tf32_up2, arenas=None, chunk=4):
    """Forward, taps, and per stage the region maxima of the needed alpha over the arenas `arenas` (default: all)."""
    A = bits.shape[0]
    n = A * P
    r = pol.forward(bits, vec.cuda(), P, want_ptr=True)
    torch.cuda.synchronize()
    taps = {"pool2": pol.debug_tap(1, A, (100, 100, 8)).cpu(), "pool3": pol.debug_tap(2, A, (50, 50, 8)).cpu(),
            "flat": pol.debug_tap(3, A, (5000,)).cpu(), "hflat": pol.debug_tap(4, A, (100,)).cpu(),
            "up2": pol.debug_tap(5, n, (100, 100, 8)).cpu(), "up3": pol.debug_tap(6, n, (200, 200, 8)).cpu()}
    assert float(taps["up2"][..., 4:].abs().max()) == 0.0          # channel padding stays zero
    act, ptr = r["act"].cpu(), r["ptr"].cpu()
    arenas = list(range(A)) if arenas is None else list(arenas)
    out = {}

    def acc(stage, x, st):
        rr = pl.ratio(x, st)
        reg = pl.region_max(rr) if rr.dim() >= 3 else {"all": float(rr.max())}
        cur = out.setdefault(stage, {})
        for k, v in reg.items():
            cur[k] = max(cur.get(k, 0.0), v)

    for c in range(0, len(arenas), chunk):
        a = arenas[c:c + chunk]
        s = [i * P + p for i in a for p in range(P)]
        acc("trunk12", taps["pool2"][a], pl.trunk12(w, imgs[a]))
        acc("conv3", taps["pool3"][a], pl.conv_level(w, taps["pool2"][a], 3))
        acc("conv4", taps["flat"][a], pl.conv_level(w, taps["pool3"][a], 4))
        acc("dense1", taps["hflat"][a], pl.dense1_flat(w, taps["flat"][a]))
        st_act, st_up2 = pl.heads(w, taps["hflat"][a], vec[s], P, bilinear, tf32_up2)
        acc("act", act[s], st_act)
        acc("up2", taps["up2"][s][..., :4], st_up2)
        acc("up3", taps["up3"][s], pl.up3(w, taps["up2"][s][..., :4], bilinear))
        acc("ptr", ptr[s], pl.up4(w, taps["up3"][s], bilinear))
    return out, r


def _report_and_check(tag, out):
    print("\n%s" % tag)
    for stage, reg in out.items():
        print("  %-8s %s" % (stage, " ".join("%s %.3f" % (k, v) for k, v in reg.items())))
        _WORST[stage] = max(_WORST.get(stage, 0.0), max(reg.values()))
    bad = {st: max(reg.values()) for st, reg in out.items() if not max(reg.values()) <= ALPHA[st]}
    assert not bad, (tag, bad)


def _first_argmax_xy(ptr):
    k = np.argmax(ptr.reshape(ptr.shape[0], -1).numpy(), axis=1)
    return torch.from_numpy(np.stack([k % 400, k // 400], axis=1)).long()


@pytest.mark.parametrize("path", list(PATHS))
def test_stages_against_float64(maps, path):
    kw, engine, P = PATHS[path]
    bilinear = kw.get("bilinear", "tf2")
    w = po.init_weights(5, randomize_bn=True)
    A = len(maps["names"]) if P == 1 else 6
    bits = maps["bits"][:A].contiguous() if P == 1 else maps["bits"][[0, 1, 2, 5, 12, 16]].contiguous()
    imgs = maps["imgs"][:A] if P == 1 else maps["imgs"][[0, 1, 2, 5, 12, 16]]
    vec = maps["vec"][:A * P]
    pol = _policy(w, kw, engine, A * P)
    out, r = _stage_ratios(w, pol, bits, imgs, vec, P, bilinear, _tf32_up2(kw, engine))
    _report_and_check(path, out)
    # decisions: exactly the first argmax of the library's own outputs
    assert torch.equal(r["xy"].cpu().long(), _first_argmax_xy(r["ptr"].cpu()))
    assert torch.equal(r["iaction"].cpu().long(), (r["act"][:, 1] > r["act"][:, 0]).long().cpu())


@pytest.mark.parametrize("wname", ["keras_default", "neg_gamma", "dead"])
def test_stages_edge_weights(maps, wname):
    """The product path and the CUDA-core engine with the Keras defaults, negative BN scales on some channels of every BN layer,
    and ReLU-dead channels (tiny variance, large |beta|: max-pools over ties)."""
    w = po.init_weights(0) if wname == "keras_default" else pl.edge_weights(wname)
    A = len(maps["names"])
    for path in ("product", "cuda_core"):
        kw, engine, P = PATHS[path]
        pol = _policy(w, kw, engine, A)
        out, _ = _stage_ratios(w, pol, maps["bits"], maps["imgs"], maps["vec"][:A], 1, "tf2", _tf32_up2(kw, engine))
        _report_and_check("%s/%s" % (wname, path), out)
        del pol


@pytest.mark.parametrize("n", [1, 5, 149, 2 * 148 + 1])
def test_stages_batch_sizes(maps, n):
    """Several arenas per persistent CTA, the tail's ship_of clamp (a CTA past the last ship repeats it), k_heads groups of
    fewer than 4 ships: the stages of the first, second, middle and last two ships of an n-ship batch."""
    w = po.init_weights(5, randomize_bn=True)
    A0 = len(maps["names"])
    idx = [i % A0 for i in range(n)]
    bits = maps["bits"][idx].contiguous()
    vec = torch.cat([maps["vec"]] * (n // len(maps["vec"]) + 1))[:n]
    sample = sorted(set([0, 1, n // 2, n - 2, n - 1]) & set(range(n)))
    for path in ("product", "pair_tail"):
        kw, engine, _ = PATHS[path]
        pol = _policy(w, kw, engine, n)
        out, r = _stage_ratios(w, pol, bits, maps["imgs"][idx], vec, 1, "tf2", True, arenas=sample)
        _report_and_check("n=%d/%s" % (n, path), out)
        assert torch.equal(r["xy"].cpu().long(), _first_argmax_xy(r["ptr"].cpu()))
        del pol


def _all_paths_forward(w, bits, vec, P=1):
    for path, (kw, engine, p) in PATHS.items():
        if p != 1:
            continue
        pol = _policy(w, kw, engine, bits.shape[0] * P)
        r = pol.forward(bits, vec.cuda(), P, want_ptr=True)
        torch.cuda.synchronize()
        yield path, {k: v.cpu() for k, v in r.items()}
        del pol


def test_argmax_with_a_large_upconv4_bias(maps):
    """upconv4's bias = 2^17 on O(1) maps: pixels whose pre-bias values differ round to the same v + bias.  Every path's (x, y) is
    the FIRST flat argmax of the map it returns (ofb_policy.h), and the scene really holds such ties: counted from the same
    weights with bias 0 (ptr - bias in float64 of that run)."""
    w = pl.edge_weights("bias4")
    w0 = dict(w)
    w0["upconv4/bias"] = torch.zeros(1)
    A = len(maps["names"])
    vec = maps["vec"][:A]
    pol0 = _policy(w0, {}, "tensor", A)
    r0 = pol0.forward(maps["bits"], vec.cuda(), 1, want_ptr=True)
    torch.cuda.synchronize()
    pre = r0["ptr"].cpu().double().reshape(A, -1)
    biased = (pre.float() + float(w["upconv4/bias"][0])).double()                          # what the fused tail stores: fp32(v + bias)
    top = biased == biased.max(dim=1, keepdim=True).values
    ties = 0
    for s in range(A):
        vals = pre[s][top[s]]
        ties += int(vals.numel() > 1 and float(vals.max() - vals.min()) > 0)
    first_is_not_pre_max = int((np.argmax(biased.numpy(), axis=1) != np.argmax(pre.numpy(), axis=1)).sum())
    print("\nbias 2^17: %d of %d ships have a maximum of ptr whose pre-bias values differ; on %d the first argmax of ptr is not the "
          "pre-bias argmax" % (ties, A, first_is_not_pre_max))
    assert ties > 0 and first_is_not_pre_max > 0
    for path, r in _all_paths_forward(w, maps["bits"], vec):
        assert torch.equal(r["xy"].long(), _first_argmax_xy(r["ptr"])), path


@pytest.mark.parametrize("kind", ["const_ptr", "zero_ptr"])
def test_argmax_of_a_constant_map(maps, kind):
    """upnorm3's beta very negative: up3 == 0 and ptr == upconv4's bias everywhere (0.5, or 0 with the signed zeros of the
    products): the first flat argmax is (0, 0) for every ship on every path."""
    w = pl.edge_weights(kind)
    A = len(maps["names"])
    b4 = float(w["upconv4/bias"][0])
    for path, r in _all_paths_forward(w, maps["bits"], maps["vec"][:A]):
        assert bool((r["ptr"] == b4).all()), path
        print("%s/%s: all %d pixels of every ship tie, %d of them -0.0" % (kind, path, 160000, int(torch.signbit(r["ptr"]).sum())))
        assert torch.equal(r["xy"].long(), torch.zeros((A, 2), dtype=torch.long)), (path, r["xy"][:4])


def test_equal_action_values(maps):
    """output1's kernel 0 and equal biases: both action values are equal and iaction is the lower index, 0."""
    w = pl.edge_weights("equal_act")
    A = len(maps["names"])
    for path, r in _all_paths_forward(w, maps["bits"], maps["vec"][:A]):
        assert bool((r["act"][:, 0] == r["act"][:, 1]).all()), path
        assert int(r["iaction"].abs().sum()) == 0, path


def test_zz_report_worst():
    """Summary of the largest alpha per stage over every test of this module that ran."""
    print("\nlargest alpha needed per stage: " + " ".join("%s %.3f" % kv for kv in _WORST.items()))


@pytest.mark.parametrize("n_arenas, P", [(65536, 1), (16384, 7)])
def test_full_size_handle(n_arenas, P):
    """The bench's handle size: the whole batch in one launch per kernel (max_ships = N * P), against a max_ships = 8192 handle
    (several chunks) and against three windows of arenas (start, middle, end) run on their own: act, iaction and (x, y)
    bit for bit.  About 0.18 MB of workspace per ship: each handle is freed before the next is created."""
    from ofighters_b200 import BatchedBattleground
    from ofighters_b200.policy import PolicyB200
    w = po.init_weights(0)
    bg = BatchedBattleground(n_arenas, ships={"random": 7}, seed=2024)
    maps = bg.raster("bits")
    for _ in range(30):
        bg.frame(maps=maps)
    vec = bg.obs_vec[:, :P, :].contiguous().reshape(-1, 8)
    outs = {}
    for name, ms in (("full", n_arenas * P), ("chunked", 8192)):
        pol = PolicyB200(w, max_ships=ms)
        r = pol.forward(maps, vec, P, want_ptr=False)
        outs[name] = {k: r[k].clone() for k in ("act", "iaction", "xy")}
        if name == "chunked":
            W = 1024
            for a0 in (0, n_arenas // 2 - W // 2, n_arenas - W):
                rw = pol.forward(maps[a0:a0 + W].contiguous(), vec[a0 * P:(a0 + W) * P].contiguous(), P, want_ptr=False)
                for k in ("act", "iaction", "xy"):
                    assert torch.equal(rw[k], outs["full"][k][a0 * P:(a0 + W) * P]), (k, a0)
        del pol, r
        torch.cuda.synchronize()
    for k in ("act", "iaction", "xy"):
        assert torch.equal(outs["full"][k], outs["chunked"][k]), k
