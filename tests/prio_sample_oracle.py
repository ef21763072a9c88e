"""Host reference of the prioritized sampler, ofb_replay_sample_prioritized (csrc/ofb_replay.cu) -- numpy only.

Draw b of a sample of B from masses m (age order, the order of ofb_replay_index):
  - U_b = ((c0 >> 5) * 2^26 + (c1 >> 6)) / 2^53, (c0, c1, ., .) = Philox4x32-10 of the counter (b, counter_lo, counter_hi,
    0x50524552) under the key (seed_lo, seed_hi), with ofb_common.cuh's philox4x32_10 (Random123's);
  - u = ((b + U_b) / B) * total in fp64, with the kernel's own total (last_total()): the kernel is built with -fmad=false,
    so numpy rounds u the same way;
  - the first candidate whose exact inclusive prefix of the masses exceeds u; when u is at or past the exact total, the last
    candidate of non-zero mass.  A zero mass is never drawn;
  - weight (m / m_min) ** -beta with m_min the smallest non-zero mass.

The counter is the number of earlier ofb_replay_sample_prioritized calls on the memory that had candidates (n_cand > 0):
a call on an all-zero memory counts, a call before the memory holds a candidate does not.

The kernel sums the masses in its own orders (tile sums, a chunked scan of the tiles, a block scan inside a tile), each
within about 60 eps * total of the exact prefix.  A draw whose u lies within WINDOW * total of a prefix boundary is flagged
ambiguous: the kernel may take any candidate between the exact picks at u - WINDOW * total and u + WINDOW * total."""
import math
from collections import namedtuple

import numpy as np

WINDOW = 2.0 ** -44
TAG = 0x50524552                 # fourth counter word of the sampler's stream
_M32 = 0xFFFFFFFF
_SCALE = 200                     # exact block sums are integers in units of 2^-200 (float32 masses are multiples of 2^-149)

Draws = namedtuple("Draws", "pos ambiguous lo hi u")


def philox4x32_10(ctr, key):
    """Philox4x32-10: ctr = 4 words (ints or uint32 arrays, broadcast), key = 2 ints -> the 4 output words, uint32 arrays."""
    c = [x.astype(np.uint64) for x in np.broadcast_arrays(*[np.asarray(w, dtype=np.uint64) & np.uint64(_M32) for w in ctr])]
    k0, k1 = int(key[0]) & _M32, int(key[1]) & _M32
    m32, s32 = np.uint64(_M32), np.uint64(32)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c[0]          # 32 x 32 bits: exact in uint64
        p1 = np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> s32) ^ c[1] ^ np.uint64(k0), p1 & m32, (p0 >> s32) ^ c[3] ^ np.uint64(k1), p0 & m32]
        k0, k1 = (k0 + 0x9E3779B9) & _M32, (k1 + 0xBB67AE85) & _M32
    return tuple(x.astype(np.uint32) for x in c)


def uniforms(seed, counter, B):
    """The kernel's U in [0, 1) for the draws b = 0 .. B-1 of the sample with this counter (float64 [B])."""
    b = np.arange(B, dtype=np.uint64)
    c0, c1, _, _ = philox4x32_10((b, counter & _M32, (counter >> 32) & _M32, TAG), (seed & _M32, (seed >> 32) & _M32))
    return ((c0 >> 5).astype(np.float64) * 67108864.0 + (c1 >> 6).astype(np.float64)) / 9007199254740992.0


def _pieces(k):
    """k * 2^-_SCALE (a non-negative int) as a short list of doubles whose exact sum it is."""
    out = []
    while k:
        f = float(k)
        out.append(math.ldexp(f, -_SCALE))
        k -= int(f)
    return out


class Reference:
    """The inverse CDF of one set of masses, decided exactly.  A float64 prefix locates a candidate; where it cannot decide
    (u within its error bound of a boundary), math.fsum of an exact block prefix and the block's masses up to the candidate
    does."""

    def __init__(self, masses, block=2048):
        m = np.asarray(masses, dtype=np.float32).astype(np.float64).reshape(-1)
        if not (np.isfinite(m).all() and (m >= 0).all()):
            raise ValueError("masses must be finite and >= 0")
        self.m, self.n, self.block = m, m.size, int(block)
        nz = np.flatnonzero(m > 0)
        self.n_valid = int(nz.size)
        self.last = int(nz[-1]) if nz.size else -1
        self.m_min = float(m[nz].min()) if nz.size else 0.0
        self.total = math.fsum(m)                                   # exact total, rounded once
        # exact block sums: each float32 mass is q * 2^e with an integer q < 2^24, so per (block, e) the sum of the q is
        # below 2^35 and exact in float64
        nb = max(1, -(-self.n // self.block))
        mant, ex = np.frexp(m)
        q = np.ldexp(mant, 24)
        assert bool((q == np.floor(q)).all())
        e = (ex - 24 + _SCALE).astype(np.int64)
        E = int(e.max()) + 1 if self.n else 1
        blk = np.arange(self.n) // self.block
        sums = np.bincount(blk * E + e, weights=q, minlength=nb * E).reshape(nb, E)
        bsum = [0] * nb
        r, c = np.nonzero(sums)
        for i, k, s in zip(r.tolist(), c.tolist(), sums[r, c].astype(np.int64).tolist()):
            bsum[i] += s << k
        prefix, run = [], 0
        for s in bsum:
            prefix.append(run)
            run += s
        self._bpre = [_pieces(k) for k in prefix]                  # exact exclusive prefix of each block
        # float64 inclusive prefix, made non-decreasing: within (block + 2) eps * total of the exact one
        pad = np.zeros(nb * self.block)
        pad[:self.n] = m
        within = pad.reshape(nb, self.block).cumsum(axis=1).reshape(-1)[:self.n]
        approx = np.array([float(k) for k in prefix]) * 2.0 ** -_SCALE
        self.approx = np.maximum.accumulate(approx[blk] + within) if self.n else np.zeros(0)
        self.delta = 4.0 * (self.block + 2) * 2.0 ** -53 * self.total

    def excess(self, i, v):
        """exact (inclusive prefix of candidate i) - v, rounded once; i = -1 is the empty prefix."""
        if i < 0:
            return -v
        b0 = (i // self.block) * self.block
        return math.fsum(self._bpre[i // self.block] + self.m[b0:i + 1].tolist() + [-v])

    def pick(self, v):
        """For each v (float64 array): the first candidate whose exact inclusive prefix exceeds max(v, 0), or the last
        candidate of non-zero mass when there is none."""
        v = np.maximum(np.asarray(v, dtype=np.float64).reshape(-1), 0.0)
        if self.last < 0:
            raise ValueError("no candidate of non-zero mass")
        a, d, n = self.approx, self.delta, self.n
        i0 = np.searchsorted(a, v, side="right")
        hi_ok = (i0 < n) & (a[np.minimum(i0, n - 1)] - v > d)
        lo_ok = (i0 == 0) | (v - a[np.maximum(i0 - 1, 0)] >= d)
        out = i0.copy()
        for k in np.flatnonzero(~(hi_ok & lo_ok)):
            x = float(v[k])
            lo = int(np.searchsorted(a, x - d, side="right"))   # below lo: prefix <= a + d <= x
            hi = int(np.searchsorted(a, x + d, side="right"))   # from hi on: prefix >= a - d > x
            while lo < hi:                                      # first i in [lo, hi) with prefix > x, else hi
                mid = (lo + hi) // 2
                if self.excess(mid, x) > 0.0:
                    hi = mid
                else:
                    lo = mid + 1
            out[k] = lo
        out = np.where(out >= n, self.last, out)
        assert bool((self.m[out] > 0).all())
        return out

    def draw(self, total_kernel, U, B):
        """The draws of a sample of B with the uniforms U (float64 [B]) and the kernel's total -> Draws(pos, ambiguous,
        lo, hi, u): the reference pick, whether the window holds a boundary, and the range [lo, hi] a kernel may pick."""
        U = np.asarray(U, dtype=np.float64).reshape(-1)
        assert U.size == B
        u = ((np.arange(B, dtype=np.float64) + U) / float(B)) * float(total_kernel)
        w = WINDOW * float(total_kernel)
        lo, pos, hi = self.pick(u - w), self.pick(u), self.pick(u + w)
        return Draws(pos, lo != hi, lo, hi, u)

    def weights(self, pos, beta):
        """(m / m_min) ** -beta in fp64 for the candidates pos."""
        return (self.m[np.asarray(pos)] / self.m_min) ** -float(beta)


def draw(masses, total_kernel, U, B, beta):
    """One sample: (Draws, their fp64 weights)."""
    ref = Reference(masses)
    d = ref.draw(total_kernel, U, B)
    return d, ref.weights(d.pos, beta)
