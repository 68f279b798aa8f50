"""Inputs, float64 reference and error bound for the head_dim-64 attention kernels (csrc/attention.cu).  No GPU needed.

Error model of the kernels against softmax(scale q k^T) v computed exactly from the same fp16 inputs:
- P is rounded to fp16 before the P V product: 2^-11 relative, also for the values up to 2^8 that the lazy reference max allows;
- two of every eight exponentials use a cubic exp2 that is off by at most 8.8e-5 relative (the MUFU ones by ~1e-7);
- the row sum l is accumulated in fp32 from the unrounded p, so only the exp2 error reaches it;
- O / l is rounded to fp16.
Together that is at most ~5.8e-4 of sum_j P_j |V_j| plus ~5.8e-4 of |O| per output element, so the bound below, with
c1 = c2 = 2^-10, holds with a margin of ~1.7 for any correct kernel; a wrong tile weight, a stale max or a masking slip exceeds it.
One case is outside that model: P below 2^-14 is subnormal in fp16 and rounds by up to 2^-25 absolute, not 2^-11 relative.  In a
peaked row whose dominant V entry is near zero, those roundings make up most of the error; the 2^-24 term absorbs them, but the
margin shrinks (causal, scale 1.0, 128 keys: err/tol 0.74, the same in a CPU emulation of the kernel's rounding).

The generators return fp16 CPU tensors q [b*nq, heads*64], k and v [b*nkv, heads*64].
"""
import math

import torch

LOG2E = 1.4426950408889634
TILE = 128                      # K/V tile of k_attention_d64_p: the lazy-max rule is applied once per row and tile
THRESHOLD = 8.0                 # the reference max moves when a tile's row max exceeds it by more than 2^8 in P
C1 = C2 = 2.0 ** -10


def scale_log2(scale):
    """scale * log2(e) as the kernel holds it (fp32)."""
    return float(torch.tensor(scale, dtype=torch.float32) * torch.tensor(LOG2E, dtype=torch.float32))


def _heads(t, b, n, heads):
    return t[:, :heads * 64].reshape(b, n, heads, 64).transpose(1, 2)


def reference(q, k, v, b, heads, nq, nkv, scale, causal=False, max_elems=1 << 26):
    """(O64, PV): softmax(scale q k^T) v and softmax(scale q k^T) |v| in float64, each [b*nq, heads*64], on q's device.
    q, k, v may be row-strided views; the scores are formed in chunks of (batch, heads) of at most max_elems elements.
    causal: key j is visible to query i iff j <= i (top-left aligned, as SDPA's is_causal)."""
    o = torch.empty((b, nq, heads, 64), dtype=torch.float64, device=q.device)
    pv = torch.empty_like(o)
    hc = max(1, min(heads, max_elems // (nq * nkv)))
    mask = torch.ones((nq, nkv), dtype=torch.bool, device=q.device).tril() if causal else None
    for bi in range(b):
        qb, kb, vb = q[bi * nq:(bi + 1) * nq], k[bi * nkv:(bi + 1) * nkv], v[bi * nkv:(bi + 1) * nkv]
        for h0 in range(0, heads, hc):
            h1 = min(heads, h0 + hc)
            qh = qb[:, h0 * 64:h1 * 64].double().reshape(nq, h1 - h0, 64).transpose(0, 1)
            kh = kb[:, h0 * 64:h1 * 64].double().reshape(nkv, h1 - h0, 64).transpose(0, 1)
            vh = vb[:, h0 * 64:h1 * 64].double().reshape(nkv, h1 - h0, 64).transpose(0, 1)
            s = torch.matmul(qh, kh.transpose(1, 2)) * scale
            if mask is not None:
                s = s.masked_fill(~mask, -math.inf)
            p = torch.softmax(s, dim=-1)
            o[bi, :, h0:h1] = torch.matmul(p, vh).transpose(0, 1)
            pv[bi, :, h0:h1] = torch.matmul(p, vh.abs()).transpose(0, 1)
            del s, p
    return o.view(b * nq, heads * 64), pv.view(b * nq, heads * 64)


def tolerance(o64, pv, c1=C1, c2=C2):
    return c1 * pv + c2 * o64.abs() + 2.0 ** -24


def err_ratio(out, o64, pv, c1=C1, c2=C2):
    """max over elements of |out - O64| / tol (NaN if out has a non-finite value)."""
    d = out.to(o64.device).double() - o64
    r = (d.abs() / tolerance(o64, pv, c1, c2)).max()
    return float("nan") if not torch.isfinite(out).all() else float(r)


# ------------------------------------------------------------------ lazy-max replay
def scores32(q, k, b, heads, nq, nkv):
    """Raw scores q k^T in fp32 (the kernel's tcgen05 accumulator), [b, heads, nq, nkv]."""
    return torch.matmul(_heads(q, b, nq, heads).float(), _heads(k, b, nkv, heads).float().transpose(-1, -2))


def replay(s, sl2, tile=TILE):
    """The lazy reference-max rule of k_attention_d64_p on fp32 scores s [..., nq, nkv].  Returns (overshoot, moved), each
    [..., nq, n_tiles]: overshoot = (tile max - reference max) * sl2 in fp32 (NaN for the first tile, whose max always
    becomes the reference) and whether the reference moved."""
    nkv = s.shape[-1]
    nt = (nkv + tile - 1) // tile
    sl2 = torch.tensor(sl2, dtype=torch.float32)
    ov = torch.full(s.shape[:-1] + (nt,), math.nan)
    moved = torch.zeros(s.shape[:-1] + (nt,), dtype=torch.bool)
    m = None
    for j in range(nt):
        mx = s[..., j * tile:min(nkv, (j + 1) * tile)].float().amax(-1)
        if j == 0:
            m, moved[..., 0] = mx, True
            continue
        o = (mx - m) * sl2
        ov[..., j] = o
        mv = o > THRESHOLD
        moved[..., j] = mv
        m = torch.where(mv, torch.maximum(mx, m), m)
    return ov, moved


def emulate_p(q, k, v, b, heads, nq, nkv, scale, rescale_o=True):
    """k_attention_d64_p's arithmetic in torch (fp32 unless stated): P rounded to fp16 against the lazily moved reference max,
    the cubic exp2 on two of every eight columns, l summed from the unrounded p, O rescaled by exp2(m_old - m_new) when the
    reference moves (skipped with rescale_o=False), fp16 output."""
    sl2 = scale_log2(scale)
    s = scores32(q, k, b, heads, nq, nkv)
    vh = _heads(v, b, nkv, heads).float()
    emu = (torch.arange(TILE) % 8) >= 6
    m = torch.full(s.shape[:-1], -math.inf)
    l = torch.zeros(s.shape[:-1])
    o = torch.zeros(s.shape[:-1] + (64,))
    for j in range((nkv + TILE - 1) // TILE):
        sj = s[..., j * TILE:(j + 1) * TILE]
        mx = sj.amax(-1)
        move = (mx - m) * sl2 > THRESHOLD if j else torch.ones_like(mx, dtype=torch.bool)
        m_new = torch.where(move, torch.maximum(mx, m), m)
        alpha = torch.where(move, torch.exp2((m - m_new) * sl2), torch.ones_like(m))
        m = m_new
        x = sj * sl2 - (m * sl2)[..., None]
        p = torch.where(emu[:sj.shape[-1]], ex2_cubic(x), torch.exp2(x))
        l = l * alpha + p.sum(-1)
        o = (o * alpha[..., None] if rescale_o else o) + p.half().float() @ vh[..., j * TILE:(j + 1) * TILE, :]
    return (o / l[..., None]).half().transpose(1, 2).reshape(b * nq, heads * 64)


def ex2_cubic(x):
    """ex2_emulated of attention.cu in fp32: 2^floor(x) * cubic(x - floor(x)), x clamped to >= -126."""
    x = x.clamp_min(-126.0)
    n = torch.floor(x)
    f = x - n
    c = ((0.0771190897 * f + 0.2275643945) * f + 0.6951461434) * f + 1.0
    return torch.ldexp(c, n)


# ------------------------------------------------------------------ input generators
def _gen(seed):
    return torch.Generator("cpu").manual_seed(seed)


def tile_signature_v(b, nkv, heads, g, noise=0.05):
    """V whose column (tile index mod 64) is 1 on the keys of that K/V tile, plus N(0, noise^2): a tile that is dropped or
    weighted wrongly moves its own column."""
    tiles = torch.arange(nkv) // TILE
    onehot = torch.nn.functional.one_hot(tiles % 64, 64).float()
    v = onehot[None, :, None, :] + noise * torch.randn((b, nkv, heads, 64), generator=g)
    return v.reshape(b * nkv, heads * 64).half()


# Per-tile overshoot classes (log2 units) of the late-max rows.  Rows below 8 accumulate k * w until that passes 8 and then
# move (0.37 -> 7.77 then 8.14, 2.7 -> 8.1, 3.1 -> 9.3, 7.93 -> 15.86, ...); 8.6 and up move on every tile; 130 and 300 make
# the optimistic first-half exponentials overflow, so that half must be recomputed.  With STRADDLE the class list has 13 entries,
# prime to the 32 rows of a warp, so every warp mixes moving and non-moving rows.  STRADDLE lands within 2^-8 of the threshold: its
# outcome may differ in the last bits between the CPU replay and the tensor cores, and no test depends on it.
LATE_MAX_W = (0.37, 1.3, 2.7, 3.1, 7.93, 8.6, 9.5, 12.0, 17.0, 40.0, 130.0, 300.0)
STRADDLE = -1.0


def late_max_classes(nq, bh):
    classes = list(LATE_MAX_W) + [STRADDLE]
    return [classes[(i + 5 * bh) % len(classes)] for i in range(nq)]


def late_max(b, heads, nq, nkv, seed, scale=0.125):
    """Row maxima that grow from tile to tile.  q_i = a_i e_0, k_j[0] = t + 0 at one peak key per tile t and t - U(0.25, 2)
    elsewhere, so the row max of tile t is a_i * t exactly (fp16 products are exact in fp32) and a_i = w / (scale log2 e)
    sets the per-tile overshoot w of row i (LATE_MAX_W).  The peak sits in the first half of even tiles, the second half of
    odd ones, and on the last valid key of the last tile.  V carries a per-tile signature."""
    g = _gen(seed)
    sl2 = scale_log2(scale)
    nt = (nkv + TILE - 1) // TILE
    q = torch.zeros((b, nq, heads, 64))
    k = torch.zeros((b, nkv, heads, 64))
    t = (torch.arange(nkv) // TILE).float()
    for bi in range(b):
        for h in range(heads):
            bh = bi * heads + h
            w = torch.tensor([THRESHOLD if c == STRADDLE else c for c in late_max_classes(nq, bh)])
            q[bi, :, h, 0] = w / sl2
            kk = t - torch.round((0.25 + 1.75 * torch.rand(nkv, generator=g)) * 32) / 32
            for j in range(nt):
                lo, hi = j * TILE, min(nkv, (j + 1) * TILE)
                if j == nt - 1:
                    pos = hi - 1
                else:
                    half = j % 2
                    pos = lo + 64 * half + int(torch.randint(0, 64, (1,), generator=g))
                kk[pos] = j
            k[bi, :, h, 0] = kk
            k[bi, :, h, 1:] = torch.randn((nkv, 63), generator=g)
    v = tile_signature_v(b, nkv, heads, g)
    return q.reshape(b * nq, heads * 64).half(), k.reshape(b * nkv, heads * 64).half(), v


def all_negative(b, heads, nq, nkv, seed, scale=0.125):
    """Every score strongly negative: q[:, 0] = 18, k[:, 0] = -18 shift the logits by -324 while the other 63 dimensions give
    them a spread of ~8, so every row max is below -30 in scaled log2 units (for scale 0.125) and P against a reference of 0 --
    a zero-filled key past nkv that slipped into the max -- underflows fp16.  V carries a per-tile signature."""
    g = _gen(seed)
    q = torch.randn((b, nq, heads, 64), generator=g)
    k = torch.randn((b, nkv, heads, 64), generator=g)
    q[..., 0] = 18.0
    k[..., 0] = -18.0
    v = tile_signature_v(b, nkv, heads, g)
    return q.reshape(b * nq, heads * 64).half(), k.reshape(b * nkv, heads * 64).half(), v


def constant_rows(b, heads, nq, nkv, seed, scale=0.125):
    """q_i = a_i e_0 and k_j[0] = 3 for every key: each row's scores are one constant, so its output is the mean of V."""
    g = _gen(seed)
    q = torch.zeros((b, nq, heads, 64))
    q[..., 0] = torch.randn((b, nq, heads), generator=g) * 8
    k = torch.randn((b, nkv, heads, 64), generator=g)
    k[..., 0] = 3.0
    q[..., 1:] = 0.0
    v = torch.randn((b * nkv, heads * 64), generator=g)
    return q.reshape(b * nq, heads * 64).half(), k.reshape(b * nkv, heads * 64).half(), v.half()


def normal(b, heads, nq, nkv, seed, scale=0.125):
    """N(0, 1) q, k, v.  With scale 1.0 instead of 1/sqrt(64) the logits have a spread of ~8 and the rows are peaked."""
    g = _gen(seed)
    return tuple(torch.randn((b * n, heads * 64), generator=g).half() for n in (nq, nkv, nkv))


GENERATORS = {"late_max": late_max, "all_negative": all_negative, "constant": constant_rows, "normal": normal}

# Shapes of the self-attention (k_attention_d64_p) rescale tests: key counts with ragged last tiles of 1, 69, 1, 77 and 17 keys
# and 2 to 32 tiles; 300 queries make two 256-row items per (batch, head), the second with 44 rows.
P_B, P_HEADS, P_NQ = 2, 3, 300
P_NKV = (129, 197, 257, 333, 785, 1024, 4096)
# Key counts of the cross-attention (k_attention_d64_kv1) tests: one to a full 128-key tile, not only multiples of 16.
KV1_NKV = (1, 15, 16, 17, 77, 127, 128)
KV1_B, KV1_HEADS, KV1_NQ = 2, 3, 300
