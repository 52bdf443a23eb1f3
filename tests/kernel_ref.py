"""Float64 references, per-element error bars and tile-level failure reports for the tcgen05 kernels (not a test
module; imported by tests/test_kernel_ref_cpu.py and tests/test_kernels_at_scale_gpu.py).

References take the exact fp16 operands the kernel read and evaluate the layer in float64 (torch, on the operands'
device), chunked so that the float64 intermediates stay near `budget_bytes`:

* GEMM layer:  y = fp16(relu(acc + bias + res) + pe),  acc = x (*) w  -- the order of the epilogue in
  csrc/fp_gemm.cu (fp32: +bias, +residual, ReLU, +positional embedding, one rounding to fp16).
* Attention:   y = fp16(softmax(q k^T / sqrt(128)) v)  per (sequence, head[, group]).

Error model (the bar every output element is held to):

GEMM.  The kernel multiplies fp16 operands exactly and adds them into an fp32 accumulator, one tcgen05 MMA of K = 16
per step, so `steps` = ceil(K / 16) (the stem: 28 MMAs of 7 filter rows x 4 tap pairs).  Each step may lose up to
2^-22 of the sum of the magnitudes it has added so far (a truncating fp32 add, 2^-23, with one bit of slack for the
alignment of the 16 products); the epilogue's two fp32 adds (bias, residual) and the post-activation add lose as much
again.  ReLU is 1-Lipschitz, and the final rounding to fp16 costs half an ulp of the kernel's value, at most one ulp of
the reference.  So, with  S = |x| (*) |w| + |bias| + |res| + |pe|  computed by a second float64 pass on the absolute
values,

    |y_kernel - y_ref| <= ulp16(y_ref) + 2^-22 * (steps + 2) * S.

Unlike a flat `atol + rtol * |ref|` this grows with the contraction depth and the operands' magnitude, and it is tight on
outputs near zero, where a flat absolute term hides small errors.

Attention.  Per query row: S = q k^T in fp32 (8 MMA steps of K = 16, error <= 2^-22 * 10 * (|q| |k|^T)), the scaled
logits through exp2 (relative error 2^-22 plus the argument's rounding), P = exp(s - max) rounded to fp16 (relative
2^-11, or 2^-25 absolute below fp16's normal range), the row sum l in fp32 (400 adds: 402 * 2^-24 relative), O = P v in
fp32 (25 MMA steps).  With  eps_p = 2 * scale * 2^-22 * 10 * max_j(|q| |k_j|) + 2^-22 * (2 + max_j |s_j| * log2 e),

    |y_kernel - y_ref| <= ulp16(y_ref) + ((2^-11 + eps_p + 27 * 2^-22) * (p (*) |v|) + 2^-25 * sum_j |v_j|) / l
                          + (402 * 2^-24 + eps_p) * |y_ref|.

On failure the checker names the failing tiles, not only the worst element: image, tile row and column, channel block,
and -- from the launch plan (foundationpose_b200.ops.gemm_last_plan) -- the work tile, the CTA that ran it and in which
of its loop iterations.
"""
import math

import torch
import torch.nn.functional as F

U22 = 2.0 ** -22
LOG2E = 1.4426950408889634
ATTN_SCALE = 1.0 / math.sqrt(128.0)


def fp16_ulp(x):
    """Spacing of fp16 numbers at |x| (2^-24 in the subnormal range), float64."""
    x = x.double().abs()
    e = torch.floor(torch.log2(x.clamp_min(2.0 ** -14)))
    return torch.pow(2.0, e - 10.0)


# --------------------------------------------------------------------------------------------------------- GEMM layers
def _epilogue(acc, mag, bias, res, pe, relu, steps):
    """acc / mag: float64 [..., Co] of x (*) w and |x| (*) |w|; res NHWC-shaped like acc; pe [Ho*Wo, Co] broadcast."""
    y = acc + bias.double()
    mag = mag + bias.double().abs()
    if res is not None:
        y = y + res.double()
        mag = mag + res.double().abs()
    if relu:
        y = y.clamp_min(0.0)
    if pe is not None:
        pe = pe.double().reshape(y.shape[1:])
        y = y + pe
        mag = mag + pe.abs()
    return y, fp16_ulp(y) + U22 * (steps + 2) * mag


def conv_reference(x, w, bias, *, stride=1, res=None, post_add=None, relu=False, steps=None):
    """x fp16 NHWC [n, H, W, Ci]; w [Co, Ci, k, k] (fp16 values); bias [Co]; res fp16 NHWC like the output; post_add
    [Ho*Wo, Co].  Padding k // 2.  -> (ref, bar) float64 NHWC [n, Ho, Wo, Co]."""
    k = w.shape[-1]
    if steps is None:
        steps = math.ceil(w.shape[1] * k * k / 16)
    xd = x.permute(0, 3, 1, 2).double()
    wd = w.double()
    acc = F.conv2d(xd, wd, stride=stride, padding=k // 2).permute(0, 2, 3, 1)
    mag = F.conv2d(xd.abs(), wd.abs(), stride=stride, padding=k // 2).permute(0, 2, 3, 1)
    return _epilogue(acc, mag, bias, res, post_add, relu, steps)


def linear_reference(x, w, bias, *, res=None, relu=False):
    """x fp16 [M, K]; w [Co, K]; res fp16 [M, Co] -> (ref, bar) float64 shaped [1, 1, M, Co] (the kernel's view: one
    image, one row of M pixels)."""
    xd, wd = x.double(), w.double()
    acc, mag = xd @ wd.t(), xd.abs() @ wd.abs().t()
    ref, bar = _epilogue(acc[None, None], mag[None, None], bias, None if res is None else res[None, None], None, relu,
                         math.ceil(x.shape[1] / 16))
    return ref, bar


# ------------------------------------------------------------------------------------------------------- tile geometry
class TileMap:
    """Which tile, work tile and CTA produced output element (image, row, column, channel) of one launch, from the plan
    fp_op_gemm_last_plan reported (ops.gemm_last_plan) and the output's spatial size (LINEAR: 1 x M)."""

    def __init__(self, plan, Ho, Wo):
        self.p = plan
        self.tiles_w = -(-Wo // plan["bw"])
        self.tiles_h = -(-Ho // plan["bh"])

    def locate(self, img, i, j, c):
        p = self.p
        tw, th, tn, cb = j // p["bw"], i // p["bh"], img // p["bimg"], c // p["bn"]
        m_tile = (tn * self.tiles_h + th) * self.tiles_w + tw
        d = dict(img=img, tile_row=th, tile_col=tw, cblock=cb, m_tile=m_tile)
        if p["kernel"] == "tile":
            cg = p["cg"]
            vt = (m_tile // cg) * p["n_tiles"] + cb
            slots = p["grid"] // cg
            d.update(work_tile=vt, cta=(vt % slots) * cg + m_tile % cg, iteration=vt // slots)
        else:
            if p["kernel"] == "swap":
                vt = (m_tile // 2) * p["n_tiles"] + cb
            elif p["kernel"] == "swap_patch":
                vt = m_tile * p["n_tiles"] + cb
            else:  # stem: one 16 x 8 tile of 64 channels per work tile
                vt = m_tile
            d.update(work_tile=vt, cta=vt % p["grid"], iteration=vt // p["grid"])
        return d

    def describe(self, d):
        p = self.p
        return (f"image {d['img']} tile (row {d['tile_row']}, col {d['tile_col']}) channels "
                f"[{d['cblock'] * p['bn']}, {(d['cblock'] + 1) * p['bn']}): work tile {d['work_tile']} = CTA {d['cta']}, "
                f"iteration {d['iteration']}")


def plan_name(plan):
    """'tile<256,2,4,patch>' / 'swap' / 'swap_patch' / 'stem'."""
    if plan["kernel"] != "tile":
        return plan["kernel"]
    return f"tile<{plan['bn']},{plan['cg']},{plan['slabs']}{',patch' if plan['patch'] else ''}>"


def tiles_per_cta(plan):
    return plan["work_tiles"] / plan["grid"]


# ------------------------------------------------------------------------------------------------------------ checking
class Result:
    """Outcome of one comparison: worst error in fp16 ulps of the reference and as a fraction of the bar, the number
    of elements over the bar, and per-tile failure records."""

    def __init__(self, what):
        self.what = what
        self.max_ulps = 0.0
        self.max_ratio = 0.0
        self.n_bad = 0
        self.n = 0
        self.tiles = {}  # key -> [count, worst ratio, err, ref, got, (img, i, j, c)]

    @property
    def ok(self):
        return self.n_bad == 0

    def _note(self, key, cnt, ratio, err, ref, got, where):
        t = self.tiles.get(key)
        if t is None:
            self.tiles[key] = [cnt, ratio, err, ref, got, where]
        else:
            t[0] += cnt
            if ratio > t[1]:
                t[1:] = [ratio, err, ref, got, where]

    def report(self, tilemap=None, limit=12):
        head = (f"{self.what}: {self.n_bad} of {self.n} elements over the bar in {len(self.tiles)} tiles; worst "
                f"{self.max_ratio:.3g} x bar, {self.max_ulps:.3g} fp16 ulps")
        lines = [head]
        for key, (cnt, ratio, err, ref, got, where) in sorted(self.tiles.items(), key=lambda kv: -kv[1][1])[:limit]:
            loc = tilemap.describe(tilemap.locate(*where)) if tilemap else f"tile {key}"
            lines.append(f"  {loc}: {cnt} elements over the bar, worst at (image, row, col, ch) {where}: "
                         f"got {got:.6g} ref {ref:.6g} err {err:.3g} = {ratio:.3g} x bar")
        if len(self.tiles) > limit:
            lines.append(f"  ... {len(self.tiles) - limit} more tiles")
        return "\n".join(lines)


def _tile_keys(idx, tile):
    """idx [k, 4] (image, row, col, channel) -> one int64 key per tile of shape `tile` = (bimg, bh, bw, bn)."""
    bimg, bh, bw, bn = tile
    return ((idx[:, 0] // bimg) << 44) | ((idx[:, 1] // bh) << 28) | ((idx[:, 2] // bw) << 12) | (idx[:, 3] // bn)


def _tile_of(plan):
    return (1, 8, 8, 64) if plan is None else (plan["bimg"], plan["bh"], plan["bw"], plan["bn"])


def _note_tiles(result, idx, score, err, ref, got, tile, offset, limit=64):
    """Groups the flagged elements idx [k, 4] (absolute indices; `offset` maps them back into err / ref / got) by tile
    and records the `limit` worst tiles in `result`."""
    keys = _tile_keys(idx, tile)
    uk, inv = torch.unique(keys, return_inverse=True)
    counts = torch.bincount(inv, minlength=len(uk))
    worst = torch.full((len(uk),), -1.0, dtype=score.dtype, device=score.device).scatter_reduce(0, inv, score, "amax")
    for k in worst.argsort(descending=True)[:limit].tolist():
        sel = (inv == k).nonzero()[:, 0]
        w = idx[sel[score[sel].argmax()]]
        rel = tuple(int(v) - o for v, o in zip(w, offset))
        result._note(int(uk[k]), int(counts[k]), float(worst[k]), float(err[rel]), float(ref[rel]), float(got[rel]),
                     tuple(int(v) for v in w))


def compare(got, ref, bar, *, result, tile, offset=(0, 0, 0, 0)):
    """Accumulates |got - ref| against `bar` (all [n, Ho, Wo, Co]) into `result`; `offset` is the position of this
    chunk in the whole launch's output (so that tiles are named in the launch's numbering)."""
    got = got.double()
    err = (got - ref).abs()
    err = torch.where(torch.isnan(got), torch.full_like(err, math.inf), err)
    ratio = err / bar
    result.n += err.numel()
    result.max_ulps = max(result.max_ulps, float((err / fp16_ulp(ref)).max()))
    result.max_ratio = max(result.max_ratio, float(ratio.max()))
    bad = ratio > 1.0
    nb = int(bad.sum())
    if nb:
        result.n_bad += nb
        idx = bad.nonzero() + torch.tensor(offset, device=bad.device)
        _note_tiles(result, idx, ratio[bad], err, ref, got, tile, offset)
    return result


def check_chunked(got, reference, *, what, plan=None, ranges=None, chunk_dim=0, budget_bytes=4 << 30):
    """Compares `got` [n, Ho, Wo, Co] with reference(lo, hi) -> (ref, bar) of indices lo:hi along `chunk_dim` (images
    of a convolution: 0, rows of a LINEAR: 2), over `ranges` [(lo, hi)] of that axis (default all), in chunks whose
    float64 work (about eight arrays of the output chunk's size) stays near `budget_bytes`."""
    res = Result(what)
    tile = _tile_of(plan)
    size = got.shape[chunk_dim]
    step = max(1, budget_bytes // (max(1, got.numel() // size) * 8 * 8))
    for lo, hi in ranges or [(0, size)]:
        for a in range(lo, hi, step):
            b = min(hi, a + step)
            ref, bar = reference(a, b)
            off = [0, 0, 0, 0]
            off[chunk_dim] = a
            compare(got.narrow(chunk_dim, a, b - a), ref, bar, result=res, tile=tile, offset=tuple(off))
            del ref, bar
    return res


def bitwise_diff(a, b, *, what, plan=None):
    """Result over the elements of two fp16 tensors [n, Ho, Wo, Co] whose bits differ (bar 0)."""
    res = Result(what)
    d = a.view(torch.int16) != b.view(torch.int16)
    res.n = d.numel()
    nb = int(d.sum())
    if nb:
        res.n_bad = nb
        res.max_ratio = math.inf
        err = (a.double() - b.double()).abs()
        _note_tiles(res, d.nonzero(), err[d], err, b, a, _tile_of(plan), (0, 0, 0, 0))
    return res


# ------------------------------------------------------------------------------------------------------------ attention
def attention_reference(qkv, n_groups, b0, b1):
    """qkv fp16 [B*400, 1536 * n_groups] (per group: q | k | v, 4 heads of 128) -> (ref, bar) float64 of sequences
    b0:b1, shaped [n_groups, (b1 - b0) * 400, 512] like ops.attention_grouped's output."""
    T, H, D = 400, 4, 128
    x = qkv[b0 * T:b1 * T].double().reshape(b1 - b0, T, n_groups, 3, H, D).permute(2, 3, 0, 4, 1, 5)  # g, qkv, b, h, t, d
    q, k, v = x[:, 0], x[:, 1], x[:, 2]
    S = q @ k.transpose(-1, -2)
    A = q.abs() @ k.abs().transpose(-1, -2)
    s = S * ATTN_SCALE
    m = s.amax(-1, keepdim=True)
    p = torch.exp(s - m)
    l = p.sum(-1, keepdim=True)
    ref = (p @ v) / l
    pav = p @ v.abs()
    vsum = v.abs().sum(-2, keepdim=True)
    eps_p = (2 * ATTN_SCALE * U22 * 10) * A.amax(-1, keepdim=True) + U22 * (2 + s.abs().amax(-1, keepdim=True) * LOG2E)
    bar = (fp16_ulp(ref) + ((2.0 ** -11 + eps_p + 27 * U22) * pav + 2.0 ** -25 * vsum) / l
           + (402 * 2.0 ** -24 + eps_p) * ref.abs())
    shape = (n_groups, (b1 - b0) * T, H * D)
    return ref.permute(0, 1, 3, 2, 4).reshape(shape), bar.permute(0, 1, 3, 2, 4).reshape(shape)


def check_attention(got, qkv, n_groups, *, what, budget_bytes=4 << 30):
    """got [n_groups, B*400, 512] (or [B*400, 512] for one group).  Failing tiles are (group, sequence, 128-query tile,
    head)."""
    if got.dim() == 2:
        got = got[None]
    B = qkv.shape[0] // 400
    res = Result(what)
    per = n_groups * 4 * 400 * 400 * 8 * 6
    step = max(1, budget_bytes // per)
    for b0 in range(0, B, step):
        b1 = min(B, b0 + step)
        ref, bar = attention_reference(qkv, n_groups, b0, b1)
        g = got[:, b0 * 400:b1 * 400]
        # [g, b*400 + t, h*128 + d] -> (image = g * B + b, row = t, col = 0, channel = h*128 + d): tiles of 128 rows
        shp = (n_groups * (b1 - b0), 400, 1, 512)
        sub = Result(what)
        compare(g.reshape(shp), ref.reshape(shp), bar.reshape(shp), result=sub, tile=(1, 128, 1, 128))
        res.n += sub.n
        res.n_bad += sub.n_bad
        res.max_ulps = max(res.max_ulps, sub.max_ulps)
        res.max_ratio = max(res.max_ratio, sub.max_ratio)
        nb = b1 - b0
        for cnt, ratio, err, r, gv, (img, t, _, c) in sub.tiles.values():
            grp, seq = img // nb, b0 + img % nb
            res._note((grp, seq, t // 128, c // 128), cnt, ratio, err, r, gv, (grp, seq, t, c))
    return res


def attention_report(res, limit=12):
    lines = [f"{res.what}: {res.n_bad} of {res.n} elements over the bar in {len(res.tiles)} tiles; worst "
             f"{res.max_ratio:.3g} x bar, {res.max_ulps:.3g} fp16 ulps"]
    for key, (cnt, ratio, err, ref, got, (g, b, t, c)) in sorted(res.tiles.items(), key=lambda kv: -kv[1][1])[:limit]:
        lines.append(f"  group {g} sequence {b} query tile {t // 128} head {c // 128}: {cnt} elements over the bar, worst "
                     f"at query {t} dim {c % 128}: got {got:.6g} ref {ref:.6g} err {err:.3g} = {ratio:.3g} x bar")
    return "\n".join(lines)


def attention_inputs(kind, B, n_groups, *, seed, device):
    """Seeded qkv fp16 [B*400, 1536 * n_groups]:
    'std'   q, k, v ~ N(0, 1.5^2) (the existing attention test's distribution);
    'sharp' one key dominates every query: q_i = k_pi(i) scaled so that its logit q.k / sqrt(128) is 30, the others
            ~ N(0, 2.7^2), so p is ~1 for one key and below e^-15 for nearly all others;
    'flat'  all keys of a (sequence, head) identical: every logit equal, the output is the mean of v."""
    g = torch.Generator(device=device).manual_seed(seed)
    shape = (B, 400, n_groups, 4, 128)

    def r(scale=1.0, shp=shape):
        return torch.randn(shp, generator=g, device=device) * scale

    if kind == "std":
        q, k, v = r(1.5), r(1.5), r(1.5)
    elif kind == "sharp":
        k, v = r(), r()
        kp = k[:, torch.randperm(400, generator=g, device=device)]
        q = kp * (30.0 * math.sqrt(128.0) / (kp * kp).sum(-1, keepdim=True))
    elif kind == "flat":
        q, v = r(1.5), r(1.5)
        k = r(1.5, (B, 1, n_groups, 4, 128)).expand(shape)
    else:
        raise ValueError(kind)
    return torch.stack([q, k, v], 3).reshape(B * 400, n_groups * 1536).half()
