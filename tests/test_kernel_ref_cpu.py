"""CPU: the float64 checker of tests/kernel_ref.py accepts what a correct kernel produces (the fp16 rounding of the
float64 result, and an fp32-accumulating emulation of the kernels' arithmetic) and rejects, at small shapes, the
faults a tiled tensor-core kernel typically has -- naming the tile."""
import math

import pytest
import torch
import torch.nn.functional as F

import kernel_ref as kr

N, H, CI, CO = 4, 16, 128, 128
# a plan as fp_op_gemm_last_plan reports it: 8 x 8 pixels x 2 images x 64 channels per tile
PLAN = dict(kernel="tile", bn=64, cg=1, slabs=2, patch=0, grid=5, work_tiles=32, bw=8, bh=8, bimg=2, m_tiles=8, n_tiles=2)


@pytest.fixture(scope="module")
def conv():
    g = torch.Generator().manual_seed(0)
    x = torch.randn(N, H, H, CI, generator=g).half()
    w = (torch.randn(CO, CI, 3, 3, generator=g) * (9 * CI) ** -0.5).half()
    b = torch.randn(CO, generator=g)
    res = torch.randn(N, H, H, CO, generator=g).half()
    pe = torch.randn(H * H, CO, generator=g)
    ref, bar = kr.conv_reference(x, w, b, res=res, post_add=pe, relu=True)
    return dict(x=x, w=w, b=b, res=res, pe=pe, ref=ref, bar=bar)


def _acc32(c, w=None):
    x = c["x"].permute(0, 3, 1, 2).float()
    return F.conv2d(x, (c["w"] if w is None else w).float(), padding=1).permute(0, 2, 3, 1)


def _epi32(c, acc, res=True, pe_first=False):
    y = acc + c["b"]
    if res:
        y = y + c["res"].float()
    pe = c["pe"].reshape(H, H, CO)
    if pe_first:
        return (y + pe).relu().half()
    return (y.relu() + pe).half()


def _check(c, got):
    return kr.check_chunked(got, lambda a, b: (c["ref"][a:b], c["bar"][a:b]), what="conv", plan=PLAN)


def _rejects(c, got, img=None, row=None, col=None, cblock=None):
    r = _check(c, got)
    assert not r.ok, "checker accepted a faulty output"
    tm = kr.TileMap(PLAN, H, H)
    rep = r.report(tm)
    if img is not None:
        d = tm.locate(*max(r.tiles.values(), key=lambda t: t[1])[5])
        assert (d["img"], d["tile_row"], d["tile_col"], d["cblock"]) == (img, row, col, cblock), rep
        assert len(r.tiles) == 1, rep  # the fault is confined to that tile, and the report says so
        assert f"image {img} tile (row {row}, col {col})" in rep
    return r


def test_accepts_fp16_rounding_of_float64(conv):
    r = _check(conv, conv["ref"].half())
    assert r.ok and r.max_ratio < 0.51 and r.max_ulps < 0.501, r.report()  # torch rounds float64 -> fp32 -> fp16


def test_accepts_fp32_accumulation(conv):
    r = _check(conv, _epi32(conv, _acc32(conv)))
    assert r.ok, r.report()
    assert r.max_ratio < 0.6


def test_rejects_tile_copied_from_neighbour(conv):
    got = _epi32(conv, _acc32(conv))
    got[1, 8:16, 0:8, :] = got[1, 8:16, 8:16, :]
    # both 64-channel blocks of that pixel tile are wrong
    r = _check(conv, got)
    assert not r.ok
    blocks = {kr.TileMap(PLAN, H, H).locate(*t[5])["cblock"] for t in r.tiles.values()}
    assert blocks == {0, 1} and all(t[5][0] == 1 and t[5][1] // 8 == 1 and t[5][2] // 8 == 0 for t in r.tiles.values())


def test_rejects_one_dropped_k_block(conv):
    w = conv["w"].clone()
    w[:, 64:128, 1, 2] = 0  # tap (1, 2), second 64-channel k-block
    got = _epi32(conv, _acc32(conv))
    got[2, 0:8, 8:16, 0:64] = _epi32(conv, _acc32(conv, w))[2, 0:8, 8:16, 0:64]
    _rejects(conv, got, img=2, row=0, col=1, cblock=0)


def test_rejects_fp16_accumulation(conv):
    x = conv["x"].permute(0, 3, 1, 2).float()
    cols = F.unfold(x, 3, padding=1)  # [n, Ci*9, H*W]
    wf = conv["w"].float().reshape(CO, -1)
    acc = torch.zeros(N, CO, H * H, dtype=torch.float16)
    for k0 in range(0, wf.shape[1], 16):  # one K = 16 MMA step at a time, accumulator kept in fp16
        acc = (acc.float() + torch.einsum("ok,nkl->nol", wf[:, k0:k0 + 16], cols[:, k0:k0 + 16])).half()
    got = _epi32(conv, acc.float().reshape(N, CO, H, H).permute(0, 2, 3, 1))
    r = _rejects(conv, got)
    assert r.n_bad > 100


def test_rejects_missing_residual_on_one_tile(conv):
    got = _epi32(conv, _acc32(conv))
    got[3, 8:16, 8:16, 64:128] = _epi32(conv, _acc32(conv), res=False)[3, 8:16, 8:16, 64:128]
    _rejects(conv, got, img=3, row=1, col=1, cblock=1)


def test_rejects_positional_embedding_before_relu(conv):
    _rejects(conv, _epi32(conv, _acc32(conv), pe_first=True))


def test_linear_reference_and_row_chunks():
    g = torch.Generator().manual_seed(1)
    M, K, C = 300, 128, 64
    x = torch.randn(M, K, generator=g).half()
    w = (torch.randn(C, K, generator=g) * K ** -0.5).half()
    b = torch.randn(C, generator=g)
    good = (x.float() @ w.float().t() + b).half()[None, None]
    plan = dict(PLAN, bw=128, bh=1, bimg=1, bn=64, n_tiles=1, m_tiles=3, grid=3, work_tiles=3)
    refn = lambda a, c: kr.linear_reference(x[a:c], w, b)  # noqa: E731
    r = kr.check_chunked(good, refn, what="linear", plan=plan, chunk_dim=2, budget_bytes=64 * 64 * 64)
    assert r.ok, r.report()
    bad = good.clone()
    bad[0, 0, 260, 5] += 0.05  # row 260: third 128-row tile, the last and partial one
    r = kr.check_chunked(bad, refn, what="linear", plan=plan, chunk_dim=2, budget_bytes=64 * 64 * 64)
    assert not r.ok and list(r.tiles.values())[0][5] == (0, 0, 260, 5)
    assert "tile (row 0, col 2)" in r.report(kr.TileMap(plan, 1, M))


def _schedule(plan, Ho, Wo):
    """(cta, iteration) of every (m_tile, channel block), walking the kernels' persistent loops as the CUDA code does."""
    p, out = plan, {}
    if p["kernel"] == "tile":
        cg, slots = p["cg"], p["grid"] // p["cg"]
        total_vt = -(-p["m_tiles"] // cg) * p["n_tiles"]
        for cta in range(p["grid"]):
            for it, vt in enumerate(range(cta // cg, total_vt, slots)):
                m = (vt // p["n_tiles"]) * cg + cta % cg
                if m < p["m_tiles"]:
                    out[(m, vt % p["n_tiles"])] = (cta, it)
    else:
        pair = p["kernel"] == "swap"
        total_vt = (-(-p["m_tiles"] // 2) if pair else p["m_tiles"]) * p["n_tiles"]
        for cta in range(p["grid"]):
            for it, vt in enumerate(range(cta, total_vt, p["grid"])):
                for m in ((2 * (vt // p["n_tiles"]), 2 * (vt // p["n_tiles"]) + 1) if pair else (vt // p["n_tiles"],)):
                    if m < p["m_tiles"]:
                        out[(m, vt % p["n_tiles"])] = (cta, it)
    return out


@pytest.mark.parametrize("plan", [
    dict(kernel="tile", bn=256, cg=2, slabs=4, patch=1, grid=148, bw=8, bh=8, bimg=2, n_tiles=1),
    dict(kernel="tile", bn=256, cg=2, slabs=2, patch=0, grid=148, bw=4, bh=4, bimg=8, n_tiles=2),
    dict(kernel="swap", bn=128, cg=1, slabs=0, patch=0, grid=148, bw=8, bh=8, bimg=2, n_tiles=1),
    dict(kernel="swap_patch", bn=128, cg=1, slabs=0, patch=1, grid=148, bw=8, bh=8, bimg=4, n_tiles=1),
    dict(kernel="stem", bn=64, cg=1, slabs=0, patch=0, grid=148, bw=8, bh=16, bimg=1, n_tiles=1),
])
def test_tilemap_follows_the_persistent_schedule(plan):
    Ho = Wo = {4: 20, 16: 80}.get(plan["bh"], 40)
    n_img = 63
    tw, th = Wo // plan["bw"], Ho // plan["bh"]
    plan = dict(plan, m_tiles=tw * th * -(-n_img // plan["bimg"]))
    sched = _schedule(plan, Ho, Wo)
    tm = kr.TileMap(plan, Ho, Wo)
    for (m, cb), (cta, it) in list(sched.items())[::7]:
        img = (m // (tw * th)) * plan["bimg"]
        i, j = ((m // tw) % th) * plan["bh"], (m % tw) * plan["bw"]
        d = tm.locate(img, i, j, cb * plan["bn"])
        assert d["m_tile"] == m and (d["cta"], d["iteration"]) == (cta, it), (plan["kernel"], m, cb)


def _attn32(qkv, keep=None):
    """Emulation of fp_attn_tc.cu's arithmetic for one group: S fp32, p = exp2(s c - m c), l fp32, P fp16, O fp32."""
    B = qkv.shape[0] // 400
    x = qkv.float().reshape(B, 400, 3, 4, 128).permute(2, 0, 3, 1, 4)
    q, k, v = x[0], x[1], x[2]
    c = kr.ATTN_SCALE * kr.LOG2E
    S = q @ k.transpose(-1, -2)
    if keep is not None:
        S = S.masked_fill(~keep, -math.inf)
    m = S.amax(-1, keepdim=True)
    p = torch.exp2(S * c - m * c)
    l = p.sum(-1, keepdim=True)
    o = (p.half().float() @ v) / l
    return o.half().permute(0, 2, 1, 3).reshape(B * 400, 512)


@pytest.mark.parametrize("kind", ["std", "sharp", "flat"])
def test_attention_accepts_rounding_and_kernel_arithmetic(kind):
    qkv = kr.attention_inputs(kind, 1, 1, seed=3, device="cpu")
    ref, _ = kr.attention_reference(qkv, 1, 0, 1)
    r = kr.check_attention(ref[0].half(), qkv, 1, what=kind)
    assert r.ok and r.max_ulps < 0.501, kr.attention_report(r)
    r = kr.check_attention(_attn32(qkv), qkv, 1, what=kind)
    assert r.ok, kr.attention_report(r)
    if kind == "flat":  # identical keys: the output is the mean of v
        v = qkv.double().reshape(400, 3, 4, 128)[:, 2].mean(0).reshape(512)
        assert torch.allclose(ref[0], v.expand(400, 512), atol=1e-12)


def test_attention_two_groups_layout():
    qkv = kr.attention_inputs("std", 2, 2, seed=4, device="cpu")
    halves = qkv.reshape(800, 2, 1536)
    got = torch.stack([_attn32(halves[:, gi].contiguous()) for gi in range(2)])
    r = kr.check_attention(got, qkv, 2, what="grouped")
    assert r.ok, kr.attention_report(r)
    swapped = got.flip(0)
    assert not kr.check_attention(swapped, qkv, 2, what="groups swapped").ok


def test_attention_rejects_one_dropped_key_block():
    qkv = kr.attention_inputs("std", 1, 1, seed=5, device="cpu")
    keep = torch.ones(4, 400, 400, dtype=torch.bool)
    keep[1, 256:384, 80:160] = False  # head 1, query tile 2 loses the keys of one 80-key V chunk
    got = _attn32(qkv)
    got[256:384, 128:256] = _attn32(qkv, keep[None])[256:384, 128:256]
    r = kr.check_attention(got, qkv, 1, what="dropped key block")
    assert not r.ok
    assert {k[2:] for k in r.tiles} == {(2, 1)}, kr.attention_report(r)
    assert "query tile 2 head 1" in kr.attention_report(r)
