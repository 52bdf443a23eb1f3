"""The register path's GEMM kernels and the attention kernel against float64, at the batch sizes production runs.

Every distinct layer of run_encoder / run_refine_heads / run_score_feats (csrc/fp_api.cu) runs with its production
flags at N = 1, 31, 32, 63, 126 and 252 hypotheses (encodeA side: M = Np + N images, Np = N rounded up to a multiple
of 4), so that the persistent CTAs walk many tiles (both TMEM accumulators, the smem rings wrapping from tile to tile,
the residual prefetch) and the batch edges leave partial tiles.  Each output element is held to the per-element bar of
tests/kernel_ref.py; fp_op_gemm_last_plan says which kernel ran, so the test also pins the dispatch: the set of
kernels the table reaches, that each wide kernel ran with at least three tiles per CTA, and the plan of every layer at
N = 252.  Determinism: every case is launched twice (bitwise equal), and each layer's outputs at N = 248 and N = 252
(same kernels, different tile counts and schedules) are bitwise equal on every image the two share.

Attention runs through fp_op_attention_grouped in both production layouts (scorer: one group, refiner: two heads in
one launch) for B = 1, 31, 252 on three input distributions.
"""
import pytest
import torch

import kernel_ref as kr

pytestmark = pytest.mark.gpu

NS = (1, 31, 32, 63, 126, 252)
N_INV = 248  # compared bitwise with N = 252

# the kernels the table must reach (fp_gemm.cu gemm_layer_launch with the default switches on a 148-SM B200)
KERNELS = {"stem", "swap", "swap_patch", "tile<128,2,2>", "tile<128,2,4>", "tile<256,2,2,patch>",
           "tile<256,2,4,patch>", "tile<256,2,2>", "tile<256,2,4>", "tile<256,1,8>", "tile<256,1,4>"}
NARROW = {"tile<128,2,2>", "tile<128,2,4>"}  # one tracked pose (N = 1): a few tiles by design

# name: (kind, side, H in, Cin, Cout, res, post_add, relu, out_split, plan at N = 252)
#   side A: encodeA, M = Np + N images; AB: N images; rows: LINEAR over N * 400 token rows
LAYERS = {
    "stem_160_6_64": ("stem", "A", 160, 6, 64, False, False, True, False, "stem"),
    "conv_s2_80_64_128": ("s2", "A", 80, 64, 128, False, False, True, False, "swap"),
    "conv_40_128": ("s1", "A", 40, 128, 128, False, False, True, False, "swap_patch"),
    "conv_40_128_res": ("s1", "A", 40, 128, 128, True, False, True, False, "swap_patch"),
    "conv_40_128_res_concat": ("s1", "A", 40, 128, 128, True, False, True, True, "swap_patch"),
    "conv_40_256": ("s1", "AB", 40, 256, 256, False, False, True, False, "tile<256,2,2,patch>"),
    "conv_40_256_res": ("s1", "AB", 40, 256, 256, True, False, True, False, "tile<256,2,4,patch>"),
    "conv_s2_40_256_512": ("s2", "AB", 40, 256, 512, False, False, True, False, "tile<256,2,2>"),
    "conv_20_512": ("s1", "AB", 20, 512, 512, False, False, True, False, "tile<256,2,2>"),
    "conv_20_512_res": ("s1", "AB", 20, 512, 512, True, False, True, False, "tile<256,2,4>"),
    "conv_20_512_res_pe": ("s1", "AB", 20, 512, 512, True, True, True, False, "tile<256,2,4>"),
    "linear_512_3072": ("linear", "rows", 1, 512, 3072, False, False, False, False, "tile<256,1,8>"),
    "linear_512_1536": ("linear", "rows", 1, 512, 1536, False, False, False, False, "tile<256,1,8>"),
    "linear_512_512_relu": ("linear", "rows", 1, 512, 512, False, False, True, False, "tile<256,1,8>"),
    "linear_512_512_res": ("linear", "rows", 1, 512, 512, True, False, False, False, "tile<256,1,4>"),
}


def _np(n):
    return (n + 3) & ~3


def _count(side, n):
    return {"A": _np(n) + n, "AB": n, "rows": 400 * n}[side]


class Layer:
    """Seeded operands of one layer for the largest batch; a batch of n uses the first images / rows."""

    def __init__(self, name, seed):
        from foundationpose_b200 import _lib, ops, packing

        self.ops, self.lib = ops, _lib
        self.name = name
        (self.kind, self.side, self.H, self.ci, self.co, has_res, has_pe, self.relu, self.split,
         self.plan_252) = LAYERS[name]
        nmax = _count(self.side, max(NS))
        g = torch.Generator(device="cuda").manual_seed(seed)
        rnd = lambda *s, scale=1.0: torch.randn(*s, generator=g, device="cuda") * scale  # noqa: E731
        self.Ho = {"s1": self.H, "s2": self.H // 2, "stem": self.H // 2, "linear": 1}[self.kind]
        if self.kind == "linear":
            self.x = rnd(nmax, self.ci).half()
            self.w = rnd(self.co, self.ci, scale=self.ci ** -0.5).half()
            self.wp = packing.pack_linear(self.w)
            self.lk = _lib.LAYER_LINEAR
        elif self.kind == "stem":
            self.x = rnd(nmax, self.H, self.H, self.ci).half()
            self.w = rnd(self.co, self.ci, 7, 7, scale=(49 * self.ci) ** -0.5).half()
            self.wp = packing.pack_conv7(self.w.cpu()).cuda()
            self.xin = packing.pad_image_c8(self.x.permute(0, 3, 1, 2))
            self.lk = _lib.LAYER_CONV7_S2
        else:
            self.x = rnd(nmax, self.H, self.H, self.ci).half()
            self.w = rnd(self.co, self.ci, 3, 3, scale=(9 * self.ci) ** -0.5).half()
            self.wp = packing.pack_conv3(self.w.cpu()).cuda()
            self.lk = _lib.LAYER_CONV3_S1 if self.kind == "s1" else _lib.LAYER_CONV3_S2
        self.b = rnd(self.co)
        rshape = (nmax, self.co) if self.kind == "linear" else (nmax, self.Ho, self.Ho, self.co)
        self.res = rnd(*rshape).half() if has_res else None
        self.pe = rnd(self.Ho * self.Ho, self.co) if has_pe else None

    def shape(self, n):
        if self.kind == "linear":
            return f"M={400 * n} K={self.ci} -> {self.co}"
        return f"{_count(self.side, n)} x {self.H}x{self.H}x{self.ci} -> {self.Ho}x{self.Ho}x{self.co}"

    def launch(self, n):
        """One launch at batch n -> (logical output [m, Ho, Wo, Co] with the images the layer stored, their ranges,
        plan).  Outputs start as NaN, so an element the kernel never wrote fails the comparison."""
        cnt = _count(self.side, n)
        nan = float("nan")
        if self.kind == "linear":
            out = torch.full((1, 1, cnt, self.co), nan, dtype=torch.float16, device="cuda")
            self.ops.gemm_layer(self.lk, self.x[:cnt], self.wp, self.b, n_img=1, Hin=1, Win=cnt, Cin=self.ci,
                                Cout=self.co, out=out, out_ld=self.co, res=None if self.res is None else self.res[:cnt],
                                res_ld=self.co, relu=self.relu)
            return out, [(0, cnt)], self.ops.gemm_last_plan()
        xin = self.xin[:cnt] if self.kind == "stem" else self.x[:cnt]
        kw = dict(n_img=cnt, Hin=self.H, Win=self.H, Cin=8 if self.kind == "stem" else self.ci, Cout=self.co,
                  res=None if self.res is None else self.res[:cnt], res_ld=self.co, post_add=self.pe, relu=self.relu)
        if not self.split:
            out = torch.full((cnt, self.Ho, self.Ho, self.co), nan, dtype=torch.float16, device="cuda")
            self.ops.gemm_layer(self.lk, xin, self.wp, self.b, out=out, out_ld=self.co, **kw)
            return out, [(0, cnt)], self.ops.gemm_last_plan()
        # the last encodeA layer: images [0, Np) -> channels [0, 128) of the concat buffer, [Np, Np + N) -> [128, 256);
        # the padding images [N, Np) fall outside the buffer.  One guard image behind it must stay untouched.
        Np = _np(n)
        buf = torch.full((n + 1, self.Ho, self.Ho, 2 * self.co), nan, dtype=torch.float16, device="cuda")
        self.ops.gemm_layer(self.lk, xin, self.wp, self.b, out=buf, out_ld=2 * self.co, out_split=Np, **kw)
        plan = self.ops.gemm_last_plan()
        assert torch.isnan(buf[n].float()).all(), f"{self.name} N={n}: the concat store wrote past its {n} images"
        got = torch.full((cnt, self.Ho, self.Ho, self.co), nan, dtype=torch.float16, device="cuda")
        got[:n] = buf[:n, ..., :self.co]
        got[Np:] = buf[:n, ..., self.co:]
        return got, [(0, n), (Np, cnt)], plan

    def reference(self, a, b):
        res = None if self.res is None else self.res[a:b]
        if self.kind == "linear":
            return kr.linear_reference(self.x[a:b], self.w, self.b, res=res, relu=self.relu)
        if self.kind == "stem":  # 7 filter rows x 4 tap pairs = 28 MMAs of K = 16
            return kr.conv_reference(self.x[a:b], self.w, self.b, stride=2, relu=self.relu, steps=28)
        return kr.conv_reference(self.x[a:b], self.w, self.b, stride=2 if self.kind == "s2" else 1, res=res,
                                 post_add=self.pe, relu=self.relu)


class Table:
    """Runs each layer's cases on first request and keeps their records (plans, error statistics, failures)."""

    def __init__(self):
        self.done = {}

    def layer(self, name):
        if name not in self.done:
            self.done[name] = self._run(name)
        return self.done[name]

    def _run(self, name):
        L = Layer(name, seed=1000 + list(LAYERS).index(name))
        recs, fails = [], []
        cdim = 2 if L.kind == "linear" else 0
        keep = None
        for n in NS:
            got, ranges, plan = L.launch(n)
            again, _, plan2 = L.launch(n)
            torch.cuda.synchronize()
            what = f"{name} N={n} ({L.shape(n)}) on {kr.plan_name(plan)}"
            tm = kr.TileMap(plan, L.Ho, _count(L.side, n) if L.kind == "linear" else L.Ho)
            r = kr.check_chunked(got, L.reference, what=what, plan=plan, ranges=ranges, chunk_dim=cdim)
            if not r.ok:
                fails.append(r.report(tm))
            twice = kr.bitwise_diff(got, again, what=what + ": second launch", plan=plan)
            if not twice.ok or plan2 != plan:
                fails.append(twice.report(tm) + f"\n  plans {plan} / {plan2}")
            recs.append(dict(layer=name, n=n, shape=L.shape(n), plan=plan, name=kr.plan_name(plan), result=r))
            if n == max(NS):
                keep = (got, plan, tm)
            del got, again
        # N = 248 against N = 252: same images in, same bits out, whatever the tile counts and schedules
        got, ranges, plan = L.launch(N_INV)
        ref_out, ref_plan, tm = keep
        for lo, hi in ranges:  # every image / row the smaller launch stored is also in the larger one
            inv = kr.bitwise_diff(got.narrow(cdim, lo, hi - lo), ref_out.narrow(cdim, lo, hi - lo), plan=ref_plan,
                                  what=f"{name}: N={N_INV} ({kr.plan_name(plan)}) vs N={max(NS)}, [{lo}, {hi})")
            if not inv.ok:
                fails.append(inv.report(tm))
        if kr.plan_name(plan) != kr.plan_name(ref_plan):
            fails.append(f"{name}: N={N_INV} ran {kr.plan_name(plan)}, N={max(NS)} {kr.plan_name(ref_plan)}")
        return recs, fails


@pytest.fixture(scope="module")
def table():
    torch.cuda.set_device(0)
    return Table()


@pytest.mark.parametrize("layer", list(LAYERS))
def test_layer_matches_float64_at_production_batches(table, layer):
    recs, fails = table.layer(layer)
    assert not fails, "\n".join(fails)


def test_plans_at_252(table):
    got = {name: [r["name"] for r in table.layer(name)[0] if r["n"] == 252][0] for name in LAYERS}
    want = {name: spec[-1] for name, spec in LAYERS.items()}
    assert got == want


def test_dispatch_coverage_and_summary(table, capsys):
    recs = [r for name in LAYERS for r in table.layer(name)[0]]
    by_kernel = {}
    for r in recs:
        by_kernel.setdefault(r["name"], []).append(r)
    lines = ["", f"{'kernel':22s} {'tiles/CTA':>14s} {'worst ulps':>10s} {'worst/bar':>9s}  shapes (N)"]
    for k in sorted(by_kernel):
        rs = by_kernel[k]
        tpc = [kr.tiles_per_cta(r["plan"]) for r in rs]
        shapes = "; ".join(sorted({f"{r['layer']}: {r['shape']} (N={r['n']})" for r in rs}))
        lines.append(f"{k:22s} {min(tpc):6.2f}-{max(tpc):7.2f} {max(r['result'].max_ulps for r in rs):10.3g} "
                     f"{max(r['result'].max_ratio for r in rs):9.3g}  {shapes}")
    with capsys.disabled():
        print("\n".join(lines))
    assert set(by_kernel) == KERNELS
    for k in KERNELS - NARROW:
        assert any(r["plan"]["work_tiles"] >= 3 * r["plan"]["grid"] for r in by_kernel[k]), \
            f"{k} never ran with at least three tiles per CTA"


@pytest.mark.parametrize("kind", ["std", "sharp", "flat"])
@pytest.mark.parametrize("n_groups", [1, 2])
@pytest.mark.parametrize("B", [1, 31, 252])
def test_attention_grouped_matches_float64(B, n_groups, kind, capsys):
    from foundationpose_b200 import ops

    torch.cuda.set_device(0)
    seed = 7 + 100 * B + 10 * n_groups + ["std", "sharp", "flat"].index(kind)
    qkv = kr.attention_inputs(kind, B, n_groups, seed=seed, device="cuda")
    out = ops.attention_grouped(qkv, n_groups)
    again = ops.attention_grouped(qkv, n_groups)
    torch.cuda.synchronize()
    assert torch.equal(out.view(torch.int16), again.view(torch.int16)), "two launches differ"
    what = f"attention B={B} n_groups={n_groups} {kind} ({B * 4 * n_groups / 148:.2f} items per CTA)"
    r = kr.check_attention(out, qkv, n_groups, what=what)
    with capsys.disabled():
        print(f"\n{what}: worst {r.max_ulps:.3g} fp16 ulps, {r.max_ratio:.3g} x bar")
    assert r.ok, kr.attention_report(r)
    if kind == "flat":  # identical keys: the output is the mean of v, to within the same bar
        nb = min(B, 8)
        _, bar = kr.attention_reference(qkv, n_groups, 0, nb)
        v = qkv[:nb * 400].double().reshape(nb, 400, n_groups, 3, 512)[:, :, :, 2]
        mean = v.mean(1, keepdim=True).expand(nb, 400, n_groups, 512).permute(2, 0, 1, 3).reshape(n_groups, nb * 400, 512)
        got = out.reshape(n_groups, B * 400, 512)[:, :nb * 400].double()
        assert ((got - mean).abs() <= bar).all()
