"""The tcgen05 GEMM (csrc/gemm_umma.cu), its split-K fold, the activation backward and the operand casts (csrc/ew.cu), and
``linear()`` forward / backward, checked on inputs for which the kernels' results are EXACT.

Operands are integers in {-2..2} ({-1, 0, 1} once K >= 16384), so every partial sum stays below 2^16 and the fp32
accumulation is exact in any order and at any split; the epilogue operands are short dyadic numbers (alpha in
{1, 0.5, -2}, bias and residual multiples of 1/8 in [-4, 4], column scale in {0.5, 1, 1.5, 2}, mask in {0, 2}).  With no
activation or ReLU every fp32 operation of the epilogue is then exact: an fp32 result must EQUAL the fp64 reference, a bf16
one the reference rounded to nearest even.  A misplaced tile, a dropped k-block or a wrong batch offset cannot hide in a
tolerance.  GELU and sigmoid leave only the activation's own error, bounded next to each check.

Every GEMM goes through the C entry with row pitches wider than N, extra rows and a sentinel in every byte it must not
write.  Run with ``-m gpu`` on a B200."""
import math
import zlib

import pytest
import torch

from cor_b200 import _lib as L
from cor_b200 import linear as lin
from cor_b200 import ops
from cor_b200._lib import ACT_GELU, ACT_NONE, ACT_RELU, ACT_SIGMOID, CorError

pytestmark = pytest.mark.gpu

F64 = torch.float64
SENT32, SENT16 = 0x7FA5A5A5, 0x7FA5          # NaN bit patterns: what no store may leave behind outside [batch*M, N]
WORST = {}                                   # worst |error| / bound per bounded check (reported at the end of the module)

# Bounds on the fp32 evaluation of the activations, for |pre-activation| as large as these tests make it:
#  - erff form (fp32 output, split-K fold): libdevice erff is within 2 ulp; with the roundings of 0.5 v (1 + erf(v/sqrt 2)),
#    |error| <= 2^-21 |v|.
#  - gelu_fast (bf16 output, common.cuh): Abramowitz-Stegun 7.1.26 is within 1.5e-7 of Phi; the approximate reciprocal and
#    exponential and the fp32 roundings add at most 2^-21, so |error| <= (1.5e-7 + 2^-21) |v|.  Its derivative
#    gelu_grad_fast likewise stays within 1.5e-7 + 2^-21 of Phi(x) + x phi(x) for |x| <= 4.
#  - sigmoid 1 / (1 + __expf(-v)): __expf is within 2 + 1.17 |v| ulp; through the division that is at most
#    s (1 - s) (2 + 1.17 |v|) 2^-24 + 2^-24 <= 2^-21 absolute.
GELU_ERF, GELU_FAST, SIGMOID_ABS = 2.0 ** -21, 1.5e-7 + 2.0 ** -21, 2.0 ** -21


def dev():
    return torch.device("cuda:0")


@pytest.fixture(scope="module", autouse=True)
def _report_worst(request):
    """Writes the worst |error| / bound of every bounded check to the terminal once the module's tests have run (through
    the terminal reporter, so that it shows without ``-s``)."""
    yield
    tr = request.config.pluginmanager.get_plugin("terminalreporter")
    cap = request.config.pluginmanager.get_plugin("capturemanager")
    if tr is None or cap is None or not WORST:
        return
    with cap.global_and_fixture_disabled():
        tr.write("\n")
        for k, v in sorted(WORST.items()):
            tr.write_line(f"worst |error| / bound  {k}: {v:.3g}")


def _gen(*key):
    return torch.Generator().manual_seed(zlib.crc32(repr(key).encode()))


def ints(shape, lim, g):
    return torch.randint(-lim, lim + 1, shape, generator=g).to(F64)


def pick(values, shape, g):
    return torch.tensor(values, dtype=F64)[torch.randint(len(values), shape, generator=g)]


def eighths(shape, g, lim=4):
    return torch.randint(-8 * lim, 8 * lim + 1, shape, generator=g).to(F64) / 8


def bf16r(x):
    """fp64 -> the bf16 value round-to-nearest-even makes of it (via fp32, exact for these inputs), as fp64."""
    return x.float().bfloat16().to(F64)


def half_ulp_bf16(x):
    _, e = torch.frexp(x.abs().float())
    return torch.ldexp(torch.ones_like(x), (e - 9).to(torch.int64).to(x.device))


def within(got, ref, tol, what):
    err = (got.to(F64) - ref).abs()
    assert torch.isfinite(got).all(), f"{what}: non-finite result"
    ratio = float((err / tol).max()) if err.numel() else 0.0
    WORST[what] = max(WORST.get(what, 0.0), ratio)
    i = int((err - tol).argmax())
    assert ratio <= 1.0, f"{what}: |error| {float(err.flatten()[i]):.3g} > bound {float(tol.flatten()[i]):.3g} at {i}"


def act64(v, act):
    if act == ACT_RELU:
        return v.clamp_min(0)
    if act == ACT_GELU:
        return 0.5 * v * (1 + torch.erf(v / math.sqrt(2)))
    if act == ACT_SIGMOID:
        return torch.sigmoid(v)
    return v


# ---------------------------------------------------------------------------------------------------------------------
# GEMM through the C entry
# ---------------------------------------------------------------------------------------------------------------------
def _sentinel(n, dtype):
    if dtype == torch.float32:
        return torch.full((n,), SENT32, dtype=torch.int32, device=dev()).view(torch.float32)
    return torch.full((n,), SENT16, dtype=torch.int16, device=dev()).view(torch.bfloat16)


def _untouched(buf, off, rows_total, ld, rows, N):
    """Every element of ``buf`` outside the [rows, N] window at ``off`` with pitch ``ld`` still holds the sentinel."""
    it = torch.int32 if buf.dtype == torch.float32 else torch.int16
    s = SENT32 if buf.dtype == torch.float32 else SENT16
    bits = buf.view(it)
    grid = bits[off:off + rows_total * ld].view(rows_total, ld)
    return bool((bits[:off] == s).all() and (bits[off + rows_total * ld:] == s).all() and (grid[:rows, N:] == s).all()
                and (grid[rows:] == s).all())


def _placed(vals, off, dtype, ld=None, fill=float("nan")):
    """``vals`` [rows, N] fp64 on the device, stored ``off`` elements into a fresh buffer with row pitch ``ld``; the gap
    columns hold NaN so that a read of them poisons the result."""
    rows, N = vals.shape
    ld = ld or N
    buf = torch.full((off + rows * ld,), fill, dtype=dtype, device=dev())
    buf[off:].view(rows, ld)[:, :N] = vals.to(dtype)
    return buf[off:]


class Epi(dict):
    """One epilogue configuration: alpha, bias, pre, act, emul, cs (column scale), res (None / 'f32' / 'bf16'),
    out ('f32' / 'bf16'), off ('all': start C, pre, residual, emul, bias and colscale one element into their buffers; 'bias',
    'cs', 'res', 'pre', 'emul': only that operand, with C aligned -- the one offset operand alone must send the chunk to
    the per-element path)."""
    def __getattr__(self, k):
        return self.get(k, dict(alpha=1.0, act=ACT_NONE, out="f32").get(k))

    def __str__(self):
        return ",".join(f"{k}={v}" for k, v in sorted(self.items())) or "plain"


_ALL = dict(alpha=-2.0, bias=True, pre=True, emul=True, cs=True)
VARIANTS = ([Epi()] + [Epi(alpha=a) for a in (0.5, -2.0)] + [Epi(bias=True), Epi(pre=True), Epi(emul=True), Epi(cs=True),
            Epi(res="f32"), Epi(res="bf16"), Epi(out="bf16")]
            + [Epi(act=a, out=o) for a in (ACT_RELU, ACT_GELU, ACT_SIGMOID) for o in ("f32", "bf16")]
            + [Epi(_ALL, act=a, res=r, out=o) for a in (ACT_NONE, ACT_RELU, ACT_GELU, ACT_SIGMOID) for r, o in (("f32", "f32"), ("bf16", "bf16"))]
            + [Epi(_ALL, act=a, res=r, out=o, off="all") for a, r, o in ((ACT_RELU, "f32", "f32"), (ACT_RELU, "bf16", "bf16"),
                                                                          (ACT_GELU, "bf16", "bf16"), (ACT_SIGMOID, "f32", "f32"))]
            + [Epi(_ALL, act=ACT_RELU, res="f32", out="f32", off=o) for o in ("bias", "cs", "res", "pre", "emul")]
            + [Epi(_ALL, act=ACT_RELU, res="bf16", out="bf16", off=o) for o in ("bias", "cs", "res")]
            + [Epi(_ALL, act=ACT_GELU, res="bf16", out="bf16", off=o) for o in ("bias", "cs")])


def _operands(batch, M, N, K, key):
    g = _gen("ops", *key)
    lim = 1 if K >= 16384 else 2
    return ints((batch, M, K), lim, g), ints((batch, N, K), lim, g), lim


def _store(X, mn, shared=False, pad_rows=None, g=None):
    """X [batch, R, K] fp64 -> (2-D bf16 operand as cor_gemm_bf16 reads it, x_batch_rows).  K-major: [rows][K], rows
    optionally padded per batch entry (pad rows hold non-zero junk); MN-major: [K][R] per entry; shared: entry 0 only."""
    batch, R, K = X.shape
    if shared:
        X = X[:1]
    if mn:
        st = X.transpose(1, 2).reshape(-1, R)
        br = 0 if shared else K
    else:
        Rp = pad_rows or R
        st = torch.full((X.shape[0], Rp, K), 0.0, dtype=F64)
        st[:, R:] = ints((X.shape[0], Rp - R, K), 2, g) if Rp > R else 0
        st[:, :R] = X
        st = st.reshape(-1, K)
        br = 0 if shared else Rp
    return st.to(torch.bfloat16).contiguous().to(dev()), br     # (a batch of one transposes into a strided view)


def run_gemm(A, B, ep, *, a_mn=0, b_mn=0, shared_a=False, pad_a=None, ksplit=0, key=()):
    """One cor_gemm_bf16 call of epilogue ``ep`` on A [batch, M, K], B [batch, N, K] (fp64, CPU); checks the result against
    the fp64 reference and that nothing outside [batch*M, N] of C / pre changed.  Returns (C, pre) views for comparisons."""
    batch, M, K = A.shape
    N = B.shape[1]
    rows = batch * M
    g = _gen("epi", str(Epi({k: v for k, v in ep.items() if k != "off"})), *key)     # the offset run gets the aligned run's operands
    Ad, Bd = A.to(dev()), B.to(dev())
    acc = (Ad[:1].expand(batch, M, K) if shared_a else Ad) @ Bd.transpose(1, 2)
    acc = acc.reshape(rows, N)
    alpha = ep.alpha
    if ep.act == ACT_SIGMOID:          # keep |v| <= 8, the range the sigmoid bound is stated for; a power of two stays exact
        alpha = math.copysign(2.0 ** -math.ceil(math.log2(max(1.0, float(acc.abs().max()) / 4))), ep.alpha)
    bias = eighths((N,), g).to(dev()) if ep.bias else None
    cs = pick([0.5, 1.0, 1.5, 2.0], (N,), g).to(dev()) if ep.cs else None
    emul = pick([0.0, 2.0], (rows, N), g).to(dev()) if ep.emul else None
    res = eighths((rows, N), g).to(dev()) if ep.res else None
    if ep.act == ACT_SIGMOID and bias is not None:
        bias = bias / 2
    # the fp64 reference, in the epilogue's order
    v = acc * alpha + (bias if bias is not None else 0)
    if ep.act == ACT_SIGMOID:
        assert float(v.abs().max()) <= 8
    z = act64(v, ep.act)
    scale = (emul if emul is not None else 1) * (cs if cs is not None else 1)
    y = z * scale + (res if res is not None else 0)

    shift = lambda name: 1 if ep.off in ("all", name) else 0
    off = shift("C")
    a2, abr = _store(A, a_mn, shared_a, pad_a, g)
    b2, bbr = _store(B, b_mn)
    cdt = torch.bfloat16 if ep.out == "bf16" else torch.float32
    ldc = N + (8 if N % 8 == 0 else 3)
    ldr = N + (16 if N % 8 == 0 else 5)
    extra = 5
    Cbuf = _sentinel(off + (rows + extra) * ldc + 7, cdt)
    offp = shift("pre")
    Pbuf = _sentinel(offp + (rows + extra) * ldc + 7, torch.bfloat16) if ep.pre else None
    rdt = torch.bfloat16 if ep.res == "bf16" else torch.float32
    rt = _placed(res, shift("res"), rdt, ldr) if res is not None else None
    bt = _placed(bias[None], shift("bias"), torch.float32)[0:N] if bias is not None else None
    ct = _placed(cs[None], shift("cs"), torch.float32)[0:N] if cs is not None else None
    et = _placed(emul, shift("emul"), torch.float32) if emul is not None else None
    lib = L.load()
    work = ops._work(lib.cor_gemm_bf16_work_bytes(M, N, K, batch, ksplit), dev())
    split = lib.cor_gemm_bf16_work_bytes(M, N, K, batch, ksplit) > 16
    ops._call("cor_gemm_bf16", dev(), L.ptr(a2), a_mn, ops._ll(a2.shape[0]), ops._ll(abr), L.ptr(b2), b_mn, ops._ll(b2.shape[0]), ops._ll(bbr),
              M, N, K, batch, ops._f(alpha), L.ptr(bt), ep.act, L.ptr(et), L.ptr(ct), L.ptr(rt), L.dtype_code(rt) if rt is not None else L.F32,
              ops._ll(ldr), L.ptr(Cbuf[off:]), L.dtype_code(Cbuf), ops._ll(ldc), L.ptr(Pbuf[offp:] if Pbuf is not None else None), ksplit, L.ptr(work))
    torch.cuda.synchronize()
    what = f"{'split' if split else 'one-pass'} {ep}"
    assert _untouched(Cbuf, off, rows + extra, ldc, rows, N), f"{what}: C written outside [batch*M, N]"
    C = Cbuf[off:off + (rows + extra) * ldc].view(rows + extra, ldc)[:rows, :N]
    pre = None
    if Pbuf is not None:
        assert _untouched(Pbuf, offp, rows + extra, ldc, rows, N), f"{what}: pre written outside [batch*M, N]"
        pre = Pbuf[offp:offp + (rows + extra) * ldc].view(rows + extra, ldc)[:rows, :N]
        assert torch.equal(pre.to(F64), bf16r(v)), f"{what}: pre-activation"
    if ep.act in (ACT_NONE, ACT_RELU):
        want = y if cdt == torch.float32 else bf16r(y)
        bad = (C.to(F64) != want)
        assert not bad.any(), f"{what}: {int(bad.sum())} of {bad.numel()} differ, first at {tuple(bad.nonzero()[0].tolist())}"
    else:
        a_err = (GELU_FAST if cdt == torch.bfloat16 and not split else GELU_ERF) * v.abs() if ep.act == ACT_GELU else SIGMOID_ABS
        tol = a_err * scale.abs() if torch.is_tensor(scale) else a_err * torch.ones_like(v)
        tol = tol + 2.0 ** -23 * ((z * scale).abs() + y.abs()) + 1e-30
        if cdt == torch.bfloat16:
            tol = tol + half_ulp_bf16(y.abs() + tol)
        name = {ACT_GELU: "gelu", ACT_SIGMOID: "sigmoid"}[ep.act]
        within(C, y, tol, f"gemm {name} {'fold' if split else 'epilogue'} {ep.out} out")
    return C, pre


def run_variants(A, B, key, variants=VARIANTS, **kw):
    aligned = {}
    for ep in variants:
        C, _ = run_gemm(A, B, ep, key=key, **kw)
        base = Epi({k: v for k, v in ep.items() if k != "off"})
        if ep.off:                                     # the per-element path must give what the aligned run gave, bit for bit
            assert base in variants, base
            assert torch.equal(C.view(torch.int16 if C.dtype == torch.bfloat16 else torch.int32), aligned[str(base)]), f"offset {ep}"
        else:
            aligned[str(ep)] = C.clone().view(torch.int16 if C.dtype == torch.bfloat16 else torch.int32)


def _shapes():
    out = []
    for M in (1, 33, 129, 200):
        for N in (256, 200, 37, 8):
            for K in (8, 64, 72):
                for a_mn in (0, 1):
                    for b_mn in (0, 1):
                        if (a_mn and M % 8) or (b_mn and N % 8):      # TMA: an MN-major operand's rows must span 16 bytes
                            continue
                        out.append((M, N, K, a_mn, b_mn))
    return out


@pytest.mark.parametrize("shape", _shapes(), ids=lambda s: "M{}-N{}-K{}-a{}-b{}".format(*s))
def test_gemm_exact_one_pass(shape):
    """Every epilogue term alone and all together, on the fast store path (N = 256), fast chunks then a ragged last chunk
    (N = 200), the per-element path (N = 37, 8), in all four operand orientations, K below one k-block, one k-block and a
    ragged k-block, M from one row to one row into the second tile."""
    M, N, K, a_mn, b_mn = shape
    A, B, _ = _operands(1, M, N, K, shape)
    run_variants(A, B, shape, a_mn=a_mn, b_mn=b_mn)


@pytest.mark.parametrize("case", [
    (200, 256, 36864, 1, 1, 0), (128, 200, 36864, 1, 1, 0), (33, 37, 36864, 0, 0, 0), (200, 8, 36864, 1, 1, 0),   # automatic
    (33, 37, 512, 0, 0, 3), (129, 200, 512, 0, 1, 7), (200, 256, 512, 1, 1, 3), (1, 8, 512, 0, 1, 7), (200, 200, 512, 1, 0, 7),
    (33, 256, 72, 0, 0, 7), (200, 37, 72, 1, 0, 5),                     # more splits than k-blocks: clamped to 2
    (200, 256, 36864, 1, 1, 1),                                         # 576 k-blocks in one accumulator, no split
], ids=lambda c: "M{}-N{}-K{}-a{}-b{}-ks{}".format(*c))
def test_gemm_exact_split_k(case):
    """Split-K partials and gemm_fold_kernel with every epilogue term, term by term and together; K = 36 864 with both
    operands MN-major is the weight-gradient shape."""
    M, N, K, a_mn, b_mn, ks = case
    A, B, _ = _operands(1, M, N, K, case)
    split = L.load().cor_gemm_bf16_work_bytes(M, N, K, 1, ks) > 16
    assert split == (ks != 1)
    run_variants(A, B, case, a_mn=a_mn, b_mn=b_mn, ksplit=ks)


_FEW = [Epi(), Epi(_ALL, act=ACT_RELU, res="f32"), Epi(_ALL, act=ACT_RELU, res="bf16", out="bf16"), Epi(_ALL, act=ACT_GELU, res="f32", out="bf16")]


@pytest.mark.parametrize("kind", ["shared_a_kmajor_b", "shared_a_mn_b", "padded_a", "per_entry_mn", "per_entry_split"])
def test_gemm_exact_batched(kind):
    """batch = 3: A shared by every entry (a_batch_rows = 0); K-major A padded per entry to Qp = ceil64(M) rows of junk
    beyond M, as the adapter's softmax-map tail stores it; both operands per entry and MN-major; per entry with split-K."""
    M, N, K, kw = {"shared_a_kmajor_b": (33, 200, 72, dict(shared_a=True)), "shared_a_mn_b": (33, 200, 64, dict(shared_a=True, b_mn=1)),
                   "padded_a": (20, 136, 72, dict(pad_a=64)), "per_entry_mn": (200, 256, 64, dict(a_mn=1, b_mn=1)),
                   "per_entry_split": (129, 200, 512, dict(ksplit=3))}[kind]
    A, B, _ = _operands(3, M, N, K, (kind,))
    run_variants(A, B, (kind,), variants=_FEW, **kw)


@pytest.mark.parametrize("Mm,B,Cc,P", [(20, 3, 136, 200), (50, 2, 64, 256), (1, 4, 128, 64)])
def test_gemm_pool_backward_layout_exact(Mm, B, Cc, P):
    """The pooling-backward GEMM exactly as region._pool_bwd_gemm builds it: both operands MN-major, A = the gradient rows
    zero-padded to Kp = ceil64(M) per image, B = the bf16 weights with Rp = ceil16(M + 1) < Kp rows per image, so a k-block
    reads the next image's (non-zero) rows, and the last image's runs past the tensor.  Must equal the per-image product."""
    from cor_b200 import region
    g = _gen("pool", Mm, B)
    Kp, Rp = (Mm + 63) // 64 * 64, (Mm + 1 + 15) // 16 * 16
    assert Rp < Kp or Mm > 47
    gs = ints((B, Mm, Cc), 2, g)
    w = ints((B, Rp, P), 2, g)                  # rows Mm..Rp: the ones row and padding, all non-zero junk here
    w[w == 0] = 1
    a16 = torch.zeros((B, Kp, Cc), dtype=F64)
    a16[:, :Mm] = gs
    a16 = a16.reshape(B * Kp, Cc).to(torch.bfloat16).to(dev())
    w16 = w.to(torch.bfloat16).to(dev())
    for out_dtype in (torch.float32, torch.bfloat16):
        got = region._pool_bwd_gemm(a16, w16, B, Cc, P, Kp, out_dtype)
        ref = (gs.transpose(1, 2) @ w[:, :Mm]).reshape(B * Cc, P).to(dev())
        assert torch.equal(got.to(F64), ref if out_dtype == torch.float32 else bf16r(ref)), out_dtype


def test_gemm_refuses_batched_mn_major_with_ragged_k():
    a = torch.zeros((2 * 72, 64), dtype=torch.bfloat16, device=dev())
    b = torch.zeros((2 * 64, 72), dtype=torch.bfloat16, device=dev())
    with pytest.raises(CorError, match="K % 64"):
        lin.gemm(a, b, 64, 64, 72, a_mn=True, batch=2, a_batch_rows=72, b_batch_rows=64)
    with pytest.raises(CorError, match="K % 64"):
        lin.gemm(b, a, 64, 64, 72, b_mn=True, batch=2, a_batch_rows=64, b_batch_rows=72)


# ---------------------------------------------------------------------------------------------------------------------
# cor_act_bwd
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dy_dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("kernel", ["vec", "scalar", "scalar_offset"])
@pytest.mark.parametrize("M", [1, 63, 64, 65, 36865])
def test_act_bwd_exact(M, kernel, dy_dtype):
    """dz = bf16(dy * emul * colscale * act'), db = column sums of the unrounded dz, dcs = column sums of dy * emul * pre:
    the vec kernel (N = 256), the scalar kernel (N = 37, and N = 256 with dy one element into its buffer), one row to many
    row chunks with a chunk tail.  dy dyadic, sigmoid outputs in {1/4, 1/2, 3/4}: everything but GELU is exact."""
    N = 37 if kernel == "scalar" else 256
    off = 1 if kernel == "scalar_offset" else 0
    g = _gen("actbwd", M, kernel, str(dy_dtype))
    lib = L.load()
    dy = eighths((M, N), g).to(dev())
    dyb = torch.empty(off + M * N, dtype=dy_dtype, device=dev())
    dyb[off:] = dy.flatten().to(dy_dtype)
    dyt = dyb[off:]
    pre = eighths((M, N), g).to(dev())
    pre16 = pre.to(torch.bfloat16)
    e = pick([0.0, 2.0], (M, N), g).to(dev())
    cs = pick([0.5, 1.0, 1.5, 2.0], (N,), g).to(dev())
    y_of = {ACT_RELU: pick([0.0, 0.25, 1.5, 3.0], (M, N), g).to(dev()), ACT_SIGMOID: pick([0.25, 0.5, 0.75], (M, N), g).to(dev())}
    for act in (ACT_NONE, ACT_RELU, ACT_GELU, ACT_SIGMOID):
        for use_e in (False, True):
            for use_cs in (False, True):
                want_dcs = use_cs and act == ACT_NONE
                y = y_of.get(act)
                y32 = y.float() if y is not None else None
                dz = _sentinel(M * N, torch.bfloat16)
                db = torch.full((N,), float("nan"), device=dev())
                dcs = torch.full((N,), float("nan"), device=dev()) if want_dcs else None
                work = ops._work(lib.cor_act_bwd_work_bytes(M, N), dev())
                e32, cs32 = (e.float() if use_e else None), (cs.float() if use_cs else None)
                ops._call("cor_act_bwd", dev(), L.ptr(dyt), L.dtype_code(dyt), L.ptr(y32), L.ptr(pre16 if act == ACT_GELU or want_dcs else None),
                          L.ptr(e32), L.ptr(cs32), act, ops._ll(M), N, L.ptr(dz), L.ptr(db), L.ptr(dcs), L.ptr(work))
                # reference, in the kernel's order
                gr = dy * (e if use_e else 1)
                dcs_ref = (gr * pre16.to(F64)).sum(0) if want_dcs else None
                gr = gr * (cs if use_cs else 1)
                if act == ACT_RELU:
                    gr = gr * (y > 0)
                elif act == ACT_SIGMOID:
                    gr = gr * y * (1 - y)
                what = f"act={act} emul={use_e} cs={use_cs}"
                if act != ACT_GELU:
                    assert torch.equal(dz.view(M, N).to(F64), bf16r(gr)), f"dz {what}"
                    assert torch.equal(db.to(F64), gr.sum(0)), f"db {what}"
                else:
                    x = pre16.to(F64)
                    gg = 0.5 * (1 + torch.erf(x / math.sqrt(2))) + x * torch.exp(-x * x / 2) / math.sqrt(2 * math.pi)
                    t = gr * gg
                    tol = gr.abs() * GELU_FAST + 2.0 ** -24 * t.abs()
                    within(dz.view(M, N).float(), t, tol + half_ulp_bf16(t.abs() + tol) + 1e-30, "act_bwd gelu dz")
                    # sum of M fp32 terms, each within GELU_FAST |g|: the recursive-summation bound on top
                    within(db, t.sum(0), (gr.abs() * GELU_FAST).sum(0) + (M + 64) * 2.0 ** -24 * t.abs().sum(0) + 1e-30, "act_bwd gelu db")
                if want_dcs:
                    assert torch.equal(dcs.to(F64), dcs_ref), f"dcs {what}"


# ---------------------------------------------------------------------------------------------------------------------
# casts
# ---------------------------------------------------------------------------------------------------------------------
_SPECIAL = [1 + 2 ** -8, -(3 + 2 ** -7) * 2 ** 10, 1 + 3 * 2 ** -8, -(1 + 2 ** -8) * 2 ** -20, float("inf"), float("-inf"),
            3.3e38, -3.4028234e38, 2 ** -130, -1e-40, 0.0, -0.0, 65504.0, 1.0]


def _cast_input(rows, c, g):
    x = (torch.randn((rows, c), generator=g) * torch.pow(2.0, torch.randint(-20, 21, (rows, c), generator=g).float())).float()
    sp = torch.tensor(_SPECIAL, dtype=torch.float32)
    pos = torch.randperm(rows * c, generator=g)[:min(rows * c, 4 * len(_SPECIAL))]
    x.view(-1)[pos] = sp.repeat(4)[:pos.numel()]
    return x


@pytest.mark.parametrize("c0,c1,off", [(64, 32, 0), (64, 0, 0), (13, 7, 0), (13, 0, 0), (64, 32, 1), (64, 0, 1)])
def test_cast_cat_bf16_exact(c0, c1, off):
    """cor_cast_cat_bf16 == torch.cat(a, b).bfloat16() bit for bit: the vec kernel (c0, c1 multiples of 4, aligned), the
    scalar kernel (c0 = 13, c1 = 7; and an input that starts one element into its buffer), with and without b; rounding
    ties, +-Inf, overflow to Inf, subnormals and signed zeros included."""
    rows = 301
    g = _gen("cast", c0, c1, off)
    a = _cast_input(rows, c0, g)
    b = _cast_input(rows, c1, g) if c1 else None
    abuf = torch.empty(off + rows * c0, dtype=torch.float32, device=dev())
    abuf[off:] = a.flatten().to(dev())
    ad = abuf[off:].view(rows, c0)
    got = lin.cast_bf16(ad, b.to(dev()) if b is not None else None)
    want = (torch.cat((a, b), 1) if b is not None else a).bfloat16().to(dev())
    assert torch.equal(got.view(torch.int16), want.view(torch.int16))


@pytest.mark.parametrize("batch,rows,rows_padded,cols", [(3, 20, 64, 136), (2, 64, 64, 8), (1, 1, 128, 4)])
def test_cast_pad_rows_bf16_exact(batch, rows, rows_padded, cols):
    """Rows round to nearest even exactly; the padding rows are +0 even where the buffer held something else."""
    g = _gen("pad", batch, rows)
    src = _cast_input(batch * rows, cols, g)
    out = _sentinel(batch * rows_padded * cols, torch.bfloat16)
    ops._call("cor_cast_pad_rows_bf16", dev(), L.ptr(src.to(dev())), batch, rows, rows_padded, cols, L.ptr(out))
    got = out.view(torch.int16).view(batch, rows_padded, cols)
    assert torch.equal(got[:, :rows], src.bfloat16().view(torch.int16).view(batch, rows, cols).to(dev()))
    assert bool((got[:, rows:] == 0).all())


# ---------------------------------------------------------------------------------------------------------------------
# linear() end to end
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N", [256, 200])
def test_gemm_and_linear_with_offset_bias_and_colscale_views(N):
    """A bias or column scale sliced out of a larger fp32 buffer at an odd float offset, while gemm() / linear() allocate C
    and pre themselves (aligned): the per-element path must give exactly the aligned result, on shapes whose chunks would
    otherwise all (N = 256) or mostly (N = 200) take the fast path."""
    g = _gen("offset_views", N)
    rows, K = 200, 64
    x = ints((rows, K), 2, g).float().to(dev())
    w = ints((N, K), 2, g).float().to(dev())
    b, cs, r = eighths((N,), g).float().to(dev()), pick([0.5, 1.0, 1.5, 2.0], (N,), g).float().to(dev()), eighths((rows, N), g).float().to(dev())

    def shifted(t):
        buf = torch.full((t.numel() + 1,), float("nan"), device=dev())
        buf[1:] = t
        return buf[1:]

    ref = ((x.double() @ w.double().t() + b.double()) * cs.double() + r.double()).float()
    for bv, cv in ((shifted(b), cs), (b, shifted(cs)), (shifted(b), shifted(cs))):
        assert torch.equal(lin.linear(x, w, bv, None, None, None, cv, r), ref)
    x16, w16 = x.bfloat16(), w.bfloat16()
    want, want_pre = lin.gemm(x16, w16, rows, N, K, bias=b, act=ACT_GELU, colscale=cs, residual=r, out_dtype=torch.bfloat16, want_pre=True)
    for bv, cv in ((shifted(b), cs), (b, shifted(cs))):
        got, got_pre = lin.gemm(x16, w16, rows, N, K, bias=bv, act=ACT_GELU, colscale=cv, residual=r, out_dtype=torch.bfloat16, want_pre=True)
        assert torch.equal(got.view(torch.int16), want.view(torch.int16)) and torch.equal(got_pre.view(torch.int16), want_pre.view(torch.int16))


@pytest.mark.parametrize("cfg", [
    dict(res=True), dict(cs=True, res=True, x_bf16=True), dict(cs=True, res=True, out_bf16=True),
    dict(act="relu", out_bf16=True), dict(act="relu", mask=True, x2=True), dict(x_bf16=True, bias=False), dict(act="relu", mask=True),
], ids=lambda c: "-".join(sorted(c)))
def test_linear_forward_backward_exact(cfg):
    """linear() forward and every gradient (x, x2, weight, bias, column scale, residual) against an fp64 reference that
    rounds the saved pre-activation and dZ to bf16 where the kernels do: no activation with a residual, the ConvNeXt form
    (column scale with its gradient, plus residual), bf16 output, concatenated x2, bf16 x, ReLU with a dropout mask."""
    g = _gen("linear", str(sorted(cfg.items())))
    rows, cin, cin2, cout = 48, 64, 32, 40
    xdt = torch.bfloat16 if cfg.get("x_bf16") else torch.float32
    x64 = ints((rows, cin), 2, g)
    x2_64 = ints((rows, cin2), 2, g) if cfg.get("x2") else None
    K = cin + (cin2 if x2_64 is not None else 0)
    w64 = ints((cout, K), 2, g)
    b64 = eighths((cout,), g) if cfg.get("bias", True) else None
    m64 = pick([0.0, 2.0], (rows, cout), g) if cfg.get("mask") else None
    cs64 = pick([0.5, 1.0, 1.5, 2.0], (cout,), g) if cfg.get("cs") else None
    r64 = eighths((rows, cout), g) if cfg.get("res") else None
    gy64 = eighths((rows, cout), g)

    leaf = lambda t, dt=torch.float32: None if t is None else t.to(dt).to(dev()).requires_grad_(True)
    x, x2, w, b, cs, r = leaf(x64, xdt), leaf(x2_64), leaf(w64), leaf(b64), leaf(cs64), leaf(r64)
    m = m64.float().to(dev()) if m64 is not None else None
    y = lin.linear(x, w, b, cfg.get("act"), m, x2, cs, r, out_bf16=cfg.get("out_bf16", False))
    y.backward(gy64.to(y.dtype).to(dev()))

    D = lambda t: None if t is None else t.to(dev())
    x64, x2_64, w64, b64, m64, cs64, r64, gy64 = map(D, (x64, x2_64, w64, b64, m64, cs64, r64, gy64))
    xc = torch.cat((x64, x2_64), 1) if x2_64 is not None else x64
    z = xc @ w64.t() + (b64 if b64 is not None else 0)
    a = z.clamp_min(0) if cfg.get("act") == "relu" else z
    yr = a * (m64 if m64 is not None else 1) * (cs64 if cs64 is not None else 1) + (r64 if r64 is not None else 0)
    assert torch.equal(y.to(F64), bf16r(yr) if cfg.get("out_bf16") else yr)
    gd = gy64 * (m64 if m64 is not None else 1)
    if cs64 is not None:
        assert torch.equal(cs.grad.to(F64), (gd * bf16r(z)).sum(0)), "colscale"
        gd = gd * cs64
    if cfg.get("act") == "relu":
        gd = gd * (z > 0)
    dz = bf16r(gd)
    gx = dz @ w64
    if xdt == torch.bfloat16 and x2 is None:
        gx = bf16r(gx)
    assert torch.equal(x.grad.to(F64), gx[:, :cin]), "x"
    if x2 is not None:
        assert torch.equal(x2.grad.to(F64), gx[:, cin:]), "x2"
    assert torch.equal(w.grad.to(F64), dz.t() @ xc), "weight"
    if b is not None:
        assert torch.equal(b.grad.to(F64), gd.sum(0)), "bias"
    if r is not None:
        assert torch.equal(r.grad.to(F64), gy64), "residual"
