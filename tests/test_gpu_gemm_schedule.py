"""The tcgen05 GEMM (csrc/gemm_tcgen05.cuh, csrc/gemm.cu) across its persistent schedules.

Both kernels are persistent: CTA (or CTA pair) i runs tiles i, i + grid, ... and two TMEM accumulator stages alternate from one
tile to the next. The operator tests in test_gpu_ops.py give almost every CTA a single tile; here the SM limit
(vqacl_set_gemm_sm_limit) and shapes sized from the device's SM count give every CTA several tiles, with a partial last wave.

Every result is checked element by element against an fp64 reference of the same operation:

    |C - ref| <= C_BOUND * sqrt(K) * 2^-24 * |alpha| * (|A| @ |B|^T)_ij  +  2^-8 |ref| (bf16 outputs) or 2^-23 |ref| (fp32 outputs)

with C_BOUND = 16. The second term is the rounding of the stored result (and of the residual / accumulate add). For K = 768 the
first term is several hundred times below the error of one dropped 64-deep k-block, and about 5x below it at K = 17 920. Operands
are stored with NaN past their logical extent (and NaN rows below), so a read outside the operand poisons the result, and outputs
are pre-filled with NaN or live inside sentinel-filled buffers, so an unwritten or stray element is seen.

A tile's arithmetic does not depend on which CTA runs it or when, so for a fixed tile shape every output is also compared bit for
bit across SM limits and, for the CTA-pair kernel, with the dynamic tile schedule on and off. The one exception is the atomic
epilogue with split-K, whose red.global.add order varies: it gets the fp64 bound only.

The SM limit and the dynamic schedule are process-wide settings; `schedule()` restores them even when a test fails.
"""
import contextlib
import math
import os

import pytest
import torch

import cabi
from vqacl_b200._lib import VqaclError

pytestmark = pytest.mark.gpu

DEV = "cuda"
C_BOUND = 16.0
LIMITS = (0, 2, 6, 22, 132)          # 132 = 148 SMs minus the 16 left to NCCL during multi-GPU backward
MAJORS = {"KK": (0, 0), "KM": (0, 1), "MM": (1, 1)}
ALPHA = {0: -0.75, 1: 1.5, 2: -1.25, 3: 0.5, 4: -2.0, 5: 0.375}
SENT = 3.25                          # sentinel of the buffers around an output window

_WORST = [0.0]                       # largest observed |C - ref| / (sqrt(K) 2^-24 |alpha| |A||B|^T) beyond the rounding term


@pytest.fixture(scope="module", autouse=True)
def _report_worst():
    yield
    print(f"\n[gemm schedule] worst accumulation error: {_WORST[0]:.3f} x sqrt(K) 2^-24 |A||B|^T (bound {C_BOUND})")


def _default_dynamic():
    return 1 if os.environ.get("VQACL_GEMM_DYN", "").startswith("1") else 0


@contextlib.contextmanager
def schedule(sm_limit=0, dynamic=None):
    """Run the body with the GEMM SM limit (0 = all) and, if given, the dynamic schedule on or off; restore the library's
    defaults (no limit; dynamic schedule only if VQACL_GEMM_DYN starts with 1) afterwards, whatever happens."""
    try:
        cabi.set_gemm_sm_limit(sm_limit)
        if dynamic is not None:
            cabi.set_gemm_dynamic_schedule(dynamic)
        yield
    finally:
        cabi.set_gemm_sm_limit(0)
        cabi.set_gemm_dynamic_schedule(_default_dynamic())


def n_sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def ctas(limit, pair):
    """CTAs (pairs for the CTA-pair kernel) a launch may occupy: mirrors gemm_sms() in gemm.cu."""
    n = n_sms()
    lim = limit & ~1 if limit > 0 else 0
    if lim and lim < n:
        n = lim
    return n // 2 if pair else n


def tiles_of(M, N, bn, splits=1):
    bm, bw = (256, 256) if bn == 512 else (128, bn)
    return -(-M // bm) * -(-N // bw) * splits


def schedule_shape(bn, M=1100, min_per_cta=3):
    """N (ragged, multiple of 8) such that at every limit of LIMITS each CTA gets >= min_per_cta tiles at no limit, and the
    number of CTAs does not divide the tile count (the last wave is partial), whatever the device's SM count."""
    pair = bn == 512
    bw = 256 if pair else bn
    mt = -(-M // (256 if pair else 128))
    nt = max(1, -(-min_per_cta * ctas(0, pair) // mt))
    while True:
        t = mt * nt
        if all(c == 1 or t % c for c in (min(ctas(l, pair), t) for l in LIMITS)):
            break
        nt += 1
    return M, nt * bw - 24


def rand_bf16(*shape, scale=1.0):
    return (torch.randn(*shape, device=DEV) * scale).bfloat16()


def operand(t, mn, pad=8):
    """Store a logical [R, K] bf16 operand the way the kernel reads it: K-major (rows of K) or MN-major (stored transposed,
    [K, R]). The stored rows are padded to a multiple of 8 elements plus `pad`, and the padding and one extra row hold NaN."""
    src = t.t() if mn else t
    r, c = src.shape
    pitch = (c + 7) // 8 * 8 + pad
    buf = torch.full((r + 1, pitch), float("nan"), dtype=torch.bfloat16, device=DEV)
    buf[:r, :c] = src
    return buf[:r, :c]


def ref64(At, Bt):
    a, b = At.double(), Bt.double()
    return a @ b.t(), a.abs() @ b.abs().t()


def assert_bound(C, ref, absprod, K, scale=1.0, what=""):
    """Element-wise fp64 bound (module docstring); NaN or unwritten elements fail."""
    bf16_out = C.dtype == torch.bfloat16
    err = (C.double() - ref).abs()
    rnd = (2.0 ** -8 if bf16_out else 2.0 ** -23) * ref.abs()
    acc = (math.sqrt(K) * 2.0 ** -24 * abs(scale)) * absprod
    ok = err <= C_BOUND * acc + rnd
    if not bool(ok.all()):
        bad = (~ok).nonzero()[:4].tolist()
        i = tuple(bad[0])
        raise AssertionError(f"{what}: {int((~ok).sum())} of {ok.numel()} elements outside the fp64 bound, e.g. {bad}: "
                             f"got {C[i].item()}, want {ref[i].item()}, bound {(C_BOUND * acc + rnd)[i].item():.3g}")
    _WORST[0] = max(_WORST[0], ((err - rnd).clamp_min(0) / acc.clamp_min(1e-300)).max().item())


def pack_bits(bits):
    """[M, N] bool -> [M, ceil(N/32)] int32, bit i of word w = column 32 w + i (the ReLU mask layout of the epilogues)."""
    M, N = bits.shape
    W = (N + 31) // 32
    b = torch.zeros(M, W * 32, device=bits.device, dtype=torch.int64)
    b[:, :N] = bits
    v = (b.view(M, W, 32) << torch.arange(32, device=bits.device)).sum(-1)
    return torch.where(v >= 2 ** 31, v - 2 ** 32, v).to(torch.int32)


def unpack_bits(R, N):
    M, W = R.shape
    return ((R.long().unsqueeze(-1) >> torch.arange(32, device=R.device)) & 1).view(M, W * 32)[:, :N].bool()


def nan_like(M, N, dtype):
    return torch.full((M, N), float("nan"), device=DEV, dtype=dtype)


class Case:
    """One epilogue on one problem: fresh output buffers per run, the fp64 reference of the epilogue math."""

    def __init__(self, epi, M, N, K, acc, absprod, splits=1, seed=0):
        self.epi, self.M, self.N, self.K, self.splits = epi, M, N, K, splits
        self.alpha = ALPHA[epi]
        g = torch.Generator(device=DEV).manual_seed(seed)
        self.R = None
        ref = self.alpha * acc
        if epi == 1:
            ref = ref.clamp_min(0)
        elif epi == 2:
            self.R = torch.randn(M, N, device=DEV, generator=g) * 4
            ref = ref + self.R.double()
        elif epi == 3:
            self.C0 = torch.randn(M, N, device=DEV, generator=g)
            ref = ref + self.C0.double()
        elif epi == 4:
            keep = torch.rand(M, N, device=DEV, generator=g) > 0.5
            self.R = pack_bits(keep)
            ref = ref * keep
        self.ref, self.absprod = ref, absprod

    def run(self, A, a_mn, B, b_mn, bn):
        M, N, epi = self.M, self.N, self.epi
        if epi == 3:
            C = self.C0.clone()
        else:
            C = nan_like(M, N, torch.float32 if epi in (2, 5) else torch.bfloat16)
        R = self.R
        if epi == 1:
            R = torch.full((M, (N + 31) // 32), 0x5A5A5A5A, device=DEV, dtype=torch.int32)
        cabi.gemm(A, a_mn, B, b_mn, C, R, M, N, self.K, epi, alpha=self.alpha, splits=self.splits, bn=bn)
        return (C, R) if epi == 1 else (C,)

    def check(self, out, what):
        assert_bound(out[0], self.ref, self.absprod, self.K, self.alpha, what)
        if self.epi == 1:        # the sign mask marks exactly the stored non-zero activations
            assert torch.equal(unpack_bits(out[1], self.N), out[0].float() > 0), what


def same(a, b):
    return all(torch.equal(x, y) for x, y in zip(a, b))


# ------------------------------------------------------------------------------------------------ schedule invariance
@pytest.mark.parametrize("majors", list(MAJORS))
@pytest.mark.parametrize("bn", [64, 128, 256, 512])
def test_every_epilogue_is_schedule_invariant(bn, majors):
    """Epilogues 0-5 at a shape where every CTA runs >= 3 tiles and the last wave is partial: within the fp64 bound, and bit
    for bit the same at every SM limit (and, on CTA pairs, with the dynamic schedule); epilogue 3 also with 3-way split-K."""
    a_mn, b_mn = MAJORS[majors]
    pair = bn == 512
    M, N = schedule_shape(bn)
    K = 456                                   # 7 full k-blocks + 8
    tiles = tiles_of(M, N, bn)
    for lim in LIMITS:
        c = min(ctas(lim, pair), tiles)
        assert tiles >= 3 * c and (c == 1 or tiles % c), (lim, tiles, c)
    torch.manual_seed(bn + a_mn + 2 * b_mn)
    At, Bt = rand_bf16(M, K), rand_bf16(N, K)
    A, B = operand(At, a_mn), operand(Bt, b_mn)
    acc, absprod = ref64(At, Bt)
    cases = [Case(e, M, N, K, acc, absprod, seed=e) for e in range(6)] + [Case(3, M, N, K, acc, absprod, splits=3, seed=9)]
    runs = [(lim, dyn) for lim in LIMITS for dyn in ((0, 1) if pair else (None,))]
    for case in cases:
        first = None
        for lim, dyn in runs:
            with schedule(lim, dyn):
                out = case.run(A, a_mn, B, b_mn, bn)
            what = f"epi {case.epi} splits {case.splits} bn {bn} {majors} limit {lim} dynamic {dyn}"
            if case.splits > 1:
                case.check(out, what)
            elif first is None:
                case.check(out, what)
                first = out
            else:
                assert same(out, first), what + ": differs from the unlimited launch"


@pytest.mark.parametrize("bn", [64, 128, 256, 512])
def test_dropout_epilogues_schedule_invariant_with_wide_pitch(bn):
    """The fused dropout of epilogues 1 and 2 under every SM limit, with the output inside a wider buffer (ldc > N): the kept
    set equals the host hash of row * N + col bit for bit, the values are within the fp64 bound, and nothing outside the
    window changes."""
    M, N = schedule_shape(bn)
    K = 200
    torch.manual_seed(70 + bn)
    At, Bt = rand_bf16(M, K), rand_bf16(N, K)
    A, B = operand(At, 0), operand(Bt, 0)
    acc, absprod = ref64(At, Bt)
    thr = int(0.1 * 65536 + 0.5)
    inv = 65536.0 / (65536.0 - thr)
    key = 0x2468ACE1
    scale = cabi.dropout_scale_host(M, N, thr, inv, key, DEV).double()
    for epi in (1, 2):
        ref = (acc.clamp_min(0) if epi == 1 else acc) * scale      # epi 2 with R = 0: C is exactly acc * scale
        first = None
        for lim in LIMITS:
            dt = torch.bfloat16 if epi == 1 else torch.float32
            big = torch.full((M + 2, N + 24), SENT, device=DEV, dtype=dt)
            C = big[:M, 8:8 + N]
            R = torch.zeros(M, (N + 31) // 32, device=DEV, dtype=torch.int32) if epi == 1 else torch.zeros(M, N, device=DEV)
            with schedule(lim):
                cabi.gemm_dropout(A, B, C, R, M, N, K, epi, thr, inv, key, bn=bn)
            what = f"dropout epi {epi} bn {bn} limit {lim}"
            outside = torch.ones_like(big, dtype=torch.bool)
            outside[:M, 8:8 + N] = False
            assert bool((big[outside] == SENT).all()), what + ": wrote outside the output window"
            if first is None:
                assert_bound(C, ref, absprod * inv, K, 1.0, what)
                if epi == 2:
                    assert torch.equal(C != 0, scale != 0), what + ": kept set differs from the host hash"
                else:
                    clear = acc > 1e-3 * absprod
                    assert torch.equal((C != 0) & clear, (scale != 0) & clear), what + ": kept set differs from the host hash"
                    assert torch.equal(unpack_bits(R, N), C.float() > 0), what
                first = (C.clone(), R.clone())
            else:
                assert torch.equal(C, first[0]) and torch.equal(R, first[1]), what + ": differs from the unlimited launch"


@pytest.mark.parametrize("bn", [256, 512])
def test_fused_argmax_at_decode_size_schedule_invariant(bn):
    """EPI_ARGMAX at the decoding shape (M = 512 rows, N = 32 200 vocabulary) with several tiles per CTA: the partial maxima are
    bit for bit the same at every limit, slots past the last are untouched, the merged argmax is the fp64 first maximum
    (exact tie -> lower index)."""
    M, N, K = 512, 32200, 768
    pair = bn == 512
    tiles = tiles_of(M, N, bn)
    assert tiles >= 3 * ctas(0, pair), tiles
    torch.manual_seed(41)
    At, Bt = rand_bf16(M, K), rand_bf16(N, K)
    Bt[777] = Bt[31999]
    At[5] = Bt[31999] * 0.5
    ref = (At.double() @ Bt.double().t()) * 0.125
    slots = ((N + 255) // 256) * 2
    pitch = (slots + 15) // 8 * 8 + 8       # a multiple of 8 with >= 8 spare slots per row
    first = None
    for lim in LIMITS:
        pv = torch.full((M + 1, pitch), SENT, device=DEV)
        pi = torch.full((M + 1, pitch), -7, device=DEV, dtype=torch.int32)
        with schedule(lim):
            cabi.gemm(At, 0, Bt, 0, pv[:M], pi[:M], M, N, K, 6, alpha=0.125, bn=bn)
        what = f"argmax bn {bn} limit {lim}"
        assert bool((pv[:, slots:] == SENT).all() and (pv[M] == SENT).all()), what + ": value slot past the last written"
        assert bool((pi[:, slots:] == -7).all() and (pi[M] == -7).all()), what + ": index slot past the last written"
        if first is None:
            v, _ = pv[:M, :slots].max(dim=1)
            cand = torch.where(pv[:M, :slots] == v[:, None], pi[:M, :slots].long(), torch.full_like(pi[:M, :slots].long(), 1 << 40))
            idx = cand.min(dim=1).values
            assert idx[5].item() == 777, what
            top2 = ref.topk(2, dim=1)
            gap = top2.values[:, 0] - top2.values[:, 1]
            tol = 0.125 * C_BOUND * math.sqrt(K) * 2.0 ** -24 * (At.double().abs() @ Bt.double().abs().t()).max(dim=1).values
            assert bool(((idx == top2.indices[:, 0]) | (gap <= 2 * tol)).all()), what
            assert bool(((v.double() - top2.values[:, 0]).abs() <= tol).all()), what
            first = (pv, pi)
        else:
            assert torch.equal(pv, first[0]) and torch.equal(pi, first[1]), what + ": differs from the unlimited launch"


# ------------------------------------------------------------------------------------------------ row tails
@pytest.mark.parametrize("M", [300, 1000, 17920])
def test_rmsnorm_row_tail_with_several_blocks_per_pair(M):
    """GEMM + residual + RMSNorm row tail when a CTA pair owns several 256-row blocks (SM limit 2 and 6): C, the bf16 norm output
    equal the unlimited launch bit for bit; C is within the fp64 bound and the norm output within bf16 rounding of the fp64 norm."""
    K = 768
    torch.manual_seed(80 + M)
    At, Bt = rand_bf16(M, K, scale=0.5), rand_bf16(768, K, scale=0.05)
    R = torch.randn(M, 768, device=DEV) * 3
    w = torch.rand(768, device=DEV) + 0.5
    acc, absprod = ref64(At, Bt)
    ref = acc + R.double()
    C0, n0 = cabi.gemm_resid_rmsnorm(At, Bt, R, w)
    assert_bound(C0, ref, absprod, K, 1.0, f"row tail C, M {M}")
    rstd = torch.rsqrt(ref.pow(2).mean(-1, keepdim=True) + 1e-6)
    refn = ref * rstd * w.double()
    errn = (n0.double() - refn).abs()
    assert bool((errn <= 2.0 ** -7 * refn.abs() + 1e-5 * rstd * w.double()).all()), f"row tail norm, M {M}"
    assert -(-M // 256) > ctas(2, True)       # at limit 2 one pair owns every 256-row block
    for lim in (2, 6):
        with schedule(lim):
            C, n = cabi.gemm_resid_rmsnorm(At, Bt, R, w)
        assert torch.equal(C, C0) and torch.equal(n, n0), f"row tail M {M} limit {lim}: differs from the unlimited launch"


@pytest.mark.parametrize("B,N", [(17, 36), (320, 36)])
def test_visual_embedding_row_tail_with_several_blocks_per_pair(B, N):
    """The VisualEmbedding GEMM + row tail at B*N = 612 and 11 520 rows under SM limit 2 and 6: featpre and x bit for bit equal to
    the unlimited launch, featpre within the fp64 bound, x equal to the stand-alone tail kernel on that featpre and close to an
    fp64 evaluation of the module."""
    F, V = 2048, 100
    torch.manual_seed(90 + B)
    feats = torch.relu(torch.randn(B * N, F, device=DEV)).bfloat16()
    Wf = rand_bf16(768, F, scale=0.02)
    boxes = torch.rand(B, N, 4, device=DEV)
    bf, wf = torch.randn(768, device=DEV) * 0.1, torch.rand(768, device=DEV) + 0.5
    Wp, bp, wp = torch.randn(768, 5, device=DEV) * 0.3, torch.randn(768, device=DEV) * 0.1, torch.rand(768, device=DEV) + 0.5
    img, shared = torch.randn(2, 768, device=DEV), torch.randn(V, 768, device=DEV)
    args = (bf, wf, Wp, bp, wp, img, shared)
    x0, p0 = cabi.visual_embed_fused(feats, Wf, boxes, *args, B, N)
    acc, absprod = ref64(feats, Wf)
    assert_bound(p0, acc, absprod, F, 1.0, f"visual featpre B*N {B * N}")
    assert torch.equal(x0, cabi.visual_embed_fwd(p0, boxes, *args, B, N))

    def rms(t):
        return t * torch.rsqrt(t.pow(2).mean(-1, keepdim=True) + 1e-6)

    bx = boxes.view(B * N, 4).double()
    area = (bx[:, 3] - bx[:, 2]) * (bx[:, 1] - bx[:, 0])
    pos = torch.cat([bx, area[:, None]], 1) @ Wp.double().t() + bp.double()
    xr = rms(acc + bf.double()) * wf.double() + rms(pos) * wp.double() + img[0].double()
    xr = xr + shared.double()[V - 1 - torch.arange(N, device=DEV)].repeat(B, 1)
    assert bool(((x0.view(B * N, 768).double() - xr).abs() <= 1e-4 * (1 + xr.abs())).all()), "visual x vs fp64"
    for lim in (2, 6):
        with schedule(lim):
            x, p = cabi.visual_embed_fused(feats, Wf, boxes, *args, B, N)
        assert torch.equal(p, p0) and torch.equal(x, x0), f"visual B*N {B * N} limit {lim}: differs from the unlimited launch"


# ------------------------------------------------------------------------------------------------ grouped kernel
DEC_DW = [(768, 3072), (3072, 768), (768, 768), (768, 768), (768, 768), (2304, 768)]
RAGGED = [(100, 264), (520, 8), (768, 776), (1000, 40), (129, 3072), (2304, 768), (257, 520), (8, 8)]


@pytest.mark.parametrize("shapes,K", [(DEC_DW, 1600), (RAGGED, 1000)], ids=["decoder_dw", "ragged"])
def test_grouped_weight_gradients_under_sm_limits(shapes, K):
    """The grouped CTA-pair launch (decoder weight gradients) at every SM limit: the store epilogue bit for bit equal to the
    unlimited launch and within the fp64 bound, the accumulate epilogue within the bound; outputs live in sentinel buffers
    (problem M < 128: the peer CTA owns no rows; N = 8)."""
    torch.manual_seed(K + len(shapes))
    Ats = [rand_bf16(m, K, scale=0.5) for m, _ in shapes]
    Bts = [rand_bf16(n, K, scale=0.5) for _, n in shapes]
    As = [operand(a, 1) for a in Ats]
    Bs = [operand(b, 1) for b in Bts]
    refs = [ref64(a, b) for a, b in zip(Ats, Bts)]
    C0s = [torch.randn(m, n, device=DEV) for m, n in shapes]
    first = None
    for epi in (5, 3):
        for lim in LIMITS:
            bigs = [torch.full((m + 3, n + 16), SENT, device=DEV) for m, n in shapes]
            views = [g[1:1 + m, 8:8 + n] for g, (m, n) in zip(bigs, shapes)]
            if epi == 3:
                for v, c0 in zip(views, C0s):
                    v.copy_(c0)
            with schedule(lim):
                cabi.gemm_grouped_mn(As, Bs, views, epi=epi, alpha=-0.5)
            for i, (g, v, (m, n)) in enumerate(zip(bigs, views, shapes)):
                what = f"grouped epi {epi} problem {i} ({m} x {n}) limit {lim}"
                outside = torch.ones_like(g, dtype=torch.bool)
                outside[1:1 + m, 8:8 + n] = False
                assert bool((g[outside] == SENT).all()), what + ": wrote outside the output"
                if epi == 3 or lim == 0:
                    acc, absprod = refs[i]
                    assert_bound(v, -0.5 * acc + (C0s[i].double() if epi == 3 else 0), absprod, K, 0.5, what)
            if epi == 5:
                outs = [v.clone() for v in views]
                if first is None:
                    first = outs
                else:
                    assert all(torch.equal(a, b) for a, b in zip(outs, first)), f"grouped limit {lim}: differs from the unlimited launch"


# ------------------------------------------------------------------------------------------------ dynamic-schedule ring
RING_SHAPES = [(600, 1000, 128, 0), (1100, 2800, 200, 22), (2000, 5000, 136, 0), (1100, 2800, 200, 6), (600, 1000, 128, 132),
               (2000, 5000, 136, 22)]      # (M, N, K, SM limit): 12, 55 and 160 pair tiles on 74, 11, 3 or 66 pairs


def _ring_inputs():
    torch.manual_seed(123)
    ins, want = [], []
    for M, N, K, _ in RING_SHAPES:
        A, B = rand_bf16(M, K), rand_bf16(N, K)
        C = nan_like(M, N, torch.float32)
        with schedule(0, 0):
            cabi.gemm(A, 0, B, 0, C, None, M, N, K, 5, alpha=0.5, bn=512)
        ins.append((A, B))
        want.append(C)
    return ins, want


def test_dynamic_schedule_ring_reuse():
    """More than 600 back-to-back dynamically scheduled CTA-pair launches on one stream (every one of the 256 counter slots is
    reused at least twice), alternating shapes with different work and pair counts: each output equals the static schedule's."""
    ins, want = _ring_inputs()
    n, batch = 612, 36
    with schedule(0, 1):
        for b0 in range(0, n, batch):
            outs = []
            for i in range(b0, b0 + batch):
                j = i % len(RING_SHAPES)
                M, N, K, lim = RING_SHAPES[j]
                C = nan_like(M, N, torch.float32)
                cabi.set_gemm_sm_limit(lim)
                cabi.gemm(ins[j][0], 0, ins[j][1], 0, C, None, M, N, K, 5, alpha=0.5, bn=512)
                outs.append((i, j, C))
            for i, j, C in outs:
                assert torch.equal(C, want[j]), f"dynamic launch {i} (shape {RING_SHAPES[j]}) differs from the static schedule"


def test_dynamic_schedule_on_two_concurrent_streams():
    """Two streams each running a chain of dynamically scheduled launches at the same time (as the decoder backward's side
    stream does): every result equals the serial static one."""
    ins, want = _ring_inputs()
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    for s in streams:
        s.wait_stream(torch.cuda.current_stream())
    outs = []
    with schedule(0, 1):
        for i in range(48):
            for si, s in enumerate(streams):
                j = (i + 3 * si) % len(RING_SHAPES)
                M, N, K, lim = RING_SHAPES[j]
                with torch.cuda.stream(s):
                    C = nan_like(M, N, torch.float32)
                    cabi.set_gemm_sm_limit(lim)
                    cabi.gemm(ins[j][0], 0, ins[j][1], 0, C, None, M, N, K, 5, alpha=0.5, bn=512)
                outs.append((i, si, j, C))
        torch.cuda.synchronize()
    for i, si, j, C in outs:
        assert torch.equal(C, want[j]), f"stream {si} launch {i} (shape {RING_SHAPES[j]}) differs from the static schedule"


# ------------------------------------------------------------------------------------------------ edge shapes
EDGE = [(1, 8, 1), (2, 40, 13), (127, 264, 63), (129, 8, 65), (257, 40, 1000), (1, 264, 1000), (129, 264, 13), (127, 40, 65),
        (257, 8, 63), (2, 264, 65), (257, 264, 1), (129, 40, 1000)]


@pytest.mark.parametrize("majors", list(MAJORS))
@pytest.mark.parametrize("M,N,K", EDGE)
def test_edge_shapes_every_tile_width(M, N, K, majors):
    """M in {1, 2, 127, 129, 257}, N in {8, 40, 264}, K in {1, 13, 63, 65, 1000}, every tile width, NaN past every operand's
    extent: the fp32 store into a window of a sentinel buffer (ldc > N, rows below) and the atomic epilogue with more splits
    than k-blocks and with a split count that does not divide them."""
    a_mn, b_mn = MAJORS[majors]
    torch.manual_seed(M * 7 + N * 3 + K)
    At, Bt = rand_bf16(M, K), rand_bf16(N, K)
    A, B = operand(At, a_mn), operand(Bt, b_mn)
    acc, absprod = ref64(At, Bt)
    kb = -(-K // 64)
    for bn in (64, 128, 256, 512):
        big = torch.full((M + 5, N + 16), SENT, device=DEV)
        C = big[2:2 + M, 8:8 + N]
        cabi.gemm(A, a_mn, B, b_mn, C, None, M, N, K, 5, alpha=-1.5, bn=bn)
        what = f"edge {M}x{N}x{K} {majors} bn {bn}"
        outside = torch.ones_like(big, dtype=torch.bool)
        outside[2:2 + M, 8:8 + N] = False
        assert bool((big[outside] == SENT).all()), what + ": wrote outside the output window"
        assert_bound(C, -1.5 * acc, absprod, K, 1.5, what)
        Cb = nan_like(M, N, torch.bfloat16)
        cabi.gemm(A, a_mn, B, b_mn, Cb, None, M, N, K, 0, alpha=0.75, bn=bn)
        assert_bound(Cb, 0.75 * acc, absprod, K, 0.75, what + " bf16")
        for splits in (kb + 3, 7):
            C0 = torch.randn(M, N, device=DEV)
            C = C0.clone()
            cabi.gemm(A, a_mn, B, b_mn, C, None, M, N, K, 3, alpha=0.5, splits=splits, bn=bn)
            assert_bound(C, 0.5 * acc + C0.double(), absprod, K, 0.5, f"{what} splits {splits}")


@pytest.mark.parametrize("majors", list(MAJORS))
def test_strided_operands_from_wide_poisoned_buffers(majors):
    """Operands as column slices of [rows, 2304] buffers at base offset 768 (the engine's packed QKV layout), everything else NaN,
    K not a multiple of 64: every tile width gives a finite result within the fp64 bound."""
    a_mn, b_mn = MAJORS[majors]
    M, N, K = 520, 392, 700
    torch.manual_seed(11 + a_mn + b_mn)
    At, Bt = rand_bf16(M, K), rand_bf16(N, K)

    def packed(t, mn):
        src = t.t() if mn else t
        buf = torch.full((src.shape[0] + 3, 2304), float("nan"), dtype=torch.bfloat16, device=DEV)
        buf[:src.shape[0], 768:768 + src.shape[1]] = src
        return buf[:src.shape[0], 768:768 + src.shape[1]]

    A, B = packed(At, a_mn), packed(Bt, b_mn)
    assert A.stride(0) == 2304 and B.stride(0) == 2304
    acc, absprod = ref64(At, Bt)
    for bn in (64, 128, 256, 512):
        C = nan_like(M, N, torch.float32)
        cabi.gemm(A, a_mn, B, b_mn, C, None, M, N, K, 5, bn=bn)
        assert bool(torch.isfinite(C).all()), f"strided {majors} bn {bn}: read past the operand"
        assert_bound(C, acc, absprod, K, 1.0, f"strided {majors} bn {bn}")


def test_mask_and_residual_windows_leave_the_rest_untouched():
    """ReLU mask words past ceil(N / 32) and rows past M, outputs with ldc > N: only the window is written."""
    M, N, K = 300, 200, 128
    torch.manual_seed(5)
    At, Bt = rand_bf16(M, K), rand_bf16(N, K)
    acc, absprod = ref64(At, Bt)
    W = (N + 31) // 32
    for bn in (64, 128, 256, 512):
        bigc = torch.full((M + 3, N + 40), SENT, device=DEV, dtype=torch.bfloat16)
        bigr = torch.full((M + 3, W + 5), 0x0F0F0F0F, device=DEV, dtype=torch.int32)
        C, R = bigc[:M, 8:8 + N], bigr[:M, :W]
        cabi.gemm(At, 0, Bt, 0, C, R, M, N, K, 1, alpha=2.0, bn=bn)
        assert bool((bigr[:, W:] == 0x0F0F0F0F).all() and (bigr[M:] == 0x0F0F0F0F).all()), f"mask bn {bn}: words outside written"
        out = torch.ones_like(bigc, dtype=torch.bool)
        out[:M, 8:8 + N] = False
        assert bool((bigc[out] == SENT).all()), f"relu bn {bn}: wrote outside the window"
        assert_bound(C, (2.0 * acc).clamp_min(0), absprod, K, 2.0, f"relu bn {bn}")
        assert torch.equal(unpack_bits(R, N), C.float() > 0)
        Rr = torch.randn(M + 1, N + 16, device=DEV)[:M, :N]
        bigf = torch.full((M + 3, N + 24), SENT, device=DEV)
        Cf = bigf[1:1 + M, 16:16 + N]
        cabi.gemm(At, 0, Bt, 0, Cf, Rr, M, N, K, 2, alpha=-1.0, bn=bn)
        outf = torch.ones_like(bigf, dtype=torch.bool)
        outf[1:1 + M, 16:16 + N] = False
        assert bool((bigf[outf] == SENT).all()), f"residual bn {bn}: wrote outside the window"
        assert_bound(Cf, Rr.double() - acc, absprod, K, 1.0, f"residual bn {bn}")


# ------------------------------------------------------------------------------------------------ rejections
def _rejects(fn, match):
    before = cabi.launch_count()
    with pytest.raises(VqaclError, match=match):
        fn()
    torch.cuda.synchronize()
    assert cabi.launch_count() == before


def test_unsupported_calls_are_rejected_without_launching():
    """Calls the kernels cannot do correctly return an error with a message and launch nothing. Every buffer is large enough
    for the call as written, so a missing check would give a wrong answer, not an out-of-bounds access."""
    M, N, K = 256, 264, 128
    A, B = rand_bf16(M + 8, K + 64), rand_bf16(N + 8, K + 64)
    Cf = torch.zeros(M + 8, N + 64, device=DEV)
    Cb = torch.zeros(M + 8, N + 64, device=DEV, dtype=torch.bfloat16)
    mask = torch.zeros(M + 8, 16, device=DEV, dtype=torch.int32)
    Rf = torch.zeros(M + 8, N + 64, device=DEV)
    _rejects(lambda: cabi.gemm(A, 0, B, 0, Cf, None, M, 260, K, 5), "multiple of 8")
    _rejects(lambda: cabi.gemm(A, 0, B, 0, Cf.as_strided((M, N), (N + 4, 1)), None, M, N, K, 5), "multiple of 8")
    _rejects(lambda: cabi.gemm(A, 0, B, 0, Cf.as_strided((M, N), (N - 8, 1)), None, M, N, K, 5), ">= N")
    for epi, R, C in ((0, None, Cb), (1, mask, Cb), (2, Rf, Cf), (4, mask, Cb)):
        _rejects(lambda: cabi.gemm(A, 0, B, 0, C, R, M, N, K, epi, splits=2), "split-K")
    Nv = 2056                                         # 18 argmax slots per row: 16 is a valid pitch that is too small
    Bv = rand_bf16(Nv + 8, K + 64)
    slots = ((Nv + 255) // 256) * 2
    pv = torch.zeros(M + 8, 64, device=DEV)
    pi = torch.zeros(M + 8, 64, device=DEV, dtype=torch.int32)
    for bn in (64, 128):
        _rejects(lambda: cabi.gemm(A, 0, Bv, 0, pv, pi, M, Nv, K, 6, bn=bn), "256-wide")
    few = slots - 2
    _rejects(lambda: cabi.gemm(A, 0, Bv, 0, pv.as_strided((M, few), (few, 1)), pi, M, Nv, K, 6, bn=256), "slots")
    _rejects(lambda: cabi.gemm(A, 0, Bv, 0, pv, pi.as_strided((M, few), (few, 1)), M, Nv, K, 6, bn=512), "slots")
    Amn = rand_bf16(K, M + 8)                         # A stored [K, M] (MN-major) with B K-major: no such kernel
    for bn in (0, 128, 512):
        _rejects(lambda: cabi.gemm(Amn, 1, B, 0, Cf, None, M, N, K, 5, bn=bn), "not instantiated")
    Am = A.view(-1)[1:1 + M * (K + 64)].view(M, K + 64)     # base 2 bytes past a 16-byte boundary
    Bm = B.view(-1)[4:4 + N * (K + 64)].view(N, K + 64)
    for bn in (0, 64, 512):
        _rejects(lambda: cabi.gemm(Am, 0, B, 0, Cf, None, M, N, K, 5, bn=bn), "16-byte aligned")
        _rejects(lambda: cabi.gemm(A, 0, Bm, 0, Cf, None, M, N, K, 5, bn=bn), "16-byte aligned")


# ------------------------------------------------------------------------------------------------ slab split-K
@pytest.mark.parametrize("majors", ["KK", "MM"])
@pytest.mark.parametrize("splits,used", [(5, 5), (7, 6), (3, 3), (50, 36), (1, 1)])
def test_slab_split_k(splits, used, majors):
    """The deterministic split-K form (one fp32 slab per split, as the decoder FFN-out uses it), K = 2304 = 36 k-blocks: the
    returned slab count follows the rounding rule (no empty split), each slab is the fp64 partial product over its k-block range,
    and neither the gaps between slabs nor the slabs past the count are written."""
    a_mn, b_mn = MAJORS[majors]
    M, N, K = 1000, 776, 2304
    torch.manual_seed(splits)
    At, Bt = rand_bf16(M, K), rand_bf16(N, K)
    A, B = operand(At, a_mn), operand(Bt, b_mn)
    ldc = N + 8
    stride = (M + 2) * ldc
    per = -(-36 // used)
    for bn in (0, 128, 512):
        buf = torch.full(((used + 1) * stride,), SENT, device=DEV)
        C = buf.as_strided((M, N), (ldc, 1))
        n = cabi.gemm_slabs(A, a_mn, B, b_mn, C, M, N, K, stride, alpha=-0.5, splits=splits, bn=bn)
        assert n == used, (splits, n)
        written = torch.zeros_like(buf, dtype=torch.bool)
        for s in range(used):
            k0, k1 = s * per * 64, min(K, (s + 1) * per * 64)
            slab = buf[s * stride:].as_strided((M, N), (ldc, 1))
            acc, absprod = ref64(At[:, k0:k1], Bt[:, k0:k1])
            assert_bound(slab, -0.5 * acc, absprod, k1 - k0, 0.5, f"slab {s} of {used} bn {bn} {majors}")
            written[s * stride:].as_strided((M, N), (ldc, 1)).fill_(True)
        assert bool((buf[~written] == SENT).all()), f"slabs {used} bn {bn}: wrote outside the slabs"


# ------------------------------------------------------------------------------------------------ step shapes
# (name, M, N, K, splits, A MN-major, B MN-major, epilogue): the 25 GEMMs of profiles/r02_gemm_shapes.txt as the engine issues them
STEP = [("enc qkv", 17920, 2304, 768, 1, 0, 0, 0), ("enc o", 17920, 768, 768, 1, 0, 0, 2), ("enc wi", 17920, 3072, 768, 1, 0, 0, 1),
        ("enc wo", 17920, 768, 3072, 1, 0, 0, 2), ("enc dX wo", 17920, 3072, 768, 1, 0, 1, 4), ("enc dX wi", 17920, 768, 3072, 1, 0, 1, 0),
        ("enc dX o", 17920, 768, 768, 1, 0, 1, 0), ("enc dX qkv", 17920, 768, 2304, 1, 0, 1, 0),
        ("enc dW wo", 768, 3072, 17920, 4, 1, 1, 3), ("enc dW wi", 3072, 768, 17920, 4, 1, 1, 3), ("enc dW o", 768, 768, 17920, 16, 1, 1, 3),
        ("enc dW qkv", 2304, 768, 17920, 5, 1, 1, 3), ("cross KV fwd", 18560, 18432, 768, 1, 0, 0, 0),
        ("cross KV dX", 18560, 768, 18432, 1, 0, 1, 0), ("cross KV dW", 18432, 768, 18560, 1, 1, 1, 3),
        ("vis feat", 11520, 768, 2048, 1, 0, 0, 5), ("lm head", 1600, 32200, 768, 1, 0, 0, 0), ("lm dW", 32200, 768, 1600, 1, 1, 1, 3),
        ("dec qkv", 1600, 2304, 768, 1, 0, 0, 0), ("dec o", 1600, 768, 768, 1, 0, 0, 2), ("dec wi", 1600, 3072, 768, 1, 0, 0, 1),
        ("dec wo", 1600, 768, 3072, 1, 0, 0, 2), ("dec dX 768", 1600, 768, 768, 1, 0, 1, 0), ("dec dW 768", 768, 768, 1600, 3, 1, 1, 3),
        ("dec dW wi", 3072, 768, 1600, 3, 1, 1, 3)]


def cost_model_bn(M, N, K, splits, limit):
    """The tile width gemm_bf16 picks for force_bn = 0 (mirror of its cost model in gemm.cu)."""
    splits = max(1, splits)
    kb = -(-K // 64)
    splits = min(splits, kb)
    splits = -(-kb // -(-kb // splits))
    sms = ctas(limit, False)
    kbs = -(-kb // splits)
    best, bn = -1, 0
    for cand, cyc in ((256, 768), (128, 400), (64, 240)):
        if cand > 64 and N < cand // 2 + 8:
            continue
        work = -(-M // 128) * -(-N // cand) * splits
        cost = -(-work // sms) * (kbs * cyc + 600 + cand * 4)
        if best < 0 or cost < best:
            best, bn = cost, cand
    if N >= 192 and M >= 192:
        work = -(-M // 256) * -(-N // 256) * splits
        cost = -(-work // (sms // 2)) * (kbs * 512 + 900 + 1024)
        if cost < best:
            bn = 512
    return bn


@pytest.mark.parametrize("name,M,N,K,splits,a_mn,b_mn,epi", STEP, ids=[s[0].replace(" ", "_") for s in STEP])
def test_step_shapes_through_the_cost_model(name, M, N, K, splits, a_mn, b_mn, epi):
    """Every GEMM shape of the training step with the tile width left to the cost model, at no SM limit and at 132 SMs: within
    the fp64 bound (on three 128-row stripes for the largest), and bit for bit equal across the two limits whenever the cost
    model picks the same tile width for both."""
    torch.manual_seed(M + N + K)
    At, Bt = rand_bf16(M, K), rand_bf16(N, K)
    A = At.t().contiguous() if a_mn else At
    B = Bt.t().contiguous() if b_mn else Bt
    big = M * N * K > 6e10
    rows = torch.cat([torch.arange(0, 128), torch.arange(M // 2, M // 2 + 128), torch.arange(M - 128, M)]).to(DEV) if big else None
    if big:
        acc, absprod = ref64(At[rows], Bt)
    else:
        acc, absprod = ref64(At, Bt)
    case = Case(epi, M, N, K, torch.zeros(1, device=DEV, dtype=torch.float64), None, splits=splits, seed=1)
    outs = []
    for lim in (0, 132):
        with schedule(lim):
            out = case.run(A, a_mn, B, b_mn, 0)
        sel = (lambda t: t[rows]) if big else (lambda t: t)
        alpha = case.alpha
        ref = alpha * acc
        if epi == 1:
            ref = ref.clamp_min(0)
        elif epi == 2:
            ref = ref + sel(case.R).double()
        elif epi == 3:
            ref = ref + sel(case.C0).double()
        elif epi == 4:
            ref = ref * unpack_bits(sel(case.R), N)
        what = f"{name} limit {lim} bn {cost_model_bn(M, N, K, splits, lim)}"
        assert_bound(sel(out[0]), ref, absprod, K, alpha, what)
        if epi == 1:
            assert torch.equal(unpack_bits(sel(out[1]), N), sel(out[0]).float() > 0), what
        outs.append(out)
        del out
    if cost_model_bn(M, N, K, splits, 0) == cost_model_bn(M, N, K, splits, 132) and not (epi == 3 and splits > 1):
        assert same(outs[0], outs[1]), f"{name}: differs between SM limits 0 and 132 with the same tile width"
