"""Every attention kernel (csrc/attention.cu, csrc/attention_tc.cu) against an fp64 restatement of the same operation.

The reference is written here from scratch (it is checked against the oracle's T5Attention once, on the CPU):

    s = q k^T + table[bucket(k - q - q_off), h] (rel_mode 1: text x text corner only; 2: everywhere) + keymask + causal -10000
    P = softmax(s), P^ = P o scale (the host restatement of the dropout mask), O = P^ V, lse = log sum exp s
    dP = dO V^T, D = rowsum(dO o O), dS = P o (scale o dP - D), dQ = dS K, dK = dS^T Q, dV = P^^T dO, dtable = sum of dS per bucket

Inputs are bf16 and therefore exact; the kernels round P (the tcgen05 kernels the unnormalised exponentials) and dS to bf16,
form D from bf16 operands, and store bf16 results. With u = 2^-9 (one bf16 rounding moves a value by at most 2u relative:
bf16 carries 8 significant bits) every element must satisfy

    forward   |O - O64| <= 4u (P^ |V| + |O64|),          |lse - lse64| <= 2^-16 (1 + max_k |s_ik|)
    backward  |x - x64| <= 8u (env_x + |x64|),           env_dQ = E |K|, env_dK = E^T |Q|, env_dV = P^^T |dO|,
              E = P o (scale o (|dO| |V|^T) + A),        A_i = sum_j |dO_ij| |O_ij|,    env_dtable = sum of E per bucket,

and the table gradient, which goes through fp32 atomics, gets n 2^-24 sum |dS| more (n = entries of the bucket). The max in the
lse bound runs over the keys within 100 of the row maximum (a -1e9 mask would otherwise make it vacuous). The CPU tests show
that this bound catches the bugs it exists for (a neighbouring bucket, a dropped key mask, an off-by-one causal mask, swapped
dropout lanes, the wrong dropout grid, a neighbouring head's K, a neighbouring row's lse, D from the undropped P).

Every row of the dispatch table (tcgen05, single tile with 4 / 2 / 1 warps, key split, multi tile) runs forward and backward with
dropout off and on, and torch.profiler confirms the kernel that ran. The persistent kernels get shapes sized from the SM count
so that every CTA runs at least 3 items and the last wave is partial, and every batch element its own key-mask pattern.
Beyond the bound: V = I (dO = I) reads P^ (P^^T) out entry by entry, including the exact dropout pattern; the packed
layouts of the engine must give the dense results bit for bit and write nothing outside their windows; the KV-cache decode
form runs every step up to position 62; an item gives the same bits alone as inside the persistent launch; invalid calls are
rejected without a launch.
"""
import re
from typing import NamedTuple

import pytest
import torch

import cabi
from vqacl_b200._lib import VqaclError
from vqacl_b200.engine import rel_bucket_table

DEV = "cuda"
U = 2.0 ** -9
FWD_C, BWD_C = 4.0, 8.0
LSE_C = 2.0 ** -16
NB = 32                                 # relative_attention_num_buckets of t5-base
_WORST = {"fwd": 0.0, "bwd": 0.0, "lse": 0.0}


@pytest.fixture(scope="module", autouse=True)
def _report_worst():
    yield
    print(f"\n[attention] worst error ratio: forward {_WORST['fwd']:.3f} u (bound {FWD_C:g}), backward {_WORST['bwd']:.3f} u "
          f"(bound {BWD_C:g}), lse {_WORST['lse']:.3f} x 2^-16 (1 + max|s|) (bound 1)")


def dropout_params(p):
    """(thr16, inv_keep, key) as Engine::drop forms them (engine.cu); p = 0 disables dropout."""
    if p == 0:
        return (0, 1.0, 0)
    t = min(round(p * 65536.0), 65535)
    return (t, float(torch.tensor(65536.0 / (65536.0 - t), dtype=torch.float32)), 0x5EED1234)


def drop_scale(B, H, Sq, Sk, grid, drop, device, swap_lanes=False):
    """[B, H, Sq, Sk] float64 dropout scale of the attention probabilities, or None: element (q, k) of problem b * H + h has
    index ((b * H + h) * grid + q) * grid + k (grid 64: attn_pair_idx, single-tile, key-split and tcgen05 kernels; grid 256:
    mt_pair_idx, multi-tile kernels)."""
    thr, inv, key = drop
    if not thr:
        return None
    blk = torch.arange(B * H, device=device, dtype=torch.int64).view(B, H, 1, 1)
    q = torch.arange(Sq, device=device, dtype=torch.int64).view(1, 1, Sq, 1)
    k = torch.arange(Sk, device=device, dtype=torch.int64).view(1, 1, 1, Sk)
    idx = (blk * grid + q) * grid + k
    if swap_lanes:
        idx = idx ^ 1
    return cabi.dropout_scale_idx(idx, thr, inv, key).double()


def _heads(x, B, S, H):
    return x.double().reshape(B, S, H, 64).transpose(1, 2)


def _rows(x):
    B, H, S, D = x.shape
    return x.transpose(1, 2).reshape(B * S, H * D)


def reference(q, k, v, B, H, Sq, Sk, table=None, bucket=None, rel_mode=0, Lt=0, keymask=None, causal=0, q_off=0, drop=(0, 1.0, 0),
              grid=64, dO=None, mut=()):
    """fp64 results and error envelopes (module docstring). q [B*Sq, H*64], k / v [B*Sk, H*64]; `mut` names deliberate bugs
    (the teeth tests)."""
    dev = q.device
    qh, kh, vh = _heads(q, B, Sq, H), _heads(k, B, Sk, H), _heads(v, B, Sk, H)
    if "head_k" in mut:
        kh = kh.clone()
        kh[:, 0] = kh[:, 1]
    s = qh @ kh.transpose(2, 3)
    qpos = torch.arange(Sq, device=dev) + q_off
    kpos = torch.arange(Sk, device=dev)
    rel = kpos[None, :] - qpos[:, None]
    region = None
    if rel_mode:
        bk = bucket.to(dev).long().clone()
        if "bias_bucket" in mut:
            bk[63 - 1] += 1                                       # distance k - q = -1 takes the next bucket
        bidx = bk[(rel.clamp(-63, 63) + 63)]                     # [Sq, Sk]
        region = torch.ones(Sq, Sk, dtype=torch.bool, device=dev)
        if rel_mode == 1:
            region = (qpos[:, None] < Lt) & (kpos[None, :] < Lt)
        s = s + (table.double()[bidx].permute(2, 0, 1) * region)[None]
    if keymask is not None:
        km = keymask.double().clone()
        if "mask_drop" in mut:
            b0, k0 = (km < 0).nonzero()[-1].tolist()
            km[b0, k0] = 0.0
        s = s + km[:, None, None, :]
    if causal:
        s = s - 10000.0 * (kpos[None, :] > qpos[:, None] + (1 if "causal_off" in mut else 0))
    m = s.amax(-1, keepdim=True)
    e = (s - m).exp()
    l = e.sum(-1, keepdim=True)
    P = e / l
    lse = (m + l.log()).squeeze(-1)
    sc = drop_scale(B, H, Sq, Sk, 64 if "drop_grid" in mut else grid, drop, dev, swap_lanes="drop_lanes" in mut)
    scl = sc if sc is not None else torch.ones_like(P)
    Ph = P * scl
    O = Ph @ vh
    near = s >= m - 100.0
    r = dict(O=_rows(O), envO=_rows(Ph @ vh.abs()), P=P, Ph=Ph, scale=sc,
             lse=lse, smax=torch.where(near, s.abs(), torch.zeros_like(s)).amax(-1))
    if "lse_shift" in mut:                                        # row q uses row q+1's log-sum-exp
        lse_b = torch.cat([lse[..., 1:], lse[..., -1:]], -1)
        r["lse"] = lse_b
        P = torch.exp(s - lse_b[..., None])
    if dO is None:
        return r
    dOh = _heads(dO, B, Sq, H)
    dP = dOh @ vh.transpose(2, 3)
    D = (dOh * O).sum(-1, keepdim=True)
    if "D_undropped" in mut:
        D = (P * dP).sum(-1, keepdim=True)
    dS = P * (scl * dP - D)
    A = (dOh.abs() * O.abs()).sum(-1, keepdim=True)
    E = P * (scl * (dOh.abs() @ vh.abs().transpose(2, 3)) + A)
    r.update(dq=_rows(dS @ kh), dk=_rows(dS.transpose(2, 3) @ qh), dv=_rows((P * scl).transpose(2, 3) @ dOh),
             env_dq=_rows(E @ kh.abs()), env_dk=_rows(E.transpose(2, 3) @ qh.abs()), env_dv=_rows((P * scl).transpose(2, 3) @ dOh.abs()))
    if rel_mode:
        def per_bucket(x):                                        # [B, H, Sq, Sk] -> [NB, H], summed over the biased entries
            out = torch.zeros(NB, H, dtype=torch.float64, device=dev)
            out.index_add_(0, bidx.reshape(-1), (x * region).sum(0).permute(1, 2, 0).reshape(Sq * Sk, H))
            return out
        r.update(dtable=per_bucket(dS), env_dtable=per_bucket(E), abs_dtable=per_bucket(dS.abs()),
                 n_dtable=per_bucket(torch.ones_like(dS)), reached=per_bucket(torch.ones_like(dS)) > 0)
    return r


def excess(got, ref, tol):
    """Elements outside the bound (NaN counts as outside)."""
    err = (got.double() - ref).abs()
    return ~(err <= tol)


def bound_fwd(r):
    return {"O": FWD_C * U * (r["envO"] + r["O"].abs()), "lse": LSE_C * (1.0 + r["smax"])}


def bound_bwd(r):
    b = {x: BWD_C * U * (r["env_" + x] + r[x].abs()) for x in ("dq", "dk", "dv")}
    if "dtable" in r:
        b["dtable"] = BWD_C * U * (r["env_dtable"] + r["dtable"].abs()) + r["n_dtable"] * 2.0 ** -24 * r["abs_dtable"]
    return b


def assert_bounds(got, r, bounds, what, kind):
    """Every element of every named result within its bound; records the worst ratio of the error to the bound's unit
    (u (env + |x|) for O and the gradients, 2^-16 (1 + max|s|) for lse)."""
    for name, tol in bounds.items():
        g = got[name]
        bad = excess(g, r[name], tol)
        if bool(bad.any()):
            i = tuple(bad.nonzero()[0].tolist())
            raise AssertionError(f"{what}: {name}: {int(bad.sum())} of {bad.numel()} elements outside the fp64 bound, e.g. at {i}: "
                                 f"got {g[i].item()}, want {r[name][i].item()}, bound {tol[i].item():.3g}")
        err = (g.double() - r[name]).abs()
        if name == "lse":
            key, unit = "lse", tol
        else:
            key, unit = kind, U * (r["env" + name if name == "O" else "env_" + name] + r[name].abs())
            if name == "dtable":
                err = (err - r["n_dtable"] * 2.0 ** -24 * r["abs_dtable"]).clamp_min(0)
        _WORST[key] = max(_WORST[key], (err / unit.clamp_min(1e-300)).max().item())


# ---------------------------------------------------------------------------------------------------------------------------
# inputs

def item_masks(B, Sk, value, seed):
    """[B, Sk] additive key masks, a different pattern for every batch element (the bits of b + 1 over keys 1..16 plus random
    keys beyond); key 0 is never masked."""
    g = torch.Generator().manual_seed(seed)
    m = torch.rand(B, Sk, generator=g) < 0.25
    nb = min(Sk - 1, 16)
    bits = ((torch.arange(B)[:, None] + 1) >> torch.arange(nb)[None, :]) & 1
    m[:, 1:1 + nb] = bits.bool()
    m[:, 0] = False
    return torch.where(m, value, 0.0).float()


class Case(NamedTuple):
    name: str
    H: int
    Sq: int
    Sk: int
    rel_mode: int = 0
    Lt: int = 0
    causal: int = 0
    mask: float = 0.0                # additive key-mask value (0: no mask)
    fwd: str = ""
    bwd: str = ""                    # "" = no backward (a query offset is forward-only)
    o_saved: bool = False
    q_off: int = 0
    size: str = "fixed"              # "tc", "persist" (B sized from the SM count) or "fixed"
    B: int = 9

    @property
    def grid(self):
        return 256 if max(self.Sq, self.Sk) > 64 else 64


TCF, TCB = "attn_enc_fwd_tc_kernel", "attn_enc_bwd_tc_kernel"
F48, B48, F28, B28 = "attn_fwd_kernel<4, 8, 1>", "attn_bwd_kernel<4, 8, 1>", "attn_fwd_kernel<2, 8, 1>", "attn_bwd_kernel<2, 8, 1>"
F124, B124, F184 = "attn_fwd_kernel<1, 2, 4>", "attn_bwd_kernel<1, 2, 4>", "attn_fwd_kernel<1, 8, 4>"
KSF, KSB, MTF, MTB = "attn_ks_fwd_kernel", "attn_ks_bwd_kernel", "attn_mt_fwd_kernel", "attn_mt_bwd_kernel"
ALL_KERNELS = {TCF, TCB, F48, B48, F28, B28, F124, B124, F184, KSF, KSB, MTF, MTB}


def _cases():
    c = []
    for S in (33, 56, 64):
        for Lt in (1, 20, 32):
            c.append(Case(f"tc_S{S}_Lt{Lt}", 12, S, S, 1, Lt, mask=-10000.0, fwd=TCF, bwd=TCB, size="tc"))
    c += [Case("st4_S56_H11", 11, 56, 56, 1, 20, mask=-10000.0, fwd=F48, bwd=B48, size="persist"),
          Case("st4_S33_H11", 11, 33, 33, 1, 20, mask=-10000.0, fwd=F48, bwd=B48),
          Case("st4_S64_Lt48", 12, 64, 64, 1, 48, mask=-10000.0, fwd=F48, bwd=B48, size="persist"),
          Case("st4_S56_nobias", 12, 56, 56, 0, 0, mask=-10000.0, fwd=F48, bwd=B48, size="persist"),
          Case("st2_S17", 12, 17, 17, 1, 10, mask=-10000.0, fwd=F28, bwd=B28),
          Case("st2_S32", 12, 32, 32, 1, 20, mask=-10000.0, fwd=F28, bwd=B28)]
    for T in (1, 5, 16):
        c.append(Case(f"dec_T{T}", 11, T, T, 2, 0, causal=1, fwd=F124, bwd=B124, B=7))
    c += [Case("st1_Sq8_Sk24", 12, 8, 24, 1, 20, mask=-10000.0, fwd=F184, bwd=B28),
          Case("st1_dec_rect", 12, 3, 40, 2, 0, causal=1, fwd=F184, q_off=37, B=7)]
    for Sq in (1, 5, 16):
        for Sk in (17, 58, 64):
            c.append(Case(f"ks_Sq{Sq}_Sk{Sk}", 12, Sq, Sk, 0, 0, mask=-1e9, fwd=KSF, bwd=KSB, o_saved=True))
    c += [Case("ks_Sq5_Sk17_st", 12, 5, 17, 0, 0, mask=-1e9, fwd=KSF, bwd=B28),
          Case("ks_Sq16_Sk58_st", 12, 16, 58, 0, 0, mask=-1e9, fwd=KSF, bwd=B48)]
    c += [Case("mt_65", 12, 65, 65, 1, 20, mask=-10000.0, fwd=MTF, bwd=MTB, o_saved=True, B=5),
          Case("mt_150_Lt23", 12, 150, 150, 1, 23, mask=-10000.0, fwd=MTF, bwd=MTB, o_saved=True, B=3),
          Case("mt_150_Lt64", 12, 150, 150, 1, 64, mask=-10000.0, fwd=MTF, bwd=MTB, o_saved=True, B=3),
          Case("mt_5_130", 12, 5, 130, 0, 0, mask=-1e9, fwd=MTF, bwd=MTB, o_saved=True, B=5),
          Case("mt_100_200", 12, 100, 200, 1, 30, mask=-10000.0, fwd=MTF, bwd=MTB, o_saved=True, B=2),
          Case("mt_70_33", 12, 70, 33, 1, 33, mask=-10000.0, fwd=MTF, bwd=MTB, o_saved=True, B=3),
          Case("mt_256", 12, 256, 256, 1, 20, mask=-10000.0, fwd=MTF, bwd=MTB, o_saved=True, B=2)]
    return c


CASES = _cases()
# one case per kernel path for the readout, layout and placement tests
PATHS = [c for c in CASES if c.name in ("tc_S56_Lt20", "st4_S56_H11", "st4_S56_nobias", "st2_S17", "dec_T5", "dec_T16", "st1_Sq8_Sk24",
                                        "ks_Sq5_Sk58", "ks_Sq16_Sk58_st", "mt_150_Lt23", "mt_5_130", "mt_70_33")]


def n_sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def batch_of(case):
    """tcgen05: items = B * H / 2 >= 3 x the forward grid (2 CTAs per SM) with a partial last wave in both kernels (backward
    grid: 1 CTA per SM); persistent <4,8,1>: problems B * H >= 3 x its grid (3 CTAs per SM) with a partial last wave."""
    n = n_sms()
    if case.size == "tc":
        B = -(-3 * 2 * n * 2 // case.H)
        while (B * case.H // 2) % (2 * n) == 0 or (B * case.H // 2) % n == 0:
            B += 1
        return B
    if case.size == "persist":
        B = -(-3 * 3 * n // case.H)
        while (B * case.H) % (3 * n) == 0:
            B += 1
        return B
    return case.B


def make_inputs(case, B, seed, device=None):
    device = device or DEV
    g = torch.Generator(device="cpu").manual_seed(seed)
    H = case.H

    def rnd(*shape, scale=1.0):
        return (torch.randn(*shape, generator=g) * scale).bfloat16().to(device)

    x = dict(q=rnd(B * case.Sq, H * 64, scale=0.3), k=rnd(B * case.Sk, H * 64, scale=0.3), v=rnd(B * case.Sk, H * 64),
             dO=rnd(B * case.Sq, H * 64))
    kw = dict(rel_mode=case.rel_mode, Lt=case.Lt, causal=case.causal)
    if case.rel_mode:
        kw.update(table=(torch.randn(NB, H, generator=g) * 0.5).to(device), bucket=rel_bucket_table(case.rel_mode == 1))
    if case.mask:
        kw["keymask"] = item_masks(B, case.Sk, case.mask, seed).to(device)
    return x, kw


def kernel_kw(kw):
    """reference keyword arguments -> the C-ABI wrappers' (rel_table, rel_bucket, ...)"""
    out = dict(rel_mode=kw["rel_mode"], Lt=kw["Lt"], causal=kw["causal"], keymask=kw.get("keymask"))
    if kw.get("table") is not None:
        out.update(rel_table=kw["table"], rel_bucket=kw["bucket"])
    return out


def run_fwd(case, B, x, kw, drop, lse=True, q_off=None):
    o = torch.full((B * case.Sq, case.H * 64), float("nan"), dtype=torch.bfloat16, device=DEV)
    l = torch.full((B, case.H, case.Sq), float("nan"), device=DEV) if lse else None
    cabi.attention_fwd_ex(x["q"], x["k"], x["v"], o, l, B, case.H, case.Sq, case.Sk, drop=drop,
                          q_off=case.q_off if q_off is None else q_off, **kernel_kw(kw))
    return o, l


def run_bwd(case, B, x, kw, drop, lse, o, dtab=None):
    dq = torch.full_like(x["q"], float("nan"))
    dk, dv = torch.full_like(x["k"], float("nan")), torch.full_like(x["v"], float("nan"))
    if dtab is None and case.rel_mode:
        dtab = torch.zeros(NB, case.H, device=DEV)
    cabi.attention_bwd_ex(x["q"], x["k"], x["v"], x["dO"], lse, dq, dk, dv, dtab, B, case.H, case.Sq, case.Sk,
                          o_saved=o if case.o_saved else None, drop=drop, **kernel_kw(kw))
    return dict(dq=dq, dk=dk, dv=dv, dtable=dtab)


def kernels_run(fn):
    """Names of the attention kernels launched by fn() (torch.profiler, CUDA activity)."""
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = set()
    for e in prof.events():
        m = re.search(r"(attn_\w+(?:<[^>]*>)?)", e.name.replace("(int)", ""))
        if m:
            names.add(m.group(1))
    return names


# ---------------------------------------------------------------------------------------------------------------------------
# CPU: the reference itself, the dropout restatement and the teeth of the bound

def test_reference_matches_oracle_t5attention_in_double():
    from helpers import O
    cfg = O.VLT5Config()
    H = cfg.num_heads
    g = torch.Generator().manual_seed(3)
    for is_dec in (False, True):
        B, S, Lt = 3, (12 if is_dec else 40), 17
        att = O.T5Attention(cfg, is_dec, True).double().eval()
        with torch.no_grad():
            for lin in (att.q, att.k, att.v):
                lin.weight.copy_(torch.randn(H * 64, cfg.d_model, generator=g, dtype=torch.float64) * 0.04)
            att.o.weight.copy_(torch.eye(cfg.d_model, dtype=torch.float64))
            att.relative_attention_bias.weight.copy_(torch.randn(NB, H, generator=g, dtype=torch.float64) * 0.5)
        hid = torch.randn(B, S, cfg.d_model, generator=g, dtype=torch.float64)
        table = att.relative_attention_bias.weight.detach()
        if is_dec:
            bias = att.compute_bias(S, S) - 10000.0 * (1.0 - torch.tril(torch.ones(S, S, dtype=torch.float64)))[None, None]
            kw = dict(table=table, bucket=rel_bucket_table(False), rel_mode=2, causal=1)
        else:
            km = item_masks(B, S, -10000.0, 5).double()
            bias = torch.zeros(1, H, S, S, dtype=torch.float64)
            bias[:, :, :Lt, :Lt] = att.compute_bias(Lt, Lt)
            bias = bias + km[:, None, None, :]
            kw = dict(table=table, bucket=rel_bucket_table(True), rel_mode=1, Lt=Lt, keymask=km)
        with torch.no_grad():
            want = att(hid, bias)
            q, k, v = (lin(hid).reshape(B * S, H * 64) for lin in (att.q, att.k, att.v))
        got = reference(q, k, v, B, H, S, S, **kw)["O"]
        # the oracle takes its softmax in fp32 (as HF T5Attention does), so the agreement is to fp32 rounding, far below bf16
        torch.testing.assert_close(got, want.reshape(B * S, -1), rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("grid", [64, 256])
def test_dropout_restatement_matches_the_gemm_index(grid):
    B, H = 3, 5
    drop = dropout_params(0.1)
    sc = drop_scale(B, H, grid, grid, grid, drop, "cpu")
    want = cabi.dropout_scale_host(B * H * grid, grid, *drop, device="cpu").double().view(B, H, grid, grid)
    assert torch.equal(sc, want)
    dropped = (sc == 0).double().mean().item()
    assert abs(dropped - 0.1) < 5e-3, dropped
    kept = sc[sc != 0]
    assert bool((kept == drop[1]).all())


TEETH_FORMS = {
    "enc": (Case("enc", 4, 40, 40, 1, 20, mask=-10000.0), ("bias_bucket", "mask_drop", "drop_lanes", "head_k", "lse_shift")),
    "dec_self": (Case("dec_self", 4, 12, 12, 2, 0, causal=1), ("bias_bucket", "causal_off", "drop_lanes", "head_k", "lse_shift")),
    "cross": (Case("cross", 4, 5, 40, 0, 0, mask=-1e9), ("mask_drop", "drop_lanes", "head_k", "lse_shift")),
    "multi_tile": (Case("multi_tile", 4, 80, 80, 1, 23, mask=-10000.0),
                   ("bias_bucket", "mask_drop", "drop_lanes", "drop_grid", "head_k", "lse_shift")),
}


@pytest.mark.parametrize("form", list(TEETH_FORMS))
def test_bound_catches_each_mutation(form):
    """A reference with one deliberate bug, rounded the way the kernels store their results, must leave the bound somewhere —
    forward (O, lse) and backward (dq, dk, dv, dtable) separately."""
    case, muts = TEETH_FORMS[form]
    B = 3
    x, kw = make_inputs(case, B, 11, device="cpu")
    drop = dropout_params(0.1)
    args = dict(drop=drop, grid=case.grid, dO=x["dO"], **kw)
    r = reference(x["q"], x["k"], x["v"], B, case.H, case.Sq, case.Sk, **args)
    bf, bb = bound_fwd(r), bound_bwd(r)
    for name, tol in {**bf, **bb}.items():                       # the exact values, rounded as stored, pass
        got = r[name].float() if name in ("lse", "dtable") else r[name].bfloat16()
        assert not bool(excess(got, r[name], tol).any()), (form, name)
    for mut in muts + ("D_undropped",):
        m = reference(x["q"], x["k"], x["v"], B, case.H, case.Sq, case.Sk, mut=(mut,), **args)

        def caught(bounds):
            return [n for n, tol in bounds.items()
                    if bool(excess(m[n].float() if n in ("lse", "dtable") else m[n].bfloat16(), r[n], tol).any())]
        if mut != "D_undropped":
            assert caught(bf), f"{form}: forward bound misses {mut}"
        assert caught(bb), f"{form}: backward bound misses {mut}"


def test_cases_cover_every_kernel_instantiation():
    assert {c.fwd for c in CASES} | {c.bwd for c in CASES if c.bwd} == ALL_KERNELS
    assert len(ALL_KERNELS) == 13
    assert {c.fwd for c in PATHS} | {c.bwd for c in PATHS if c.bwd} == ALL_KERNELS


# ---------------------------------------------------------------------------------------------------------------------------
# GPU

@pytest.mark.gpu
@pytest.mark.parametrize("p", [0.0, 0.1])
@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_dispatch_row_against_fp64(case, p):
    B = batch_of(case)
    x, kw = make_inputs(case, B, sum(map(ord, case.name)))
    drop = dropout_params(p)
    out = {}

    def fwd():
        out["o"], out["lse"] = run_fwd(case, B, x, kw, drop)
    if p == 0:
        assert kernels_run(fwd) == {case.fwd}, case.name
    else:
        fwd()
    r = reference(x["q"], x["k"], x["v"], B, case.H, case.Sq, case.Sk, q_off=case.q_off, drop=drop, grid=case.grid,
                  dO=x["dO"] if case.bwd else None, **kw)
    assert_bounds({"O": out["o"], "lse": out["lse"]}, r, bound_fwd(r), case.name, "fwd")
    if not case.bwd:
        return

    def bwd():
        out.update(run_bwd(case, B, x, kw, drop, out["lse"], out["o"]))
    if p == 0:
        assert kernels_run(bwd) == {case.bwd}, case.name
    else:
        bwd()
    assert_bounds(out, r, bound_bwd(r), case.name, "bwd")


def _identity_blocks(B, S, H, n):
    """[B*S, H*64] bf16 with X[b, j, h, c] = 1 iff j == 64 n + c (block n of the identity, the same for every head)."""
    X = torch.zeros(B, S, H, 64, device=DEV)
    j = torch.arange(64 * n, min(S, 64 * n + 64), device=DEV)
    X[:, j, :, j - 64 * n] = 1.0
    return X.reshape(B * S, H * 64).bfloat16()


@pytest.mark.gpu
@pytest.mark.parametrize("case", PATHS, ids=[c.name for c in PATHS])
def test_probability_readout(case):
    """With V = I on one 64-key block O is P^ itself (backward: dO = I on one 64-query block gives dV = P^^T): every entry within
    2^-8 P^64 per bf16 rounding the kernel applies to it, and the dropped entries are exactly the host mask's wherever
    P64 > 2^-20. The single-tile kernels normalise P in fp32 before its one rounding (the product with 1 and the store of a
    bf16 value are exact); the tcgen05, key-split and multi-tile forwards round the unnormalised exponentials for the P V
    product and round again when the normalised O is stored. Every backward rounds P^ once."""
    B = min(batch_of(case), 6)
    x, kw = make_inputs(case, B, 7)
    drop = dropout_params(0.1)
    H, Sq, Sk = case.H, case.Sq, case.Sk
    r = reference(x["q"], x["k"], x["v"], B, H, Sq, Sk, q_off=case.q_off, drop=drop, grid=case.grid, **kw)
    Ph, P = r["Ph"], r["P"]
    live = P > 2.0 ** -20

    def check(got, want, livem, dropm, what, roundings=1):      # got / want [B, H, rows, cols]
        bad = ~((got.double() - want).abs() <= roundings * 2.0 ** -8 * want)
        assert not bool(bad.any()), f"{case.name} {what}: {int(bad.sum())} entries off, e.g. {bad.nonzero()[0].tolist()}"
        assert torch.equal((got == 0) & livem, dropm & livem), f"{case.name} {what}: dropped set differs from the host mask"

    for n in range(-(-Sk // 64)):
        xv = dict(x, v=_identity_blocks(B, Sk, H, n))
        o, _ = run_fwd(case, B, xv, kw, drop)
        cols = min(64, Sk - 64 * n)
        got = o.view(B, Sq, H, 64).transpose(1, 2).float()
        sl = slice(64 * n, 64 * n + cols)
        check(got[..., :cols], Ph[..., sl], live[..., sl], (r["scale"] == 0)[..., sl], f"forward block {n}",
              roundings=2 if case.fwd in (TCF, KSF, MTF) else 1)
        assert bool((got[..., cols:] == 0).all())
    if not case.bwd:
        return
    lse64 = r["lse"].float()
    o, _ = run_fwd(case, B, x, kw, drop)
    for n in range(-(-Sq // 64)):
        xd = dict(x, dO=_identity_blocks(B, Sq, H, n))
        g = run_bwd(case, B, xd, kw, drop, lse64, o)
        rows = min(64, Sq - 64 * n)
        got = g["dv"].view(B, Sk, H, 64).transpose(1, 2).float()    # [B, H, Sk, 64]: column c = query 64 n + c
        sl = slice(64 * n, 64 * n + rows)
        check(got[..., :rows], Ph[:, :, sl].transpose(2, 3), live[:, :, sl].transpose(2, 3),
              (r["scale"] == 0)[:, :, sl].transpose(2, 3), f"backward block {n}")


def _nan_buf(rows, cols):
    return torch.full((rows, cols), float("nan"), dtype=torch.bfloat16, device=DEV)


def _bits(t):
    return t.view(torch.int16) if t.dtype == torch.bfloat16 else t.view(torch.int32)


@pytest.mark.gpu
@pytest.mark.parametrize("pitch", [2304, 2312])
@pytest.mark.parametrize("case", PATHS, ids=[c.name for c in PATHS])
def test_engine_layouts(case, pitch):
    """q / k / v read in place from a packed [rows, pitch] QKV buffer (cross-attention: K / V from a [rows, 18432] buffer of 12
    layers), dq / dk / dv written interleaved into one packed buffer, O and lse inside sentinel borders, a pre-filled bias-table
    gradient: the results equal the dense run bit for bit, every output element is written, nothing outside the windows
    changes, and table entries of buckets the problem never reaches keep their pre-fill."""
    B = min(batch_of(case), 6)
    H, Sq, Sk, W = case.H, case.Sq, case.Sk, case.H * 64
    x, kw = make_inputs(case, B, 21)
    drop = dropout_params(0.1)
    o_d, l_d = run_fwd(case, B, x, kw, drop)
    self_attn = Sq == Sk
    if self_attn:
        qkv = _nan_buf(B * Sq + 3, pitch)
        q, k, v = qkv[:B * Sq, 0:W], qkv[:B * Sq, 768:768 + W], qkv[:B * Sq, 1536:1536 + W]
        kvbuf = qkv
    else:
        qbuf = _nan_buf(B * Sq + 3, pitch)
        q = qbuf[:B * Sq, 0:W]
        kvbuf = _nan_buf(B * Sk + 3, 18432)
        k, v = kvbuf[:B * Sk, 5 * 1536:5 * 1536 + W], kvbuf[:B * Sk, 5 * 1536 + 768:5 * 1536 + 768 + W]
    q.copy_(x["q"]); k.copy_(x["k"]); v.copy_(x["v"])
    SENT = 3.25
    obuf = torch.full((B * Sq + 4, W + 16), SENT, dtype=torch.bfloat16, device=DEV)
    o = obuf[2:2 + B * Sq, 8:8 + W]
    lbuf = torch.full((B * H * Sq + 8,), SENT, device=DEV)
    lse = lbuf[4:4 + B * H * Sq].view(B, H, Sq)
    obuf0, lbuf0 = obuf.clone(), lbuf.clone()
    cabi.attention_fwd_ex(q, k, v, o, lse, B, H, Sq, Sk, drop=drop, q_off=case.q_off, **kernel_kw(kw))
    assert torch.equal(_bits(o), _bits(o_d)) and torch.equal(_bits(lse), _bits(l_d)), case.name
    inner = torch.zeros_like(obuf, dtype=torch.bool)
    inner[2:2 + B * Sq, 8:8 + W] = True
    assert torch.equal(_bits(obuf)[~inner], _bits(obuf0)[~inner]), "O written outside its window"
    linner = torch.zeros_like(lbuf, dtype=torch.bool)
    linner[4:4 + B * H * Sq] = True
    assert torch.equal(_bits(lbuf)[~linner], _bits(lbuf0)[~linner]), "lse written outside its window"
    if not case.bwd:
        return
    g_d = run_bwd(case, B, x, kw, drop, l_d, o_d)
    if self_attn:
        gbuf = _nan_buf(B * Sq + 2, 2312)
        dq, dk, dv = gbuf[:B * Sq, 0:W], gbuf[:B * Sq, 768:768 + W], gbuf[:B * Sq, 1536:1536 + W]
        bufs = [(gbuf, [(0, B * Sq, 0, W), (0, B * Sq, 768, 768 + W), (0, B * Sq, 1536, 1536 + W)])]
    else:
        qg = _nan_buf(B * Sq + 2, pitch)
        kvg = _nan_buf(B * Sk + 2, 18432)
        dq = qg[:B * Sq, 0:W]
        dk, dv = kvg[:B * Sk, 5 * 1536:5 * 1536 + W], kvg[:B * Sk, 5 * 1536 + 768:5 * 1536 + 768 + W]
        bufs = [(qg, [(0, B * Sq, 0, W)]), (kvg, [(0, B * Sk, 5 * 1536, 5 * 1536 + W), (0, B * Sk, 5 * 1536 + 768, 5 * 1536 + 768 + W)])]
    before = [b.clone() for b, _ in bufs]
    dO = _nan_buf(B * Sq + 2, pitch)[:B * Sq, 0:W]
    dO.copy_(x["dO"])
    osv = None
    if case.o_saved:
        osv = _nan_buf(B * Sq + 2, pitch)[:B * Sq, 0:W]
        osv.copy_(o_d)
    g = torch.Generator(device="cpu").manual_seed(5)
    prefill = torch.randn(NB, H, generator=g).to(DEV)
    dtab = prefill.clone()
    cabi.attention_bwd_ex(q, k, v, dO, l_d, dq, dk, dv, dtab, B, H, Sq, Sk, o_saved=osv, drop=drop, **kernel_kw(kw))
    for got, want in ((dq, g_d["dq"]), (dk, g_d["dk"]), (dv, g_d["dv"])):
        assert torch.equal(_bits(got), _bits(want)), case.name
        assert not bool(got.isnan().any()), "output element not written"
    for (buf, wins), b0 in zip(bufs, before):
        outside = torch.ones_like(buf, dtype=torch.bool)
        for r0, r1, c0, c1 in wins:
            outside[r0:r1, c0:c1] = False
        assert torch.equal(_bits(buf)[outside], _bits(b0)[outside]), "gradient written outside its window"
    if case.rel_mode:
        r = reference(x["q"], x["k"], x["v"], B, H, Sq, Sk, drop=drop, grid=case.grid, dO=x["dO"], **kw)
        reached = r["reached"]
        tol = bound_bwd(r)["dtable"] + 2.0 ** -23 * prefill.abs().double()
        assert not bool(excess(dtab - prefill, r["dtable"], tol)[reached].any())
    else:
        reached = torch.zeros(NB, H, dtype=torch.bool, device=DEV)
    assert torch.equal(_bits(dtab)[~reached], _bits(prefill)[~reached]), "bias-table entries of unreached buckets changed"


@pytest.mark.gpu
def test_kv_cache_decode_form_every_step():
    """The decode step's self-attention as decode.cu calls it: one query at position t against the t + 1 cached keys of a
    [B, 64, 2304] cache whose rows after t are NaN, q_off = t, decoder bias, causal, no lse. Every t in 0..62 against row t of
    the fp64 reference; for t <= 15 (both forms run attn_fwd_kernel<1, 2, 4>) bit for bit against row t of the training form."""
    B, H = 7, 12
    case = Case("dec", H, 63, 63, 2, 0, causal=1)
    x, kw = make_inputs(case, B, 31)
    r = reference(x["q"], x["k"], x["v"], B, H, 63, 63, **kw)
    tol = bound_fwd(r)["O"].view(B, 63, H * 64)
    ref = r["O"].view(B, 63, H * 64)
    cache = _nan_buf(B * 64, 2304).view(B, 64, 2304)
    qs, ks, vs = (x[n].view(B, 63, H * 64) for n in ("q", "k", "v"))
    bs = 64 * 2304
    for t in range(63):
        cache[:, t, 0:768] = qs[:, t]
        cache[:, t, 768:1536] = ks[:, t]
        cache[:, t, 1536:2304] = vs[:, t]
        o = torch.full((B, H * 64), float("nan"), dtype=torch.bfloat16, device=DEV)
        names = kernels_run(lambda: cabi.attention_fwd_ex(cache[:, t, 0:768], cache[:, 0, 768:1536], cache[:, 0, 1536:2304], o, None,
                                                          B, H, 1, t + 1, bstrides=(bs, bs, bs, 0), q_off=t, ld=(2304, 2304, 2304, 768),
                                                          **kernel_kw(kw))) if t in (0, 15, 16, 62) else None
        if names is None:
            cabi.attention_fwd_ex(cache[:, t, 0:768], cache[:, 0, 768:1536], cache[:, 0, 1536:2304], o, None, B, H, 1, t + 1,
                                  bstrides=(bs, bs, bs, 0), q_off=t, ld=(2304, 2304, 2304, 768), **kernel_kw(kw))
        else:
            assert names == {F124 if t < 16 else F184}, (t, names)
        bad = excess(o, ref[:, t], tol[:, t])
        assert not bool(bad.any()), f"t={t}: {int(bad.sum())} elements outside the fp64 bound"
        if t <= 15:
            tc = Case("dec", H, t + 1, t + 1, 2, 0, causal=1)
            xt = {n: x[n].view(B, 63, -1)[:, :t + 1].reshape(B * (t + 1), -1).contiguous() for n in ("q", "k", "v")}
            ot, _ = run_fwd(tc, B, xt, kw, (0, 1.0, 0))
            assert torch.equal(_bits(o), _bits(ot.view(B, t + 1, -1)[:, t])), f"t={t}: decode form differs from the training form"


@pytest.mark.gpu
@pytest.mark.parametrize("Sk", [17, 58, 64])
def test_kv_cache_decode_cross_attention(Sk):
    """Decode-step cross-attention: one query against K / V of a [B * Sk, 18432] buffer (12 layers), -1e9 on text pads; O is
    the same bit for bit with and without lse."""
    B, H = 7, 12
    case = Case("xdec", H, 1, Sk, 0, 0, mask=-1e9)
    x, kw = make_inputs(case, B, 41 + Sk)
    kv = _nan_buf(B * Sk + 2, 18432)
    k, v = kv[:B * Sk, 3 * 1536:3 * 1536 + 768], kv[:B * Sk, 3 * 1536 + 768:3 * 1536 + 1536]
    k.copy_(x["k"]); v.copy_(x["v"])
    outs = []
    for want_lse in (False, True):
        o = torch.full((B, 768), float("nan"), dtype=torch.bfloat16, device=DEV)
        lse = torch.full((B, H, 1), float("nan"), device=DEV) if want_lse else None
        names = kernels_run(lambda: cabi.attention_fwd_ex(x["q"], k, v, o, lse, B, H, 1, Sk, **kernel_kw(kw)))
        assert names == {KSF}
        outs.append(o)
    assert torch.equal(_bits(outs[0]), _bits(outs[1]))
    r = reference(x["q"], x["k"], x["v"], B, H, 1, Sk, **kw)
    assert not bool(excess(outs[0], r["O"], bound_fwd(r)["O"]).any())


@pytest.mark.gpu
@pytest.mark.parametrize("case", PATHS, ids=[c.name for c in PATHS])
def test_item_gives_the_same_bits_alone_and_in_the_persistent_launch(case):
    """Dropout off: batch element b run alone (B = 1, pointers offset to the item) equals its slice of the full launch bit for
    bit, forward and backward (not the bias-table gradient, whose atomics have no fixed order)."""
    B = batch_of(case)
    H, Sq, Sk = case.H, case.Sq, case.Sk
    x, kw = make_inputs(case, B, 51)
    drop = (0, 1.0, 0)
    o, lse = run_fwd(case, B, x, kw, drop)
    g = run_bwd(case, B, x, kw, drop, lse, o) if case.bwd else None
    for b in sorted({0, B // 2, B - 1}):
        xb = {n: x[n][b * (Sk if n in ("k", "v") else Sq):(b + 1) * (Sk if n in ("k", "v") else Sq)] for n in x}
        kwb = dict(kw)
        if kw.get("keymask") is not None:
            kwb["keymask"] = kw["keymask"][b:b + 1]
        ob, lb = run_fwd(case, 1, xb, kwb, drop)
        assert torch.equal(_bits(ob), _bits(o[b * Sq:(b + 1) * Sq])), f"{case.name}: O of item {b}"
        assert torch.equal(_bits(lb), _bits(lse[b:b + 1])), f"{case.name}: lse of item {b}"
        if g is not None:
            gb = run_bwd(case, 1, xb, kwb, drop, lse[b:b + 1].contiguous(), o[b * Sq:(b + 1) * Sq])
            for n, rows in (("dq", Sq), ("dk", Sk), ("dv", Sk)):
                assert torch.equal(_bits(gb[n]), _bits(g[n][b * rows:(b + 1) * rows])), f"{case.name}: {n} of item {b}"


@pytest.mark.gpu
def test_invalid_calls_are_rejected_without_a_launch():
    B, H = 2, 12
    x, kw = make_inputs(Case("r", H, 64, 64), B, 61)
    q, k, v = x["q"], x["k"], x["v"]
    bucket = rel_bucket_table(True)
    table = torch.zeros(NB, H, device=DEV)
    big = (torch.randn(B * 130, H * 64, device=DEV) * 0.3).bfloat16()
    o = torch.empty(B * 130, H * 64, dtype=torch.bfloat16, device=DEV)
    lse = torch.empty(B * H * 130, device=DEV)
    dq, dk, dv = torch.empty_like(big), torch.empty_like(big), torch.empty_like(big)
    bad_bucket = bucket.clone()
    bad_bucket[70] = 64
    neg_bucket = bucket.clone()
    neg_bucket[3] = -1

    def fwd(Sq, Sk, qq=q, kk=k, vv=v, **a):
        return lambda: cabi.attention_fwd_ex(qq, kk, vv, o, lse, B, H, Sq, Sk, **a)

    def bwd(Sq, Sk, o_saved=None, lse_=lse, dq_=dq, **a):
        return lambda: cabi.attention_bwd_ex(big, big, big, big, lse_, dq_, dk, dv, None, B, H, Sq, Sk, o_saved=o_saved, **a)

    calls = {
        "Sq = 0": fwd(0, 16),
        "Sk = 257": fwd(16, 257, kk=big, vv=big),
        "causal beyond 64": fwd(65, 65, qq=big, kk=big, vv=big, causal=1),
        "rel_mode 2 beyond 64": fwd(65, 65, qq=big, kk=big, vv=big, rel_mode=2, rel_table=table, rel_bucket=bucket),
        "bias corner beyond 64": fwd(100, 100, qq=big, kk=big, vv=big, rel_mode=1, Lt=65, rel_table=table, rel_bucket=bucket),
        "q_off on a multi-tile problem": fwd(5, 130, kk=big, vv=big, q_off=1),
        "pitch not a multiple of 8": fwd(16, 16, ld=(772, None, None, None)),
        "rel_mode without table": fwd(16, 16, rel_mode=1, Lt=8, rel_bucket=bucket),
        "rel_mode without buckets": fwd(16, 16, rel_mode=2, rel_table=table),
        "bucket out of range": fwd(16, 16, rel_mode=2, rel_table=table, rel_bucket=bad_bucket),
        "negative bucket": fwd(16, 16, rel_mode=1, Lt=8, rel_table=table, rel_bucket=neg_bucket),
        "negative q_off": fwd(1, 16, q_off=-1),
        "q_off + Sq > 64": fwd(2, 40, q_off=63, rel_mode=2, rel_table=table, rel_bucket=bucket, causal=1),
        "q_off + Sq > 64 without bias": fwd(16, 16, q_off=49),
        "multi-tile backward without o_saved": bwd(130, 130),
        "backward without lse": bwd(16, 16, lse_=None),
        "backward without dq": bwd(16, 16, dq_=None),
    }
    torch.cuda.synchronize()
    for what, call in calls.items():
        n0 = cabi.launch_count()
        with pytest.raises(VqaclError):
            call()
        assert cabi.launch_count() == n0, f"{what}: launched a kernel"
    # the largest accepted query offset still runs
    o1 = torch.empty(B, H * 64, dtype=torch.bfloat16, device=DEV)
    cabi.attention_fwd_ex(q[:B], k, v, o1, None, B, H, 1, 64, q_off=63, rel_mode=2, rel_table=table, rel_bucket=bucket, causal=1,
                          bstrides=(64 * H * 64, 64 * H * 64, 64 * H * 64, 0))
    torch.cuda.synchronize()
    assert not bool(o1.isnan().any())
