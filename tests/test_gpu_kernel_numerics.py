"""Numerics of the sm_100a attention kernels against a float64 oracle, row by row.

Every kernel result is compared with a float64 attention computed on the rounded inputs (the *oracle*) and judged
against a *same-precision emulation* that rounds where the kernels round.  A row passes when

    err_kernel <= C_EMU * err_emulation + ulp_dtype(max|ref_row|) + TINY * max|ref|

where a row is one (query row, head) of out / dQ, or one (key row, kv head) of dK / dV.  A global tolerance lets a
wrong mask on late rows (whose gradients are small) or a skipped rescale on a few rows pass; a per-row budget tied
to the rounding the kernel must do does not.

The CPU tests at the top check the checker itself: a kernel-like model (fp32 accumulation, lagging row max with the
forward kernel's 2^8 rule, P and dS rounded to the model dtype) must pass, and every one of a list of small kernel
bugs (mutants) must be flagged on the same inputs the GPU tests feed the kernels.
"""
import math

import pytest
import torch

from ring_flash_attn_b200.ops import plan as P
from ring_flash_attn_b200.parallel import layouts

# ---------------------------------------------------------------------------------------------------------------
# Error budget (fixed before any kernel result was seen).
#
# C_EMU: the kernels round P (forward and backward), dS and the outputs at the same points as the emulation, so
# their error against the oracle is a second draw of the same rounding noise plus fp32 accumulation error (about
# D * 2^-24 relative, far below one bf16 / fp16 rounding).  The forward additionally keeps P relative to a lagging
# maximum (P up to 2^8 instead of <= 1), which changes which way each element rounds but not the size of the
# rounding.  Beyond the ULP slack below, the kernel-like model of this file needs a factor of at most 2.0 over 40
# seeds of every input family (random, mask-edge probes, rescale stress; the worst are probe gradients, where few
# terms dominate a row); 4 leaves room for a second draw without hiding an O(1) error.
# ULP term, one unit of the MODEL dtype at the row's largest magnitude: a row dominated by one or two terms (a
# peaked softmax, a key that few queries see) carries one or two roundings of P or dS, and either draw may happen to
# be near zero, so the ratio alone is not a fair bound there; one model-dtype unit is what such a rounding can cost.
# The same term covers outputs rounded to the model dtype that land one unit apart.
# TINY: rows whose reference is exactly zero (no visible key, a key no query sees) must stay zero up to fp32 noise.
C_EMU = 4.0
TINY = 2.0 ** -20
# lse: the kernels compute lse = (m + log2 l) * ln 2 in fp32 from fp32 scores, with ex2.approx / lg2.approx.  Per
# row, with A = scale * max over visible keys of sum_d |q_d k_d|:
#   scores  (fp32 GEMM over D products + the scaling FMA):     (D + 2) * 2^-24 * A
#   l       (<= 66 sequential fp32 adds per key tile, one more add and one rescale per tile): (66 + 2 T) * 2^-24
#   ex2.approx relative error of every P:                      2^-22
#   lg2.approx absolute error (log2 units, times ln 2):        2^-22 * ln 2
#   the final add and multiply in fp32:                        3 * 2^-24 * |lse|
# and LSE_SAFETY covers the second-order terms and accumulators that truncate instead of rounding.
LSE_SAFETY = 2.0
EPS32 = 2.0 ** -24

MANTISSA = {torch.bfloat16: 7, torch.float16: 10, torch.float32: 23, torch.float64: 52}
MIN_EXP = {torch.bfloat16: -126, torch.float16: -14, torch.float32: -126, torch.float64: -1022}
LOG2E = 1.4426950408889634
RESCALE_THRESHOLD = 8.0  # csrc/attn_fwd_sm100.cu: kRescaleThreshold (log2 units)
KEY_TILE = 128


def ulp(x: torch.Tensor, dtype) -> torch.Tensor:
    """One unit in the last place of ``dtype`` at magnitude ``x`` (subnormal spacing below the normal range)."""
    e = torch.floor(torch.log2(x.double().clamp_min(1e-300))).clamp_min(MIN_EXP[dtype])
    return torch.exp2(e - MANTISSA[dtype])


# ---------------------------------------------------------------------------------------------------------------
# masks
# ---------------------------------------------------------------------------------------------------------------

def seg_vis(sq, k_rows, kv_row0, kv_len, diag, lo, device="cpu"):
    """Key row j of the K tensor is visible to query i iff it lies in the segment [kv_row0, kv_row0 + kv_len) and,
    as segment key jj = j - kv_row0, satisfies i + lo <= jj <= i + diag (None = unbounded)."""
    i = torch.arange(sq, device=device).unsqueeze(1)
    jj = torch.arange(k_rows, device=device).unsqueeze(0) - kv_row0
    m = (jj >= 0) & (jj < kv_len)
    if diag is not None:
        m = m & (jj <= i + diag)
    if lo is not None:
        m = m & (jj >= i + lo)
    return m


def pos_vis(pos_q, doc_q, pos_k, doc_k, left=None):
    """Causal (optionally windowed) visibility by global position inside a document."""
    m = (doc_q.unsqueeze(1) == doc_k.unsqueeze(0)) & (pos_k.unsqueeze(0) <= pos_q.unsqueeze(1))
    if left is not None:
        m = m & (pos_k.unsqueeze(0) >= pos_q.unsqueeze(1) - left)
    return m


# ---------------------------------------------------------------------------------------------------------------
# float64 oracle and same-precision emulation (explicit formulas, on the inputs' device)
# ---------------------------------------------------------------------------------------------------------------

def _rnd(x, dtype):
    return x if dtype is None else x.to(dtype).double()


def _expand(t, g):
    return t.repeat_interleave(g, dim=1)


def fwd64(q, k, v, scale, vis, emu=None):
    """out (sq, hq, d), lse (hq, sq).  ``emu`` = model dtype: P rounded before PV (l from the unrounded P) and the
    output rounded, as in the forward kernel.  Rows without a visible key give out = 0, lse = -inf."""
    g = q.shape[1] // k.shape[1]
    qd, kd, vd = q.double(), _expand(k.double(), g), _expand(v.double(), g)
    s = torch.einsum("ihd,jhd->hij", qd, kd) * scale
    s = s.masked_fill(~vis, float("-inf"))
    m = s.amax(-1, keepdim=True)
    m = torch.where(torch.isinf(m), torch.zeros_like(m), m)
    p = torch.exp(s - m)
    l = p.sum(-1)
    o = torch.einsum("hij,jhd->ihd", _rnd(p, emu), vd)
    o = o / torch.where(l > 0, l, torch.ones_like(l)).t().unsqueeze(-1)
    lse = torch.where(l > 0, m.squeeze(-1) + torch.log(l.clamp_min(1e-300)), torch.full_like(l, float("-inf")))
    return _rnd(o, emu), lse


def bwd64(q, k, v, dout, scale, vis, lse, delta, emu=None):
    """Wide (unrounded) dq (sq, hq, d), dk / dv (sk, hkv, d) from the given lse / delta (hq, sq).  ``emu``: P and
    dS = P * (dP - delta) * scale rounded to the model dtype before their GEMMs, as in the backward kernel."""
    hkv = k.shape[1]
    g = q.shape[1] // hkv
    qd, kd, vd, dod = q.double(), _expand(k.double(), g), _expand(v.double(), g), dout.double()
    lse, delta = lse.double(), delta.double()
    s = torch.einsum("ihd,jhd->hij", qd, kd) * scale
    lse_ = torch.where(torch.isinf(lse), torch.full_like(lse, float("inf")), lse)
    p = torch.exp(s - lse_.unsqueeze(-1)).masked_fill(~vis, 0.0)
    dv = torch.einsum("hij,ihd->jhd", _rnd(p, emu), dod)
    dp = torch.einsum("ihd,jhd->hij", dod, vd)
    ds = _rnd(p * (dp - delta.unsqueeze(-1)) * scale, emu)
    dq = torch.einsum("hij,jhd->ihd", ds, kd)
    dk = torch.einsum("hij,ihd->jhd", ds, qd)
    sk, d = k.shape[0], k.shape[2]
    return dq, dk.view(sk, hkv, g, d).sum(2), dv.view(sk, hkv, g, d).sum(2)


def grad_floor(q, k, v, dout, scale, vis, lse, delta):
    """fp32 floor of the dQ / dK rows, (sq, hq) and (sk, hkv).  dS = P (dP - delta) scale cancels where dP ~ delta (a
    row dominated by one key gives dS ~ 0), so next to the rounding of dS its error has an absolute part: dP is an
    fp32 sum of D products and delta arrives rounded to fp32, (D + 2) 2^-24 (sum_d |dO_d V_d| + |delta|) per element.
    It is carried through the dQ = dS K and dK = dS^T Q GEMMs with the largest |K| / |Q| element of the row."""
    hkv = k.shape[1]
    g = q.shape[1] // hkv
    lse, delta = lse.double(), delta.double()
    s = torch.einsum("ihd,jhd->hij", q.double(), _expand(k.double(), g)) * scale
    lse_ = torch.where(torch.isinf(lse), torch.full_like(lse, float("inf")), lse)
    p = torch.exp(s - lse_.unsqueeze(-1)).masked_fill(~vis, 0.0)
    a = torch.einsum("ihd,jhd->hij", dout.double().abs(), _expand(v.double().abs(), g)) + delta.abs().unsqueeze(-1)
    w = p * a * (scale * (q.shape[2] + 2) * EPS32)
    f_dq = torch.einsum("hij,jh->ih", w, _expand(k.double().abs().amax(-1, keepdim=True), g).squeeze(-1))
    f_dk = torch.einsum("hij,ih->jh", w, q.double().abs().amax(-1))
    return f_dq, f_dk.view(k.shape[0], hkv, g).sum(-1)


def lse_budget(q, k, scale, vis, lse_ref, n_tiles):
    """Per (head, row) lse bound of the comment at the top of the file."""
    g = q.shape[1] // k.shape[1]
    a = torch.einsum("ihd,jhd->hij", q.double().abs(), _expand(k.double().abs(), g)) * scale
    a = a.masked_fill(~vis, 0.0).amax(-1)
    d = q.shape[2]
    lse_abs = torch.where(torch.isinf(lse_ref), torch.zeros_like(lse_ref), lse_ref.abs())
    return LSE_SAFETY * ((d + 2) * EPS32 * a + (66 + 2 * n_tiles) * EPS32 + 2.0 ** -22 * (1 + math.log(2))
                         + 3 * EPS32 * lse_abs)


# ---------------------------------------------------------------------------------------------------------------
# the checker
# ---------------------------------------------------------------------------------------------------------------

class Report:
    def __init__(self):
        self.failures = []
        # largest (err_kernel - slack) / err_emulation over rows with a non-zero emulation error: the C_EMU the
        # worst row needed
        self.ratio = 0.0

    @property
    def ok(self):
        return not self.failures

    def __repr__(self):
        return f"Report(ratio={self.ratio:.3g}, failures={self.failures[:4]})"


def check_rows(rep: Report, name, got, ref, emu, dtype, floor=None):
    """got / ref / emu (rows, heads, d).  One row = one (row, head) pair, reduced over d.  ``dtype`` is the model
    dtype: the unit of the rounding the kernels must do, also for results they return in fp32."""
    got, ref, emu = got.double(), ref.double(), emu.double()
    if not torch.isfinite(got).all():
        rep.failures.append(f"{name}: non-finite values")
        return
    ek = (got - ref).abs().amax(-1)
    ee = (emu - ref).abs().amax(-1)
    mx = ref.abs().amax(-1)
    slack = ulp(mx, dtype) + TINY * ref.abs().max()
    if floor is not None:
        slack = slack + floor
    bound = C_EMU * ee + slack
    bad = (ek > bound).nonzero()
    nz = ee > 0
    if nz.any():  # the factor each row needs beyond the fixed slack: a row passes iff it is <= C_EMU
        rep.ratio = max(rep.ratio, ((ek[nz] - slack[nz]).clamp_min(0) / ee[nz]).max().item())
    if bad.numel():
        r, h = bad[0].tolist()
        rep.failures.append(f"{name}: {bad.shape[0]} rows over budget, first row {r} head {h}: "
                            f"err {ek[r, h].item():.3e} > bound {bound[r, h].item():.3e} (emulation {ee[r, h].item():.3e})")


def check_zero_rows(rep: Report, name, got, vis_rows):
    """Rows that see no key must be exactly zero."""
    empty = ~vis_rows
    if empty.any() and (got[empty] != 0).any():
        rep.failures.append(f"{name}: a row without visible keys is not exactly zero")


def check_lse(rep: Report, got, ref, budget):
    got, ref = got.double(), ref.double()
    inf_ref = torch.isinf(ref)
    if (torch.isinf(got) != inf_ref).any() or torch.isnan(got).any():
        rep.failures.append("lse: -inf pattern differs from the oracle (or NaN)")
        return
    if inf_ref.any() and not (got[inf_ref] == float("-inf")).all():
        rep.failures.append("lse: rows without keys must be -inf")
        return
    err = (got - ref).abs().masked_fill(inf_ref, 0.0)
    over = err > budget
    if over.any():
        h, i = over.nonzero()[0].tolist()
        rep.failures.append(f"lse: {int(over.sum())} rows over budget, first head {h} row {i}: "
                            f"{err[h, i].item():.3e} > {budget[h, i].item():.3e}")


def check_fwd(rep, q, k, v, scale, vis, out, lse):
    dtype = q.dtype
    ref_o, ref_l = fwd64(q, k, v, scale, vis)
    emu_o, _ = fwd64(q, k, v, scale, vis, emu=dtype)
    check_rows(rep, "out", out, ref_o, emu_o, dtype)
    check_zero_rows(rep, "out", out, vis.any(-1))
    n_tiles = -(-k.shape[0] // KEY_TILE) + 2
    check_lse(rep, lse, ref_l, lse_budget(q, k, scale, vis, ref_l, n_tiles))
    return ref_o, ref_l


def lse_delta64(q, k, v, dout, scale, vis):
    """The oracle's lse and delta = rowsum(dO * O), in the fp32 form the backward kernel reads."""
    o, l = fwd64(q, k, v, scale, vis)
    delta = (o * dout.double()).sum(-1).t()
    return l.float().contiguous(), delta.float().contiguous()


def check_bwd(rep, q, k, v, dout, scale, vis, lse, delta, dq, dk, dv):
    """dq is the fp32 accumulator (or the model dtype behind the public API); dk / dv fp32 or model dtype."""
    dtype = q.dtype
    ref = bwd64(q, k, v, dout, scale, vis, lse, delta)
    emu = bwd64(q, k, v, dout, scale, vis, lse, delta, emu=dtype)
    f_dq, f_dk = grad_floor(q, k, v, dout, scale, vis, lse, delta)
    for name, got, r, e, f in zip(("dq", "dk", "dv"), (dq, dk, dv), ref, emu, (f_dq, f_dk, None)):
        check_rows(rep, name, got, r, _rnd(e, got.dtype), dtype, f)
    check_zero_rows(rep, "dq", dq, vis.any(-1))
    check_zero_rows(rep, "dk", dk, vis.any(0))
    check_zero_rows(rep, "dv", dv, vis.any(0))


RATIOS = {}


def note(group, rep: Report):
    RATIOS[group] = max(RATIOS.get(group, 0.0), rep.ratio)
    print(f"[numerics] group {group}: case ratio {rep.ratio:.3f}, group max {RATIOS[group]:.3f}")


# ---------------------------------------------------------------------------------------------------------------
# inputs (shared by the CPU self-tests and the GPU tests)
# ---------------------------------------------------------------------------------------------------------------

def _gen(seed, device):
    return torch.Generator(device=device).manual_seed(seed)


def rand_inputs(sq, k_rows, hq, hkv, d, dtype, seed, device="cpu"):
    g = _gen(seed, device)
    r = lambda *s: torch.randn(*s, generator=g, device=device, dtype=torch.float32)  # noqa: E731
    return (r(sq, hq, d).to(dtype), r(k_rows, hkv, d).to(dtype), r(k_rows, hkv, d).to(dtype),
            r(sq, hq, d).to(dtype))


def _unit(n, d, g, device):
    u = torch.randn(n, d, generator=g, device=device, dtype=torch.float64)
    return u / u.norm(dim=-1, keepdim=True)


def probe_inputs(sq, k_rows, hq, hkv, d, dtype, seed, edge, kv_row0=0, kv_len=None, diag=None, lo=None,
                 device="cpu"):
    """Mask-edge probes: for every query row the first key just outside its mask scores far above every visible
    key, so a one-key leak moves that row's output (or that key's dK / dV) by O(1).  q_i = a u_i, k_j = b u_pi(j)
    with near-orthogonal random unit directions (|u_i . u_j| ~ 0.4 at most for d = 64), a b scale = 40 nats.

    edge "upper": key i + diag + 1 of the segment carries row i's direction; "lower": key i + lo - 1 does; "ragged":
    every K row outside [kv_row0, kv_row0 + kv_len) points along one direction w that every query shares."""
    g = _gen(seed, device)
    scale = 1.0 / math.sqrt(d)
    ab = 40.0 / scale
    a = b = math.sqrt(ab)
    grp = hq // hkv
    q = torch.empty(sq, hq, d, dtype=torch.float64, device=device)
    k = torch.empty(k_rows, hkv, d, dtype=torch.float64, device=device)
    jj = torch.arange(k_rows, device=device) - kv_row0
    for h in range(hkv):
        u = _unit(sq + k_rows, d, g, device)
        if edge == "ragged":
            w = u[-1]
            qh = a * (0.6 * w + 0.8 * u[:sq])
            kh = b * u[sq:sq + k_rows]
            outside = (jj < 0) | (jj >= kv_len)
            kh[outside] = b * w
        else:
            qh = a * u[:sq]
            owner = jj - diag - 1 if edge == "upper" else jj - lo + 1  # the row whose first invisible key is jj
            kh = b * u[sq:sq + k_rows]
            hit = (owner >= 0) & (owner < sq)
            kh[hit] = b * u[owner[hit]]
        k[:, h] = kh
        q[:, h * grp:(h + 1) * grp] = qh.unsqueeze(1)
    gv = torch.randn(k_rows, hkv, d, generator=g, device=device, dtype=torch.float64)
    do = torch.randn(sq, hq, d, generator=g, device=device, dtype=torch.float64)
    return q.to(dtype), k.to(dtype), gv.to(dtype), do.to(dtype)


RESCALE_PATTERNS = ("grow9", "grow7.9", "alternate", "underflow", "pm80")


def rescale_inputs(pattern, sq, sk, hq, hkv, d, dtype, seed, device="cpu"):
    """Scores in log2 units s2(i, j) = a_i f_j + b_i g_j + noise, carried by the first two head dims; the rest is
    small noise.  Patterns (key tile t = j // 128):
      grow9      +9 per key tile (a rescale on every tile),      grow7.9  +7.9 per tile (P approaches 2^7.9),
      alternate  growth on even rows only (a warp mixes rows that need a rescale with rows that do not),
      underflow  0, +150, then falling (the rescale factor and later P underflow),
      pm80       +-80 offsets with +9 per tile."""
    g = _gen(seed, device)
    scale = 1.0 / math.sqrt(d)
    c = 1.0 / (scale * LOG2E)
    i = torch.arange(sq, device=device, dtype=torch.float64)
    j = torch.arange(sk, device=device, dtype=torch.float64)
    t = torch.div(j, KEY_TILE, rounding_mode="floor")
    noise = 0.1 if pattern == "grow7.9" else 0.3
    zeros_q, ones_q = torch.zeros_like(i), torch.ones_like(i)
    f = torch.zeros_like(j)
    if pattern == "grow9":
        a, b, gg = zeros_q, ones_q, 9.0 * t + 0.5 * (j % KEY_TILE) / KEY_TILE
    elif pattern == "grow7.9":
        a, b, gg = zeros_q, ones_q, 7.9 * t
    elif pattern == "alternate":
        a, b, gg = zeros_q, (i % 2 == 0).double(), 9.0 * t
    elif pattern == "underflow":
        a, b = zeros_q, ones_q
        gg = torch.tensor([0.0, 150.0, 100.0, 40.0, -20.0, -80.0], device=device, dtype=torch.float64)[t.long()]
    else:
        sign = torch.where(torch.rand(sq, generator=g, device=device) < 0.5, -1.0, 1.0).double()
        a, b, f, gg = 80.0 * sign, ones_q, torch.ones_like(j), 9.0 * t
    q = torch.randn(sq, hq, d, generator=g, device=device, dtype=torch.float64) * noise
    k = torch.randn(sk, hkv, d, generator=g, device=device, dtype=torch.float64) * noise
    q[:, :, 0], q[:, :, 1] = (a * c).unsqueeze(1), (b * c).unsqueeze(1)
    k[:, :, 0], k[:, :, 1] = f.unsqueeze(1), gg.unsqueeze(1)
    v = torch.randn(sk, hkv, d, generator=g, device=device, dtype=torch.float64)
    return q.to(dtype), k.to(dtype), v.to(dtype)


def rescale_events(q, k, scale, vis):
    """Replay of the forward kernel's threshold rule on the rounded inputs: per (head, row) the number of key tiles
    after the first visited one where the row max grew by more than 2^8 (the O accumulator is rescaled)."""
    g = q.shape[1] // k.shape[1]
    s2 = torch.einsum("ihd,jhd->hij", q.double(), _expand(k.double(), g)) * (scale * LOG2E)
    s2 = s2.masked_fill(~vis, float("-inf"))
    m2 = torch.full(s2.shape[:2], float("-inf"), dtype=torch.float64, device=s2.device)
    events = torch.zeros(s2.shape[:2], dtype=torch.long, device=s2.device)
    for t0 in range(0, s2.shape[-1], KEY_TILE):
        mx = s2[..., t0:t0 + KEY_TILE].amax(-1)
        need = (mx - m2) > RESCALE_THRESHOLD
        events += (need & torch.isfinite(m2)).long()
        m2 = torch.where(need, mx, m2)
    return events


# ---------------------------------------------------------------------------------------------------------------
# kernel-like CPU model and its mutants
# ---------------------------------------------------------------------------------------------------------------

def _kv_head_map(hq, hkv, wrong_gqa):
    g = hq // hkv
    return [(h % hkv) if wrong_gqa else (h // g) for h in range(hq)]


def kl_fwd(q, k, v, scale, vis, skip_rescale=False, drop_tile=None, wrong_gqa=False):
    """fp32 forward in 128-key tiles: P = exp2(s t2 - m) against a reference max m that only moves when the row max
    grew by more than 2^8, P rounded to the model dtype for PV, l summed from the unrounded P."""
    dtype = q.dtype
    hmap = _kv_head_map(q.shape[1], k.shape[1], wrong_gqa)
    kf, vf = k.float()[:, hmap], v.float()[:, hmap]
    t2 = scale * LOG2E
    s = torch.einsum("ihd,jhd->hij", q.float(), kf).masked_fill(~vis, float("-inf"))
    hq, sq, sk = s.shape
    m2 = torch.full((hq, sq), float("-inf"))
    l = torch.zeros(hq, sq)
    o = torch.zeros(hq, sq, q.shape[2])
    for ti, t0 in enumerate(range(0, sk, KEY_TILE)):
        if ti == drop_tile:
            continue
        st = s[..., t0:t0 + KEY_TILE]
        m_new = torch.maximum(m2, st.amax(-1) * t2)
        need = (m_new - m2) > RESCALE_THRESHOLD
        f = torch.where(need, torch.exp2(m2 - m_new), torch.ones_like(m2))
        l = l * f
        if not skip_rescale:
            o = o * f.unsqueeze(-1)
        m2 = torch.where(need, m_new, m2)
        mc = torch.where(torch.isinf(m2), torch.zeros_like(m2), m2)
        p = torch.exp2(st * t2 - mc.unsqueeze(-1))
        l = l + p.sum(-1)
        o = o + torch.einsum("hij,jhd->hid", p.to(dtype).float(), vf[t0:t0 + KEY_TILE])
    out = (o / torch.where(l > 0, l, torch.ones_like(l)).unsqueeze(-1)).to(dtype).transpose(0, 1)
    lse = torch.where(l > 0, (m2 + torch.log2(l.clamp_min(1e-38))) * math.log(2), torch.full_like(l, float("-inf")))
    return out.contiguous(), lse


def kl_bwd(q, k, v, dout, scale, vis, lse, delta, dkv_dtype, wrong_gqa=False, one_head=False):
    dtype = q.dtype
    hq, hkv = q.shape[1], k.shape[1]
    hmap = _kv_head_map(hq, hkv, wrong_gqa)
    kf, vf, qf, dof = k.float()[:, hmap], v.float()[:, hmap], q.float(), dout.float()
    s = torch.einsum("ihd,jhd->hij", qf, kf)
    lse2 = torch.where(torch.isinf(lse), torch.full_like(lse, float("inf")), lse * LOG2E)
    p = torch.exp2(s * (scale * LOG2E) - lse2.unsqueeze(-1)).masked_fill(~vis, 0.0)
    dv = torch.einsum("hij,ihd->jhd", p.to(dtype).float(), dof)
    dp = torch.einsum("ihd,jhd->hij", dof, vf)
    ds = (p * (dp - delta.unsqueeze(-1)) * scale).to(dtype).float()
    dq = torch.einsum("hij,jhd->ihd", ds, kf)
    dk = torch.einsum("hij,ihd->jhd", ds, qf)
    dk_o = torch.zeros(k.shape, dtype=torch.float32)
    dv_o = torch.zeros(k.shape, dtype=torch.float32)
    seen = set()
    for h in range(hq):
        kh = hmap[h]
        if one_head and kh in seen:
            continue
        seen.add(kh)
        dk_o[:, kh] += dk[:, h]
        dv_o[:, kh] += dv[:, h]
    return dq, dk_o.to(dkv_dtype), dv_o.to(dkv_dtype)


# ---------------------------------------------------------------------------------------------------------------
# B. CPU self-tests of the checker
# ---------------------------------------------------------------------------------------------------------------

def _kl_case_fwd(q, k, v, scale, vis, vis_kernel=None, **mut):
    rep = Report()
    out, lse = kl_fwd(q, k, v, scale, vis if vis_kernel is None else vis_kernel, **mut)
    check_fwd(rep, q, k, v, scale, vis, out, lse)
    return rep


def _kl_case_bwd(q, k, v, dout, scale, vis, dkv_dtype, vis_kernel=None, **mut):
    rep = Report()
    lse, delta = lse_delta64(q, k, v, dout, scale, vis)
    dq, dk, dv = kl_bwd(q, k, v, dout, scale, vis if vis_kernel is None else vis_kernel, lse, delta, dkv_dtype, **mut)
    check_bwd(rep, q, k, v, dout, scale, vis, lse, delta, dq, dk, dv)
    return rep


_KL_SHAPES = [  # dtype, d, sq, sk, hq, hkv, diag, lo
    (torch.bfloat16, 128, 257, 383, 4, 2, 63, None),
    (torch.float16, 64, 300, 300, 8, 2, 0, None),
    (torch.bfloat16, 64, 129, 257, 2, 1, -1, -128),
    (torch.float16, 128, 200, 256, 2, 1, None, None),
]


@pytest.mark.parametrize("seed", range(20))
def test_kernel_like_model_passes(seed):
    """No false positives: the kernel-like model passes the per-row budget on random, probe and rescale inputs."""
    dtype, d, sq, sk, hq, hkv, diag, lo = _KL_SHAPES[seed % len(_KL_SHAPES)]
    scale = 1 / math.sqrt(d)
    q, k, v, do = rand_inputs(sq, sk, hq, hkv, d, dtype, seed)
    vis = seg_vis(sq, sk, 0, sk, diag, lo)
    for rep in (_kl_case_fwd(q, k, v, scale, vis), _kl_case_bwd(q, k, v, do, scale, vis, torch.float32),
                _kl_case_bwd(q, k, v, do, scale, vis, dtype)):
        assert rep.ok, rep
    q, k, v, do = probe_inputs(300, 300, 2, 1, d, dtype, seed, "upper", diag=diag if diag is not None else 0)
    vis = seg_vis(300, 300, 0, 300, diag if diag is not None else 0, None)
    assert _kl_case_fwd(q, k, v, scale, vis).ok
    assert _kl_case_bwd(q, k, v, do, scale, vis, torch.float32).ok
    pattern = RESCALE_PATTERNS[seed % len(RESCALE_PATTERNS)]
    q, k, v = rescale_inputs(pattern, 256, 600, 2, 1, d, dtype, seed)
    rep = _kl_case_fwd(q, k, v, scale, torch.ones(256, 600, dtype=torch.bool))
    assert rep.ok, (pattern, rep)


def _leak(vis_base, sq, sk, diag, rows_from=0):
    extra = seg_vis(sq, sk, 0, sk, diag + 1, None) & ~vis_base
    extra[:rows_from] = False
    return vis_base | extra


MUTANTS = ["fwd_causal_leak", "bwd_causal_leak_late_rows", "window_lower_off_by_one", "dropped_key_tile",
           "skipped_o_rescale", "wrong_gqa_head_map", "dkdv_one_head_of_group"]


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("mutant", MUTANTS)
def test_mutant_is_flagged(mutant, dtype):
    """Every mutant must fail the budget on the inputs the GPU tests use (probes for mask edges, rescale stress for
    the O rescale, random inputs for tiles and heads), while the unmutated model passes on the same inputs."""
    d, scale = 128, 1 / math.sqrt(128)
    if mutant in ("fwd_causal_leak", "bwd_causal_leak_late_rows"):
        sq = sk = 640
        q, k, v, do = probe_inputs(sq, sk, 2, 1, d, dtype, 3, "upper", diag=0)
        vis = seg_vis(sq, sk, 0, sk, 0, None)
        if mutant == "fwd_causal_leak":
            good, bad = _kl_case_fwd(q, k, v, scale, vis), _kl_case_fwd(q, k, v, scale, vis, _leak(vis, sq, sk, 0))
        else:
            good = _kl_case_bwd(q, k, v, do, scale, vis, torch.float32)
            bad = _kl_case_bwd(q, k, v, do, scale, vis, torch.float32, _leak(vis, sq, sk, 0, rows_from=256))
    elif mutant == "window_lower_off_by_one":
        sq = sk = 383
        q, k, v, do = probe_inputs(sq, sk, 2, 1, d, dtype, 4, "lower", lo=-100)
        vis = seg_vis(sq, sk, 0, sk, 0, -100)
        good = _kl_case_fwd(q, k, v, scale, vis)
        bad = _kl_case_fwd(q, k, v, scale, vis, seg_vis(sq, sk, 0, sk, 0, -101))
    elif mutant == "skipped_o_rescale":
        q, k, v = rescale_inputs("grow9", 256, 600, 2, 1, d, dtype, 5)
        vis = torch.ones(256, 600, dtype=torch.bool)
        good, bad = _kl_case_fwd(q, k, v, scale, vis), _kl_case_fwd(q, k, v, scale, vis, skip_rescale=True)
    else:
        sq, sk = 257, 383
        q, k, v, do = rand_inputs(sq, sk, 4, 2, d, dtype, 6)
        vis = seg_vis(sq, sk, 0, sk, 128, None)
        if mutant == "dropped_key_tile":
            good, bad = _kl_case_fwd(q, k, v, scale, vis), _kl_case_fwd(q, k, v, scale, vis, drop_tile=1)
        elif mutant == "wrong_gqa_head_map":
            good, bad = _kl_case_fwd(q, k, v, scale, vis), _kl_case_fwd(q, k, v, scale, vis, wrong_gqa=True)
        else:
            good = _kl_case_bwd(q, k, v, do, scale, vis, dtype)
            bad = _kl_case_bwd(q, k, v, do, scale, vis, dtype, one_head=True)
    assert good.ok, good
    assert not bad.ok, f"{mutant} was not flagged: {bad}"
    print(f"[numerics] mutant {mutant} ({dtype}) flagged: {bad.failures[0]}")


def test_rescale_patterns_fire_on_most_rows():
    """The rescale-stress inputs reach the lazy O rescale (host replay of the kernel's threshold rule)."""
    for pattern in RESCALE_PATTERNS:
        q, k, _ = rescale_inputs(pattern, 256, 600, 2, 1, 128, torch.bfloat16, 0)
        ev = rescale_events(q, k, 1 / math.sqrt(128), torch.ones(256, 600, dtype=torch.bool))
        _assert_fires(pattern, ev)


def _assert_fires(pattern, ev):
    fired = ev > 0
    if pattern == "alternate":
        assert fired[:, 0::2].all() and not fired[:, 1::2].any(), pattern
    else:
        assert fired.float().mean().item() >= 0.9, (pattern, fired.float().mean().item())


# ---------------------------------------------------------------------------------------------------------------
# GPU: kernels
# ---------------------------------------------------------------------------------------------------------------

def _attn_cuda():
    from ring_flash_attn_b200.ops import attn_cuda, cuda_ext

    cuda_ext.load()
    return attn_cuda


def _block_plan(sq, k_rows, kv_row0, kv_len, diag, lo):
    return P.CPPlan(1, 0, sq, k_rows, [P.QChunk(0, sq)], [P.Segment(0, 0, kv_row0, kv_len, diag, lo)])


def run_block(q, k, v, do, scale, kv_row0, kv_len, diag, lo, dkv_dtype, lse=None, delta=None, fwd=True):
    """One chunk x one segment through segments_forward / segments_backward (window variants when ``lo`` is set).
    Backward uses the given (oracle) lse / delta."""
    ac = _attn_cuda()
    plan = _block_plan(q.shape[0], k.shape[0], kv_row0, kv_len, diag, lo)
    if fwd:
        return ac.segments_forward(plan, plan.segments, q, k, v, scale)
    dq = torch.zeros(q.shape, dtype=torch.float32, device=q.device)
    dk = torch.zeros(k.shape, dtype=dkv_dtype, device=q.device)
    dv = torch.zeros(k.shape, dtype=dkv_dtype, device=q.device)
    ac.segments_backward(plan, plan.segments, do, q, k, v, lse, delta, scale, dq, dk, dv)
    return dq, dk, dv


BF, FP = torch.bfloat16, torch.float16
# dtype, d, sq, sk, diag, lo, hq, hkv, dK/dV fp32
SWEEP = [
    (BF, 128, 1, 1, 0, None, 1, 1, True),
    (FP, 128, 63, 65, None, None, 2, 1, False),
    (BF, 64, 64, 64, 0, None, 4, 1, True),
    (FP, 64, 65, 129, -1, None, 2, 2, False),
    (BF, 128, 127, 383, 128, None, 8, 1, False),
    (FP, 128, 128, 255, 127, None, 16, 1, True),
    (BF, 64, 257, 257, -129, None, 2, 1, False),
    (FP, 64, 255, 256, -128, None, 1, 1, True),
    (BF, 128, 256, 127, -127, None, 4, 2, True),
    (FP, 128, 257, 383, 63, None, 8, 2, False),
    (BF, 64, 383, 128, 64, None, 16, 2, True),
    (FP, 128, 383, 383, 382, None, 1, 1, False),
    (BF, 128, 256, 257, 1, None, 2, 1, True),
    (FP, 64, 1, 383, 382, None, 4, 4, True),
    (BF, 128, 129, 63, None, None, 16, 16, False),
    (FP, 64, 383, 255, 0, None, 8, 1, True),
    # sliding window (kWindow kernels)
    (BF, 128, 383, 383, 0, -128, 2, 1, True),
    (FP, 128, 257, 383, 1, -127, 4, 1, False),
    (BF, 64, 256, 256, 0, -129, 1, 1, False),
    (FP, 64, 383, 257, 64, -64, 2, 2, True),
    (BF, 128, 129, 255, -1, -65, 8, 1, False),
    (FP, 128, 255, 383, 127, -1, 2, 1, True),
    (BF, 64, 127, 129, 128, 0, 16, 1, True),
    (FP, 128, 383, 383, None, -63, 2, 1, False),
    (BF, 128, 65, 383, 255, 127, 4, 1, True),
    (FP, 64, 256, 383, 128, 1, 2, 1, False),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", range(len(SWEEP)))
def test_block_sweep(case):
    """C: one chunk x one segment at tile-edge shapes and diagonals, every dtype / head-dim instantiation, GQA up
    to 16, dK / dV in fp32 and in the model dtype."""
    dtype, d, sq, sk, diag, lo, hq, hkv, dkv32 = SWEEP[case]
    scale = 1 / math.sqrt(d)
    q, k, v, do = rand_inputs(sq, sk, hq, hkv, d, dtype, 100 + case, device="cuda")
    vis = seg_vis(sq, sk, 0, sk, diag, lo, device="cuda")
    rep = Report()
    out, lse = run_block(q, k, v, do, scale, 0, sk, diag, lo, None)
    check_fwd(rep, q, k, v, scale, vis, out, lse)
    l64, d64 = lse_delta64(q, k, v, do, scale, vis)
    grads = run_block(q, k, v, do, scale, 0, sk, diag, lo, torch.float32 if dkv32 else dtype, l64, d64, fwd=False)
    check_bwd(rep, q, k, v, do, scale, vis, l64, d64, *grads)
    note("C", rep)
    assert rep.ok, rep


PROBES = [  # dtype, d, edge, sq, k_rows, kv_row0, kv_len, diag, lo, hq, hkv
    (BF, 128, "upper", 640, 640, 0, 640, 0, None, 2, 1),
    (FP, 128, "upper", 383, 383, 0, 383, -1, None, 2, 1),
    (BF, 64, "upper", 300, 383, 0, 383, 63, None, 4, 2),
    (FP, 64, "upper", 256, 384, 0, 384, 128, None, 2, 1),
    (BF, 128, "upper", 383, 256, 0, 256, -128, None, 2, 2),
    (BF, 128, "lower", 383, 383, 0, 383, 0, -100, 2, 1),
    (FP, 64, "lower", 300, 383, 0, 383, 64, -64, 2, 1),
    (FP, 128, "lower", 257, 383, 0, 383, None, -127, 4, 1),
    (BF, 64, "lower", 256, 256, 0, 256, 129, 1, 2, 1),
    (BF, 128, "ragged", 300, 420, 100, 200, None, None, 2, 1),
    (FP, 128, "ragged", 256, 420, 37, 250, 150, None, 2, 1),
    (FP, 64, "ragged", 129, 300, 128, 129, None, None, 4, 2),
]


@pytest.mark.gpu
@pytest.mark.parametrize("direction", ["fwd", "bwd"])
@pytest.mark.parametrize("case", range(len(PROBES)))
def test_mask_edge_probe(case, direction):
    """D: a key leaking through the causal edge, the window's lower edge or past a segment's end moves a row by O(1)."""
    dtype, d, edge, sq, k_rows, kv_row0, kv_len, diag, lo, hq, hkv = PROBES[case]
    scale = 1 / math.sqrt(d)
    q, k, v, do = probe_inputs(sq, k_rows, hq, hkv, d, dtype, 200 + case, edge, kv_row0, kv_len, diag, lo, "cuda")
    vis = seg_vis(sq, k_rows, kv_row0, kv_len, diag, lo, device="cuda")
    rep = Report()
    if direction == "fwd":
        out, lse = run_block(q, k, v, do, scale, kv_row0, kv_len, diag, lo, None)
        check_fwd(rep, q, k, v, scale, vis, out, lse)
    else:
        l64, d64 = lse_delta64(q, k, v, do, scale, vis)
        grads = run_block(q, k, v, do, scale, kv_row0, kv_len, diag, lo, torch.float32, l64, d64, fwd=False)
        check_bwd(rep, q, k, v, do, scale, vis, l64, d64, *grads)
    note("D", rep)
    assert rep.ok, rep


@pytest.mark.gpu
@pytest.mark.parametrize("pattern", RESCALE_PATTERNS)
@pytest.mark.parametrize("dtype,d", [(BF, 128), (FP, 128), (BF, 64), (FP, 64)])
def test_rescale_stress(dtype, d, pattern):
    """E: the forward's lazy O rescale (tensor-memory read-modify-write from the softmax warps) on inputs that fire it."""
    sq, sk = 256, 600
    scale = 1 / math.sqrt(d)
    q, k, v = rescale_inputs(pattern, sq, sk, 2, 1, d, dtype, 300, device="cuda")
    vis = torch.ones(sq, sk, dtype=torch.bool, device="cuda")
    ev = rescale_events(q, k, scale, vis)
    _assert_fires(pattern, ev)
    rep = Report()
    out, lse = run_block(q, k, v, None, scale, 0, sk, None, None, None)
    check_fwd(rep, q, k, v, scale, vis, out, lse)
    print(f"[numerics] E {pattern} {dtype} d{d}: rescale events {int(ev.sum())} on "
          f"{int((ev > 0).sum())}/{ev.numel()} rows")
    note("E", rep)
    assert rep.ok, rep


# ---------------------------------------------------------------------------------------------------------------
# F. multi-source tables replayed on one GPU
# ---------------------------------------------------------------------------------------------------------------

def _doc_pos(tokens, cu):
    cu_t = torch.as_tensor(cu, dtype=torch.long, device=tokens.device)
    doc = torch.searchsorted(cu_t, tokens, right=True) - 1
    return tokens - cu_t[doc], doc


PACK_CU = [0, 144, 1008, 1536]  # document lengths divisible by 2 W for every W below


def _replay_setup(scheme, rank, world, window):
    """(plan, global token index of every local row as a function of the rank, total tokens, cu_seqlens)."""
    left = 100 if window else None
    win = (left, 0) if window else (-1, -1)
    if scheme in ("ring", "zigzag", "stripe"):
        L = 192
        total, cu = world * L, [0, world * L]
        shard = {"ring": layouts.shard_ring, "zigzag": layouts.shard_zigzag, "stripe": layouts.shard_stripe}[scheme]
        rows = lambda r: shard(torch.arange(total).unsqueeze(0), r, world)[0]  # noqa: E731
        plan = {"ring": lambda: P.plan_ring(rank, world, 1, L, True, win),
                "zigzag": lambda: P.plan_zigzag(rank, world, 1, L, win),
                "stripe": lambda: P.plan_stripe(rank, world, 1, L, win)}[scheme]()
        return plan, rows, total, cu, left
    cu = PACK_CU
    total = cu[-1]
    if scheme == "varlen":
        rows = lambda r: layouts.shard_ring_varlen(torch.arange(total), cu, r, world)  # noqa: E731
        plan = P.plan_ring_varlen(rank, world, [c // world for c in cu], True, win)
    elif scheme == "llama3":
        from ring_flash_attn_b200.parallel.api import llama3_flash_attn_prepare_cu_seqlens

        rows = lambda r: layouts.shard_llama3(torch.arange(total), r, world)  # noqa: E731
        cq, ck, _, _, ks = llama3_flash_attn_prepare_cu_seqlens(torch.tensor(cu, dtype=torch.int32), True, rank, world)
        plan = P.plan_llama3(rank, world, total // world, cq.tolist(), ck.tolist(), ks.start, True, win)
    else:
        rows = lambda r: layouts.shard_zigzag_llama3(torch.arange(total), r, world)  # noqa: E731
        plan = P.plan_zigzag_llama3(rank, world, cu, True, win)
    return plan, rows, total, cu, left


@pytest.mark.gpu
@pytest.mark.parametrize("window", [False, True])
@pytest.mark.parametrize("scheme", ["ring", "zigzag", "stripe", "varlen", "llama3", "zigzag_llama3"])
def test_multi_source_replay(scheme, window):
    """F: every rank's tables with every source's K / V shard concatenated in one tensor (row_offset src * L, no
    ready flags): one forward and one backward launch walk all sources, as a fused multi-GPU launch does."""
    ac = _attn_cuda()
    from ring_flash_attn_b200.ops import cuda_ext

    C = cuda_ext.load()
    batch = scheme in ("ring", "zigzag", "stripe")
    d, hq, hkv = (128, 4, 2) if batch else (64, 4, 1)
    max_segs = {}
    for world in (2, 3, 4, 8):
        dtype = BF if world in (2, 8) else FP
        scale = 1 / math.sqrt(d)
        for rank in range(world):
            plan, rows, total, cu, left = _replay_setup(scheme, rank, world, window)
            g = _gen(1000 * world + rank, "cuda")
            Q = torch.randn(total, hq, d, generator=g, device="cuda").to(dtype)
            K = torch.randn(total, hkv, d, generator=g, device="cuda").to(dtype)
            V = torch.randn(total, hkv, d, generator=g, device="cuda").to(dtype)
            DO = torch.randn(total, hq, d, generator=g, device="cuda").to(dtype)
            L = plan.q_rows
            all_rows = torch.cat([rows(s) for s in range(world)]).to("cuda")
            mine = rows(rank).to("cuda")
            q, do = Q[mine].contiguous(), DO[mine].contiguous()
            k, v = K[all_rows].contiguous(), V[all_rows].contiguous()
            pq, dq_ = _doc_pos(mine, cu)
            pk, dk_ = _doc_pos(all_rows, cu)
            vis = pos_vis(pq, dq_, pk, dk_, left)
            offs = {s: s * L for s in range(world)}
            segs = plan.segments
            win = ac.has_window(segs)
            dev = q.device
            out = torch.zeros(q.shape, dtype=dtype, device=dev)
            lse = torch.full((hq, L), float("-inf"), device=dev)
            if win:
                items, seg_rows, seg_lo, _ = ac.fwd_tables_window_host(plan, segs, offs)
            else:
                items, seg_rows, _ = ac.fwd_tables_host(plan, segs, offs)
            if batch and not window:
                max_segs[(world, rank)] = max(it[4] for it in items)
            items_t = ac._to_dev(items, 8, dev)
            seg_t = ac._to_dev(seg_rows if seg_rows else [[0, 0, 0, -1]], 4, dev)
            if items:
                if win:
                    lo_t = torch.tensor(seg_lo if seg_lo else [ac.LO_NONE], dtype=torch.int32, device=dev)
                    C.attn_fwd_window(q, k, v, items_t, seg_t, lo_t, out, lse, L, scale)
                else:
                    C.attn_fwd(q, k, v, items_t, seg_t, out, lse, L, scale)
            rep = Report()
            check_fwd(rep, q, k, v, scale, vis, out, lse)
            l64, d64 = lse_delta64(q, k, v, do, scale, vis)
            bi, bq = (ac.bwd_tables_window_host if win else ac.bwd_tables_host)(plan, segs, offs)
            dq = torch.zeros(q.shape, dtype=torch.float32, device=dev)
            dk = torch.zeros(k.shape, dtype=torch.float32, device=dev)
            dv = torch.zeros(k.shape, dtype=torch.float32, device=dev)
            ac.backward_launch(q, do, k, v, l64, d64, ac._to_dev(bi, 8, dev),
                               ac._to_dev(bq if bq else [[0, 0, 0, 0]], 4, dev), scale, dq, dk, dv, window=win)
            check_bwd(rep, q, k, v, do, scale, vis, l64, d64, dq, dk, dv)
            note("F", rep)
            assert rep.ok, (scheme, world, rank, window, rep)
    if max_segs:
        print(f"[numerics] F {scheme}: largest segments per item by world "
              f"{ {w: max(n for (ww, _), n in max_segs.items() if ww == w) for w in (2, 3, 4, 8)} }")
        for w in (2, 3, 4, 8):
            assert max(n for (ww, _), n in max_segs.items() if ww == w) >= w, (scheme, w, max_segs)


# ---------------------------------------------------------------------------------------------------------------
# G. fp16 through the public API (world size 1)
# ---------------------------------------------------------------------------------------------------------------

def _api_check(rep, q, k, v, do, scale, vis, out, lse, dq, dk, dv, chunk=None):
    """Forward outputs and model-dtype gradients of a whole call.  The emulated backward takes delta from the
    emulated (rounded) output, as the library computes it from its own output.  ``chunk``: process the query rows
    in slices (long sequences)."""
    dtype = q.dtype
    sq = q.shape[0]
    chunk = chunk or sq
    grads_ref = [torch.zeros(t.shape, dtype=torch.float64, device=q.device) for t in (k, k)]
    grads_emu = [torch.zeros_like(x) for x in grads_ref]
    f_dk = torch.zeros(k.shape[:2], dtype=torch.float64, device=q.device)
    for i0 in range(0, sq, chunk):
        sl = slice(i0, min(sq, i0 + chunk))
        vs = vis[sl]
        ref_o, ref_l = fwd64(q[sl], k, v, scale, vs)
        emu_o, _ = fwd64(q[sl], k, v, scale, vs, emu=dtype)
        check_rows(rep, "out", out[sl], ref_o, emu_o, dtype)
        check_zero_rows(rep, "out", out[sl], vs.any(-1))
        check_lse(rep, lse[:, sl], ref_l, lse_budget(q[sl], k, scale, vs, ref_l, -(-k.shape[0] // KEY_TILE) + 2))
        d_ref = (ref_o * do[sl].double()).sum(-1).t()
        d_emu = (emu_o * do[sl].double()).sum(-1).t()
        r = bwd64(q[sl], k, v, do[sl], scale, vs, ref_l, d_ref)
        e = bwd64(q[sl], k, v, do[sl], scale, vs, ref_l, d_emu, emu=dtype)
        f = grad_floor(q[sl], k, v, do[sl], scale, vs, ref_l, d_ref)
        f_dk += f[1]
        check_rows(rep, "dq", dq[sl], r[0], _rnd(e[0], dtype), dtype, f[0])
        for acc, x in zip(grads_ref, r[1:]):
            acc += x
        for acc, x in zip(grads_emu, e[1:]):
            acc += x
    check_rows(rep, "dk", dk, grads_ref[0], _rnd(grads_emu[0], dtype), dtype, f_dk)
    check_rows(rep, "dv", dv, grads_ref[1], _rnd(grads_emu[1], dtype), dtype)


@pytest.mark.gpu
def test_fp16_api_batch_qkvpacked():
    """G: fp16 zigzag qkvpacked call (the _Unpack path and the fp16 dq_finalize) at world size 1."""
    import ring_flash_attn_b200 as rfa

    B, S, H, d = 2, 640, 4, 128
    g = _gen(400, "cuda")
    qkv = torch.randn(B, S, 3, H, d, generator=g, device="cuda").to(FP).requires_grad_(True)
    dout = torch.randn(B, S, H, d, generator=g, device="cuda").to(FP)
    out, lse, _ = rfa.zigzag_ring_flash_attn_qkvpacked_func(qkv, causal=True, return_attn_probs=True)
    out.backward(dout)
    scale = 1 / math.sqrt(d)
    vis = seg_vis(S, S, 0, S, 0, None, device="cuda")
    rep = Report()
    x, gr = qkv.detach(), qkv.grad
    for b in range(B):
        _api_check(rep, x[b, :, 0], x[b, :, 1], x[b, :, 2], dout[b], scale, vis, out[b].detach(), lse[b],
                   gr[b, :, 0], gr[b, :, 1], gr[b, :, 2])
    note("G", rep)
    assert rep.ok, rep


@pytest.mark.gpu
def test_fp16_api_varlen_kvpacked():
    import ring_flash_attn_b200 as rfa

    T, H, HK, d = 1200, 8, 2, 64
    cu = [0, 1, 130, 700, T]
    g = _gen(401, "cuda")
    q = torch.randn(T, H, d, generator=g, device="cuda").to(FP).requires_grad_(True)
    kv = torch.randn(T, 2, HK, d, generator=g, device="cuda").to(FP).requires_grad_(True)
    dout = torch.randn(T, H, d, generator=g, device="cuda").to(FP)
    cu_t = torch.tensor(cu, dtype=torch.int32, device="cuda")
    out, lse, _ = rfa.ring_flash_attn_varlen_kvpacked_func(q, kv, cu_t, 570, causal=True, return_attn_probs=True)
    out.backward(dout)
    tok = torch.arange(T, device="cuda")
    pos, doc = _doc_pos(tok, cu)
    vis = pos_vis(pos, doc, pos, doc)
    rep = Report()
    _api_check(rep, q.detach(), kv.detach()[:, 0], kv.detach()[:, 1], dout, 1 / math.sqrt(d), vis, out.detach(), lse,
               q.grad, kv.grad[:, 0], kv.grad[:, 1])
    note("G", rep)
    assert rep.ok, rep


@pytest.mark.gpu
def test_fp16_api_long_sequence_backward():
    """S = 16384 fp16 causal: P ~ 1 / S on late rows pushes dS = P (dP - delta) scale towards fp16 subnormals."""
    import ring_flash_attn_b200 as rfa

    S, H, d = 16384, 2, 128
    g = _gen(402, "cuda")
    qkv = torch.randn(1, S, 3, H, d, generator=g, device="cuda").to(FP).requires_grad_(True)
    dout = torch.randn(1, S, H, d, generator=g, device="cuda").to(FP)
    out, lse, _ = rfa.zigzag_ring_flash_attn_qkvpacked_func(qkv, causal=True, return_attn_probs=True)
    out.backward(dout)
    x, gr = qkv.detach()[0], qkv.grad[0]
    vis = seg_vis(S, S, 0, S, 0, None, device="cuda")
    rep = Report()
    _api_check(rep, x[:, 0], x[:, 1], x[:, 2], dout[0], 1 / math.sqrt(d), vis, out.detach()[0], lse[0],
               gr[:, 0], gr[:, 1], gr[:, 2], chunk=1024)
    note("G", rep)
    assert rep.ok, rep
