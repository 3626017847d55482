"""mmg_attention at the shapes and inputs where attention kernels go wrong, element by element against a float64 reference.

Every route is driven through ops.attention and compared with softmax(scale q k^T + mask) v computed in float64 from the same bf16-exact (or
fp32) inputs: key 0 is the null key and is never masked, masked logits are -finfo.max (attend.py:128-131).  The routes:
  bf16_tc_2pass   bf16, tcgen05 kernel, exact two-pass softmax (logit_bound = 0)
  bf16_tc_1pass   bf16, tcgen05 kernel, single-pass softmax against the caller's bound (2 bound scale log2e < 100)
  fp32_split      fp32 on the tensor cores (three bf16 terms per operand, mmg_attention_split.cuh)
  fp32_simt       fp32 CUDA-core kernel (ops.fp32_tc(False))
  bf16_simt       bf16 CUDA-core kernel (Tk > 4096, Tk == 1, or an output row stride that is not a multiple of 8)
Each call checks which kernel ran: the host-side dispatch rules are mirrored below and the CUDA-core launch counter must agree with them.

The tolerance is computed per element from the reference.  With p_j the reference weights and n the live keys of the row:
  fp32 routes:  |err| <= C_FP32 2^-24 (|ref| + (sqrt(n) + L) sum_j p_j |v_j|),   L = scale max_j sum_d |q_d k_jd|  (logit conditioning)
  bf16 routes:  |err| <= C_BF16 (2^-8 |ref| + 2^-9 sum_j p_j |v_j|)  + the fp32 term
2^-8 |ref| is the rounding of the bf16 output and 2^-9 sum p |v| the rounding of P to bf16 before P.V.  Rows whose only live key is the null
key (every real key masked, or Tk == 1) must give v_null exactly on the bf16 routes and within one ulp on the fp32 routes.

Probes: uniform weights (q = 0, V = +-1 with column sums in -2..2, so any key dropped or counted twice moves the output by ~1/n while the
tolerance is ~2^-8 |ref|), one dominant key at each block edge, sentinels in masked and padding rows (Tk_alloc well above Tk), masks whose
only live key sits on a 32-key chunk edge or in the tail, logit bounds (attained, 4x loose, |q.k| ~ 3 with q_scale k_scale != 1, and
2 bound scale log2e just below / above 100), kv_batch_stride_zero, a strided output with rows past B*Tq, and bitwise reproducibility.
MMG_ATTN_KB (read once per process) is exercised in child processes.  The CPU tests at the end show that the comparison rejects outputs with
a key dropped, a key counted twice, V one row off K, or a masked / padding row leaking at weight 2^-10, at every shape used here."""
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BF, F32 = torch.bfloat16, torch.float32
SCALE = 8.0
C_BF16, C_FP32 = 2.0, 8.0
V_SENT = 256.0          # V of masked and padding rows in the leak and mask probes
K_SENT = 16.0           # K of padding rows in the leak probe: |q.k| up to 128, so a padding key that gets any weight dominates its row
OUT_SENT = -1234.0      # output elements the call does not own
DEV = "cuda"
LEAK_PAD = 264          # padding rows of the leak probe: more than the largest key block, so the last block's TMA box reads only padding

ROUTES = ("bf16_tc_2pass", "bf16_tc_1pass", "fp32_split", "fp32_simt", "bf16_simt")
SIMT_ROUTES = ("fp32_simt", "bf16_simt")
REAL_KEYS = (1, 31, 32, 33, 64, 65, 96, 640, 641, 672, 700, 767, 1100, 4095)
TQS = (1, 127, 128, 129, 383)
FORCED_REAL_KEYS = (1, 31, 33, 96, 256, 257, 300, 480, 700, 1100, 4095)     # with MMG_ATTN_KB = 32 / 256: every tail width of a 256-key block
THRESHOLD_BOUNDS = (4.3125, 4.34375)    # bf16-exact; 2 bound 8 log2e = 99.55 (single pass) and 100.27 (two passes)


# ------------------------------------------------------------------------------------------------ dispatch rules (host side, mirrored)
def tc_blocks(Tk):
    """attn_blocks (mmg_attention_tc.cuh): key block KB over the Tk - 1 real keys; MMG_ATTN_KB forces it."""
    try:
        forced = int(os.environ.get("MMG_ATTN_KB", "0"))
    except ValueError:
        forced = 0
    kb = forced or (64 if Tk - 1 <= 640 else 128)
    return kb if kb in (32, 64, 128, 160, 256) else 64


def expected_route(dtype, Tk, ldo, bound, fp32_tc=True):
    """ops.attention + mmg_attention + attention_tc_supported (pointers are 16-byte aligned here)."""
    if dtype == F32:
        return "fp32_split" if fp32_tc and 2 <= Tk <= 4096 and ldo % 8 == 0 else "fp32_simt"
    if not (2 <= Tk <= 4096 and ldo % 8 == 0):
        return "bf16_simt"
    sl2e = np.float32(SCALE) * np.float32(1.4426950408889634)
    single = bound > 0 and np.float32(2) * np.float32(bound) * sl2e < np.float32(100)
    return "bf16_tc_1pass" if single else "bf16_tc_2pass"


def kind_of(route):
    return "fp32" if route.startswith("fp32") else "bf16"


def key_rows(route, Tk):
    """{label: key row} at the block edges of `route` (row 0 = the null key).  The tcgen05 kernel blocks the real keys (rows 1 .. Tk-1) by
    KB, the split kernel all rows by 64, the CUDA-core kernel all rows by 32."""
    if route.startswith("bf16_tc"):
        kb, Tr = tc_blocks(Tk), Tk - 1
        rows = dict(first=1, block_end=kb if Tr >= kb else -1, tail_start=1 + ((Tr - 1) // kb) * kb, last=Tk - 1, null=0)
    else:
        kb = 64 if route == "fp32_split" else 32
        rows = dict(first=1, block_end=kb - 1 if Tk >= kb else -1, tail_start=((Tk - 1) // kb) * kb, last=Tk - 1, null=0)
    out, seen = {}, set()
    for name, r in rows.items():
        if 0 <= r < Tk and r not in seen:
            out[name] = r
            seen.add(r)
    return out


def chunk_edge_rows(route, Tk):
    """the last key of the first 32-key liveness chunk and the first key of the second, plus the block-edge real keys"""
    off = 1 if route.startswith("bf16_tc") else 0
    rows = {31 + off, 32 + off} | set(key_rows(route, Tk).values())
    return sorted(r for r in rows if 1 <= r < Tk)


def route_cases(route):
    """(Tk, Tq, heads, B) for one route: every real-key count it can reach, Tq / heads / B rotated so that each value appears on it."""
    tks = [t + 1 for t in REAL_KEYS] + ([4097, 1] if route in SIMT_ROUTES else [])
    r = ROUTES.index(route)
    return [(Tk, TQS[(i + r) % 5], (1, 8)[(i + r) % 2], 1 + (i + r) % 3) for i, Tk in enumerate(tks)]


def ldo_pad(route, i, Tk):
    """output row stride = heads * 64 + pad; the bf16 CUDA-core route is reached at 2 <= Tk <= 4096 through a stride that is not a multiple of 8"""
    if route == "bf16_simt" and 2 <= Tk <= 4096:
        return (4, 1)[i % 2]
    return i % 2 * {"bf16_tc_2pass": 64, "bf16_tc_1pass": 64, "fp32_split": 8, "fp32_simt": 3, "bf16_simt": 64}[route]


# ------------------------------------------------------------------------------------------------ probe inputs
class Case:
    """Inputs of one mmg_attention call: q [B*heads, Tq, 64]; k, v [(B or 1)*heads, Tk_alloc, 64]; mask [B, Tk-1] bool or None."""

    def __init__(self, q, k, v, B, heads, Tk, mask=None, kv_shared=False, bound=0.0, pterm="all"):
        self.q, self.k, self.v, self.B, self.heads, self.Tk = q.contiguous(), k.contiguous(), v.contiguous(), B, heads, Tk
        self.mask, self.kv_shared, self.bound, self.pterm = mask, kv_shared, bound, pterm


def _gen(seed, device):
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    return g


def _alloc(Tk, extra=0):
    return (Tk + 1 + extra + 7) // 8 * 8          # at least one padding row


def _live(c):
    live = torch.ones((c.B, c.Tk), dtype=torch.bool, device=c.q.device)
    if c.mask is not None:
        live[:, 1:] = c.mask
    return live


def _f32_up(x):
    f = np.float32(x)
    return float(f if float(f) >= x else np.nextafter(f, np.float32(np.inf)))


def true_max(c):
    """max |q.k| over the live keys, rounded up to fp32 (the bound the logits attain)"""
    q = c.q.double().view(c.B, c.heads, -1, 64)
    k = c.k[:, :c.Tk].double().view(-1, c.heads, c.Tk, 64)
    s = (q @ k.transpose(-1, -2)).abs().masked_fill(~_live(c)[:, None, None, :], 0)
    return _f32_up(float(s.max()))


def probe_random(shape, dtype, device, seed, masked=False, kv_shared=False, scaled=True, loose=False):
    """scaled: queries and keys around 16 shared directions, times per-channel scales whose products are ~3 (|q.k| up to ~3 as in a
    trained model, peaked softmax rows), bound = max_i |q_scale_i k_scale_i| as the model passes it.  Otherwise l2-normalised q, k and
    (loose) a bound of 4x the largest |q.k|.  Padding rows are zero."""
    Tk, Tq, heads, B = shape
    g, kvb, alloc = _gen(seed, device), 1 if kv_shared else B, _alloc(Tk)
    rn = lambda *s: torch.randn(s, generator=g, device=device)
    bound = 0.0
    if scaled:
        cen = F.normalize(rn(16, 64), dim=-1)
        qi = torch.randint(0, 16, (B * heads, Tq), generator=g, device=device)
        ki = torch.randint(0, 16, (kvb * heads, alloc), generator=g, device=device)
        qs = 2.0 ** (torch.rand(64, generator=g, device=device) * 2 - 1)
        ks = 3.0 / qs * (0.9 + 0.2 * torch.rand(64, generator=g, device=device))
        q = F.normalize(cen[qi] + 0.3 * rn(B * heads, Tq, 64), dim=-1) * qs
        k = F.normalize(cen[ki] + 0.3 * rn(kvb * heads, alloc, 64), dim=-1) * ks
        bound = _f32_up(float((qs * ks).abs().max()))
    else:
        q, k = F.normalize(rn(B * heads, Tq, 64), dim=-1), F.normalize(rn(kvb * heads, alloc, 64), dim=-1)
    v = rn(kvb * heads, alloc, 64)
    k[:, Tk:] = 0
    v[:, Tk:] = 0
    mask = torch.rand((B, Tk - 1), generator=g, device=device) > 0.4 if masked and Tk > 1 else None
    c = Case(q.to(dtype), k.to(dtype), v.to(dtype), B, heads, Tk, mask, kv_shared, bound)
    if not scaled:
        c.bound = 4 * true_max(c) if loose else true_max(c)
    return c


def probe_uniform(shape, dtype, device, seed, kv_shared=False):
    """q = 0: every live key weighs the same and the output is the mean of the V rows.  V = +-1 with column sums in -2..2 over the Tk
    rows, so dropping or repeating any key moves an output element by ~1/n against a tolerance of ~2^-8 |ref| ~ 2^-8 / n.  The P rounding
    term of the tolerance is only the null key's (it is weighted in fp32, the real keys all carry the same rounded weight)."""
    Tk, Tq, heads, B = shape
    g, kvb, alloc = _gen(seed, device), 1 if kv_shared else B, _alloc(Tk)
    k = F.normalize(torch.randn((kvb * heads, alloc, 64), generator=g, device=device), dim=-1)
    k[:, Tk:] = 0
    m = torch.randint(-1, 2, (kvb * heads, 1, 64), generator=g, device=device) * 2 + Tk % 2     # sums with the parity of Tk
    m = torch.where(m.abs() > 2, m - 2 * m.sign(), m)
    rank = torch.rand((kvb * heads, Tk, 64), generator=g, device=device).argsort(1).argsort(1)
    v = torch.zeros((kvb * heads, alloc, 64), device=device)
    v[:, :Tk] = torch.where(rank < (Tk + m) // 2, 1.0, -1.0)
    q = torch.zeros((B * heads, Tq, 64), device=device)
    return Case(q.to(dtype), k.to(dtype), v.to(dtype), B, heads, Tk, None, kv_shared, 1.0, pterm="null")


def probe_dominant(shape, dtype, device, seed, row):
    """q = 4 k_row for every query of a (batch, head): the logit of key `row` is 32, the others ~N(0, 4), so the output is v_row to
    ~1e-4 and a block offset or a V row off by one shows as a different V row.  The bound is attained exactly."""
    Tk, Tq, heads, B = shape
    g, alloc = _gen(seed, device), _alloc(Tk)
    k = F.normalize(torch.randn((B * heads, alloc, 64), generator=g, device=device), dim=-1).to(dtype)
    v = torch.randn((B * heads, alloc, 64), generator=g, device=device).to(dtype)
    k[:, Tk:] = 0
    v[:, Tk:] = 0
    q = (4 * k[:, row:row + 1].float()).expand(-1, Tq, -1).to(dtype)
    c = Case(q, k, v, B, heads, Tk)
    c.bound = true_max(c)
    return c


def probe_leak(shape, dtype, device, seed):
    """Tk_alloc = Tk + ~LEAK_PAD; padding rows hold K_SENT / V_SENT, masked keys (~half) hold V_SENT.  Any weight on those rows shows."""
    Tk, Tq, heads, B = shape
    g, alloc = _gen(seed, device), _alloc(Tk, LEAK_PAD)
    q = F.normalize(torch.randn((B * heads, Tq, 64), generator=g, device=device), dim=-1)
    k = F.normalize(torch.randn((B * heads, alloc, 64), generator=g, device=device), dim=-1)
    v = torch.randn((B * heads, alloc, 64), generator=g, device=device)
    k[:, Tk:] = K_SENT
    v[:, Tk:] = V_SENT
    mask = None
    if Tk > 1:
        mask = torch.rand((B, Tk - 1), generator=g, device=device) > 0.5
        v4 = v.view(B, heads, alloc, 64)
        v4[:, :, 1:Tk] = torch.where(mask[:, None, :, None], v4[:, :, 1:Tk], V_SENT)
    c = Case(q.to(dtype), k.to(dtype), v.to(dtype), B, heads, Tk, mask)
    c.bound = true_max(c)
    return c


def probe_masks(shape, dtype, device, seed, rows):
    """One batch entry with every real key masked, then one per row in `rows` whose only live real key is that row (batch entries in
    groups of at most 3).  Masked keys hold V_SENT."""
    Tk, Tq, heads, _ = shape
    entries, cases = [None] + list(rows), []
    for gi in range(0, len(entries), 3):
        grp = entries[gi:gi + 3]
        B = len(grp)
        c = probe_random((Tk, Tq, heads, B), dtype, device, seed + gi, scaled=False)
        mask = torch.zeros((B, Tk - 1), dtype=torch.bool, device=device)
        for b, r in enumerate(grp):
            if r is not None:
                mask[b, r - 1] = True
        v4 = c.v.view(B, heads, -1, 64)
        v4[:, :, 1:Tk] = torch.where(mask[:, None, :, None], v4[:, :, 1:Tk], torch.tensor(V_SENT, dtype=dtype, device=device))
        c.mask = mask
        c.bound = true_max(c)
        cases.append(c)
    return cases


def probe_threshold(shape, dtype, device, seed, bound):
    """Every logit of every row in [-bound, -bound + 0.25] (q = e_0, k_j = -b_j e_0, b_j bf16-exact, the null key and some keys at
    b_j = bound): a single-pass softmax scales these rows by 2^(-2 bound scale log2e) ~ 2^-100 and must not underflow."""
    Tk, Tq, heads, B = shape
    g, alloc = _gen(seed, device), _alloc(Tk)
    q = torch.zeros((B * heads, Tq, 64), device=device)
    q[..., 0] = 1.0
    b = bound - 2.0 ** -5 * torch.randint(0, 9, (B * heads, alloc), generator=g, device=device)
    b[:, 0] = bound
    k = torch.zeros((B * heads, alloc, 64), device=device)
    k[..., 0] = -b
    v = torch.randn((B * heads, alloc, 64), generator=g, device=device)
    k[:, Tk:] = 0
    v[:, Tk:] = 0
    return Case(q.to(dtype), k.to(dtype), v.to(dtype), B, heads, Tk, None, False, bound)


# ------------------------------------------------------------------------------------------------ reference and comparison
class Ref:
    pass


def _rows(t):
    """[B, heads, Tq, 64] -> the output layout [B*Tq, heads*64]"""
    B, H, Tq, D = t.shape
    return t.permute(0, 2, 1, 3).reshape(B * Tq, H * D)


def reference(c, keep_p=False):
    """float64 softmax(scale q k^T, masked_fill(~mask, -finfo.max)) v over keys 0 .. Tk-1, plus what the tolerance needs"""
    B, H, Tk = c.B, c.heads, c.Tk
    q = c.q.double().view(B, H, -1, 64)
    k = c.k[:, :Tk].double().view(-1, H, Tk, 64)
    v = c.v[:, :Tk].double().view(-1, H, Tk, 64)
    live = _live(c)[:, None, None, :]
    s = (SCALE * (q @ k.transpose(-1, -2))).masked_fill(~live, -torch.finfo(torch.float64).max)
    p = s.softmax(-1)
    r = Ref()
    out = p @ v
    pav = p @ v.abs()
    L = (SCALE * (q.abs() @ k.abs().transpose(-1, -2))).masked_fill(~live, 0).amax(-1, keepdim=True)
    n = live.sum(-1, keepdim=True).double()
    vnull = v[:, :, :1].expand_as(out)
    r.out, r.pav = _rows(out), _rows(pav)
    r.absout = r.out.abs()
    r.depth = _rows((n.sqrt() + L).expand_as(out))
    r.pnull = _rows(p[..., :1] * (vnull.abs() + out.abs()))
    r.vnull = _rows(vnull)
    r.dead = _rows((n == 1).expand_as(out))
    if keep_p:
        r.p, r.v4 = p, v
    return r


def tolerance(r, kind, pterm="all"):
    t = C_FP32 * 2.0 ** -24 * (r.absout + r.depth * r.pav)
    if kind == "bf16":
        t = t + C_BF16 * (2.0 ** -8 * r.absout + 2.0 ** -9 * (r.pav if pterm == "all" else r.pnull))
    return t


def compare(got, r, kind, pterm="all"):
    """(ok, worst err / tolerance, message) for an output `got` in the layout [B*Tq, heads*64]"""
    g = got.double()
    if not bool(torch.isfinite(g).all()):
        return False, math.inf, f"{int((~torch.isfinite(g)).sum())} non-finite output elements"
    err = (g - r.out).abs()
    ratio = torch.where(err == 0, torch.zeros_like(err), err / tolerance(r, kind, pterm))
    worst = float(ratio.max())
    i = np.unravel_index(int(ratio.argmax()), tuple(ratio.shape))
    msg = f"worst err/tol {worst:.3g} at {tuple(int(x) for x in i)}: got {float(g[i]):.6g}, ref {float(r.out[i]):.6g}"
    ok = worst <= 1.0
    if bool(r.dead.any()):      # only the null key is live: exactly v_null (bf16), within one ulp (fp32)
        gd, vn = g[r.dead], r.vnull[r.dead]
        if kind == "bf16":
            exact = bool(torch.equal(gd, vn))
        else:
            a = vn.float().abs()
            exact = bool(((gd - vn).abs() <= (torch.nextafter(a, torch.full_like(a, math.inf)) - a).double()).all())
        if not exact:
            ok, msg = False, msg + f"; rows with only the null key live differ from v_null by up to {float((gd - vn).abs().max()):.3g}"
    return ok, worst, msg


# ------------------------------------------------------------------------------------------------ running the kernels
def launch(c, fp32_tc=True, pad=0, extra_rows=3):
    """ops.attention into an output buffer [B*Tq + extra_rows, heads*64 + pad] pre-filled with OUT_SENT.  Returns (owned block, whole
    buffer, route); asserts the route against the CUDA-core launch counter and that nothing outside the owned block changed."""
    from muse_maskgit_pytorch_b200 import ops, _lib
    dtype, Tq, width = c.q.dtype, c.q.shape[1], c.heads * 64
    buf = torch.full((c.B * Tq + extra_rows, width + pad), OUT_SENT, dtype=dtype, device=c.q.device)
    before = buf.clone()
    route = expected_route(dtype, c.Tk, width + pad, c.bound, fp32_tc)
    mask = None if c.mask is None else c.mask.to(torch.uint8).contiguous()
    n0, prev = _lib.simt_launch_count(), ops.fp32_tc()
    try:
        ops.fp32_tc(fp32_tc)
        ops.attention(c.q, c.k, c.v, buf, c.B, c.heads, c.Tk, key_mask=mask, kv_shared=c.kv_shared, scale=SCALE, logit_bound=c.bound)
    finally:
        ops.fp32_tc(prev)
    torch.cuda.synchronize()
    simt = _lib.simt_launch_count() - n0
    assert simt == (route in SIMT_ROUTES), f"expected route {route}, but {simt} CUDA-core attention launches"
    rows = c.B * Tq
    assert torch.equal(buf[rows:], before[rows:]), "rows past B*Tq were written"
    assert torch.equal(buf[:, width:], before[:, width:]), "columns past heads*64 were written"
    return buf[:rows, :width], buf, route


class Record:
    """per route: shapes run, probes run, worst err / tolerance; failures"""

    def __init__(self):
        self.routes, self.failures = {}, []

    def add(self, route, probe, shape, ratio):
        e = self.routes.setdefault(route, dict(shapes=[], probes={}, worst=(0.0, "")))
        if shape not in e["shapes"]:
            e["shapes"].append(shape)
        e["probes"][probe] = e["probes"].get(probe, 0) + 1
        if ratio > e["worst"][0]:
            e["worst"] = (ratio, f"{probe} at (Tk, Tq, heads, B, ldo) = {shape}")

    def summary(self):
        lines = []
        for route, e in self.routes.items():
            lines.append(f"{route}: {len(e['shapes'])} shapes (Tk, Tq, heads, B, ldo): " + " ".join(str(s).replace(" ", "") for s in e["shapes"]))
            lines.append(f"  probes: " + ", ".join(f"{p} x{n}" for p, n in e["probes"].items()))
            lines.append(f"  worst err/tol {e['worst'][0]:.3f} ({e['worst'][1]})")
        return "\n".join(lines)


def run_probe(rec, route, probe, c, fp32_tc, pad, repro=False):
    """one call of `c` on `route`: route, result against the reference, untouched output, optionally bitwise repeatability"""
    shape = (c.Tk, c.q.shape[1], c.heads, c.B, c.heads * 64 + pad)
    where = f"{route} {probe} (Tk, Tq, heads, B, ldo) = {shape}"
    try:
        if route != "bf16_tc_1pass" and probe != "threshold":
            c.bound = 0.0
        got, buf, taken = launch(c, fp32_tc, pad)
        assert taken == route, f"dispatch chose {taken}"
        ok, ratio, msg = compare(got, reference(c), kind_of(route), c.pterm)
        rec.add(route, probe, shape, ratio)
        assert ok, msg
        if repro:
            _, buf2, _ = launch(c, fp32_tc, pad)
            assert torch.equal(buf, buf2), "two identical calls differ"
    except AssertionError as e:
        rec.failures.append(f"{where}: {e}")


def run_route_case(rec, route, i, shape):
    Tk = shape[0]
    dtype = F32 if route.startswith("fp32") else BF
    fp32_tc, pad, seed = route != "fp32_simt", ldo_pad(route, i, Tk), 7919 * (ROUTES.index(route) + 1) + 31 * i
    go = lambda probe, c, **kw: run_probe(rec, route, probe, c, fp32_tc, pad, **kw)
    go("random", probe_random(shape, dtype, DEV, seed, masked=i % 2 == 1), repro=True)
    go("random kv_shared", probe_random(shape, dtype, DEV, seed + 1, masked=i % 2 == 0, kv_shared=True))
    if route == "bf16_tc_1pass":
        go("random loose bound", probe_random(shape, dtype, DEV, seed + 2, masked=i % 2 == 1, scaled=False, loose=True))
    go("uniform", probe_uniform(shape, dtype, DEV, seed + 3, kv_shared=i % 2 == 1))
    for name, row in key_rows(route, Tk).items():
        go(f"dominant {name}", probe_dominant(shape, dtype, DEV, seed + 4 + row, row))
    go("leak", probe_leak(shape, dtype, DEV, seed + 5))
    if Tk > 1:
        for c in probe_masks(shape, dtype, DEV, seed + 6, chunk_edge_rows(route, Tk)):
            go("masks", c)


@pytest.mark.gpu
@pytest.mark.parametrize("route", ROUTES)
def test_route(route):
    torch.set_grad_enabled(False)
    rec = Record()
    for i, shape in enumerate(route_cases(route)):
        run_route_case(rec, route, i, shape)
        if route == "bf16_tc_1pass" and i % 3 == 0:
            for bound in THRESHOLD_BOUNDS:
                c = probe_threshold(shape, BF, DEV, 17 + i, bound)
                run_probe(rec, expected_route(BF, c.Tk, c.heads * 64, bound), "threshold", c, True, 0)
    print(rec.summary())
    assert not rec.failures, f"{len(rec.failures)} failures:\n" + "\n".join(rec.failures[:60])


def forced_kb_main(kb):
    """Entry of the child process with MMG_ATTN_KB = kb: both tcgen05 routes at FORCED_REAL_KEYS."""
    assert tc_blocks(2) == kb, "MMG_ATTN_KB is not set to the key block under test"
    torch.set_grad_enabled(False)
    rec = Record()
    for r, route in enumerate(ROUTES[:2]):
        for i, Tr in enumerate(FORCED_REAL_KEYS):
            run_route_case(rec, route, i, (Tr + 1, TQS[(i + r) % 5], (1, 8)[(i + r) % 2], 1 + (i + r) % 3))
    print(f"MMG_ATTN_KB={kb}\n" + rec.summary())
    for f in rec.failures[:60]:
        print("FAIL", f)
    return 1 if rec.failures else 0


@pytest.mark.gpu
@pytest.mark.parametrize("kb", [32, 256])
def test_forced_key_blocks(kb):
    """MMG_ATTN_KB is read once per process: one child process per key block (32: 128-column TMEM with 32-key blocks; 256: the
    512-column TMEM kernel), running the same probes as test_route."""
    code = (f"import sys; sys.path.insert(0, {ROOT!r}); from tests import test_gpu_attention_edges as t; "
            f"sys.exit(t.forced_kb_main({kb}))")
    env = dict(os.environ, MMG_ATTN_KB=str(kb))
    p = subprocess.run([sys.executable] + subprocess._args_from_interpreter_flags() + ["-c", code], cwd=ROOT, env=env,
                       capture_output=True, text=True, timeout=600)
    print(p.stdout)
    assert p.returncode == 0, f"exit {p.returncode}\n{p.stdout[-6000:]}\n{p.stderr[-4000:]}"


# ------------------------------------------------------------------------------------------------ the comparison rejects defects (CPU)
def _all_shapes():
    return sorted({s for route in ROUTES for s in route_cases(route)})


def _defect_rows(Tk):
    return sorted({r for route in ROUTES for r in key_rows(route, Tk).values()})


def _mix(r, p_extra, v_extra, sign):
    """reference output with one extra (sign +1) or one fewer (sign -1) copy of a key of weight p_extra and value v_extra"""
    return (r.p @ r.v4 + sign * p_extra * v_extra) / (1 + sign * p_extra)


def _rejected(out4, r, pterm="all"):
    return [k for k in ("bf16", "fp32") if compare(_rows(out4), r, k, pterm)[0]]


@pytest.mark.parametrize("shape", _all_shapes(), ids=lambda s: "Tk%d-Tq%d-h%d-B%d" % s)
def test_checker_rejects_defects(shape):
    """Defective outputs computed from the float64 reference must fail the comparison the GPU tests use, under both tolerances; the
    correctly rounded reference must pass it."""
    torch.set_grad_enabled(False)
    torch.manual_seed(0)
    Tk = shape[0]
    u = probe_uniform(shape, BF, "cpu", 5)
    r = reference(u, keep_p=True)
    for kind, dt in (("bf16", BF), ("fp32", F32)):
        ok, ratio, msg = compare(r.out.to(dt), r, kind, u.pterm)
        assert ok, f"correctly rounded reference rejected ({kind}): {msg}"
    vfull = u.v.double().view(-1, u.heads, u.v.shape[1], 64)
    bad = []
    for j in _defect_rows(Tk) if Tk > 1 else []:      # with one key there is nothing to drop and doubling it changes nothing
        pj, vj = r.p[..., j:j + 1], r.v4[:, :, j:j + 1]
        bad += [(f"key {j} dropped", _rejected(_mix(r, pj, vj, -1), r, u.pterm)),
                (f"key {j} counted twice", _rejected(_mix(r, pj, vj, 1), r, u.pterm))]
    bad += [("V one row off K (uniform)", _rejected(r.p @ vfull[:, :, 1:Tk + 1], r, u.pterm))]
    for name, row in key_rows("bf16_tc_2pass", Tk).items():
        d = probe_dominant(shape, BF, "cpu", 6 + row, row)
        rd = reference(d, keep_p=True)
        vd = d.v.double().view(-1, d.heads, d.v.shape[1], 64)
        bad += [(f"V one row off K (dominant {name})", _rejected(rd.p @ vd[:, :, 1:Tk + 1], rd))]
    lk = probe_leak(shape, BF, "cpu", 7)
    rl = reference(lk, keep_p=True)
    vl = lk.v.double().view(lk.B, lk.heads, -1, 64)
    leak_rows = [Tk] + ([1 + int(torch.nonzero(~lk.mask[0])[0])] if lk.mask is not None and not bool(lk.mask[0].all()) else [])
    for row in leak_rows:
        w = 2.0 ** -10
        bad += [(f"row {row} leaks at 2^-10", _rejected((1 - w) * (rl.p @ rl.v4) + w * vl[:, :, row:row + 1], rl))]
    accepted = [(name, kinds) for name, kinds in bad if kinds]
    assert not accepted, f"defects accepted: {accepted}"
