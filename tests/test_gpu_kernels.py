"""GPU parity tests, kernel by kernel, through the C-ABI (libmmg.so) against CPU torch / the oracle.
bf16 operands are generated as bf16-representable values, so the CPU fp32 reference sees exactly the same inputs and the
only difference left is fp32 accumulation order (tolerances below reflect that, not bf16 rounding)."""
import math
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import synth, muse_oracle as O

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)


def ops():
    from muse_maskgit_pytorch_b200 import ops as _ops
    return _ops


def rnd(name, shape, dtype=torch.float32, std=1.0):
    t = torch.from_numpy(synth.normal(name, shape, 3, std))
    return t.to(torch.bfloat16).float() if dtype == torch.bfloat16 else t


def dev(t, dtype=None):
    return t.cuda().to(dtype) if dtype is not None else t.cuda()


def close(a, b, atol, rtol=1e-3):
    a, b = a.float().cpu(), b.float().cpu()
    err = (a - b).abs()
    ok = bool((err <= atol + rtol * b.abs()).all())
    return ok, f"max abs err {err.max().item():.3e} at {np.unravel_index(int(err.argmax()), a.shape)} (ref max {b.abs().max().item():.3e}, mean err {err.mean().item():.3e})"


# ------------------------------------------------------------------------------------------------ GEMM
@pytest.mark.parametrize("M,N,K", [(128, 128, 64), (256, 512, 512), (300, 192, 128), (2048, 2816, 512), (512, 4096, 512), (4096, 512, 1408), (70, 64, 192)])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32], ids=["bf16", "fp32"])
def test_linear_store(M, N, K, dtype):
    a, w = rnd(f"a{M}{K}", (M, K), dtype), rnd(f"w{N}{K}", (N, K), dtype, std=K ** -0.5)
    out = torch.empty((M, N), device="cuda", dtype=torch.float32)
    ops().linear(dev(a, dtype), dev(w, dtype), out)
    ok, msg = close(out, a @ w.t(), 2e-4)
    assert ok, msg


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32], ids=["bf16", "fp32"])
def test_linear_bias_act_bf16_out(dtype):
    M, N, K = 384, 256, 256
    a, w, bias = rnd("a", (M, K), dtype), rnd("w", (N, K), dtype, std=K ** -0.5), rnd("b", (N,))
    out = torch.empty((M, N), device="cuda", dtype=dtype)
    ops().linear(dev(a, dtype), dev(w, dtype), out, bias=dev(bias), act=1)
    ref = F.leaky_relu(a @ w.t() + bias, 0.1)
    ok, msg = close(out, ref, 2e-2 if dtype == torch.bfloat16 else 2e-4, 1e-2 if dtype == torch.bfloat16 else 1e-3)
    assert ok, msg


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32], ids=["bf16", "fp32"])
def test_linear_residual_inplace(dtype):
    M, N, K = 512, 512, 512
    a, w, x = rnd("a", (M, K), dtype), rnd("w", (N, K), dtype, std=K ** -0.5), rnd("x", (M, N))
    xd = dev(x)
    ops().linear(dev(a, dtype), dev(w, dtype), xd, epilogue=ops().EPI_RESIDUAL, resid=xd)
    ok, msg = close(xd, a @ w.t() + x, 3e-4)
    assert ok, msg


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32], ids=["bf16", "fp32"])
def test_linear_geglu(dtype):
    """W rows interleaved [x(32) | gate(32)]: out[:, u] = gate_u * gelu(x_u)  (ref: muse_maskgit_pytorch.py:76-77)."""
    M, K, Fu = 256, 128, 96
    a = rnd("a", (M, K), dtype)
    wx, wg = rnd("wx", (Fu, K), dtype, std=K ** -0.5), rnd("wg", (Fu, K), dtype, std=K ** -0.5)
    w = torch.stack((wx.view(-1, 32, K), wg.view(-1, 32, K)), 1).reshape(2 * Fu, K)
    out = torch.empty((M, Fu), device="cuda", dtype=torch.float32)
    # out is written at column c/2: ldo = Fu
    e = ops()._epi(out, Fu)
    ops().linear(dev(a, dtype), dev(w, dtype), None, epilogue=ops().EPI_GEGLU, epi=e)
    ref = (a @ wg.t()) * F.gelu(a @ wx.t())
    ok, msg = close(out, ref, 3e-4)
    assert ok, msg


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32], ids=["bf16", "fp32"])
def test_linear_qkv_epilogue(dtype):
    """fused head split + l2norm * scale + null key/value row  (ref: muse_maskgit_pytorch.py:141-153)."""
    b, n, heads, dim = 3, 20, 2, 128
    inner = heads * 64
    x = rnd("x", (b * n, dim), dtype)
    w = rnd("wqkv", (3 * inner, dim), dtype, std=dim ** -0.5)
    qs, ks = 1 + 0.1 * rnd("qs", (64,)), 1 + 0.1 * rnd("ks", (64,))
    nk, nv = rnd("nk", (heads, 64), dtype), rnd("nv", (heads, 64), dtype)
    q = torch.zeros((b * heads, n, 64), device="cuda", dtype=dtype)
    k = torch.zeros((b * heads, n + 4, 64), device="cuda", dtype=dtype)
    v = torch.zeros_like(k)
    qsd, ksd, nkd, nvd = dev(qs), dev(ks), dev(nk, dtype), dev(nv, dtype)      # keep alive: the epilogue block holds raw pointers
    e = ops().qkv_epilogue(dtype, heads, n, q=q, k=k, v=v, q_scale=qsd, k_scale=ksd, key_off=1, null_k=nkd, null_v=nvd)
    ops().linear(dev(x, dtype), dev(w, dtype), None, epilogue=ops().EPI_QKV, epi=e)
    y = (x @ w.t()).view(b, n, 3, heads, 64).permute(2, 0, 3, 1, 4)          # (3, b, h, n, 64)
    qr = F.normalize(y[0], dim=-1) * qs
    kr = F.normalize(y[1], dim=-1) * ks
    tol = 2e-2 if dtype == torch.bfloat16 else 1e-5
    for got, ref, name in ((q.view(b, heads, n, 64), qr, "q"), (k.view(b, heads, n + 4, 64)[:, :, 1:n + 1], kr, "k"), (v.view(b, heads, n + 4, 64)[:, :, 1:n + 1], y[2], "v")):
        ok, msg = close(got, ref, tol, 1e-2)
        assert ok, name + ": " + msg
    assert torch.equal(k.view(b, heads, n + 4, 64)[:, :, 0].float().cpu(), nk.expand(b, -1, -1))
    assert torch.equal(v.view(b, heads, n + 4, 64)[:, :, 0].float().cpu(), nv.expand(b, -1, -1))
    assert float(k.view(b, heads, n + 4, 64)[:, :, n + 1:].abs().max()) == 0.


# ------------------------------------------------------------------------------------------------ row kernels
@pytest.mark.parametrize("width,ld", [(512, 512), (1365, 1408), (128, 128)])
def test_layernorm(width, ld):
    rows = 77
    x = torch.zeros((rows, ld)); x[:, :width] = rnd("x", (rows, width)) * 2 + 0.5
    g = 1 + 0.1 * rnd("g", (width,))
    gp = torch.zeros(ld); gp[:width] = g
    y = torch.empty((rows, ld), device="cuda", dtype=torch.float32)
    ops().layernorm(dev(x), dev(gp), y, width=width)
    ref = F.layer_norm(x[:, :width], (width,), g, None)
    ok, msg = close(y[:, :width], ref, 2e-5)
    assert ok, msg
    assert float(y[:, width:].abs().max()) == 0. if ld > width else True
    # add + write-back variant (constant null-CFG cross-attention term)
    add = rnd("add", (width,))
    xd = dev(x[:, :width].contiguous()); y2 = torch.empty((rows, width), device="cuda", dtype=torch.bfloat16)
    ops().layernorm(xd, dev(g), y2, add=dev(add), x_out=xd)
    ok, msg = close(xd, x[:, :width] + add, 1e-6)
    assert ok, msg
    ok, msg = close(y2, F.layer_norm(x[:, :width] + add, (width,), g, None), 2e-2, 1e-2)
    assert ok, msg


def test_embed_and_final_embed():
    V, dim, n, b = 50, 128, 16, 3
    tok, pos = rnd("tok", (V + 1, dim)), rnd("pos", (n, dim))
    ids = torch.from_numpy((synth.uniform("ids", (b, n)) * (V + 1)).astype(np.int64))
    x = torch.empty((2 * b * n, dim), device="cuda")
    ops().embed(dev(ids), dev(tok), dev(pos), x, n=n, copies=2)
    ref = tok[ids] + pos[:n]
    assert torch.equal(x[:b * n].cpu().view(b, n, dim), ref) and torch.equal(x[b * n:].cpu().view(b, n, dim), ref)
    xc, xn = rnd("xc", (b * n, dim)), rnd("xn", (b * n, dim))
    g = 1 + 0.1 * rnd("g", (dim,))
    nm = 5
    mp = torch.stack([torch.sort(torch.randperm(n, generator=torch.Generator().manual_seed(i))[:nm]).values for i in range(b)]).int()
    e = torch.empty((b * nm, dim), device="cuda")
    ops().final_embed(dev(xc), dev(xn), dev(g), dev(mp), e, b, n, nm, 3.0)
    rows = (torch.arange(b)[:, None] * n + mp.long()).reshape(-1)
    lc, ln_ = O.ln(xc[rows], g), O.ln(xn[rows], g)
    ok, msg = close(e, ln_ + (lc - ln_) * 3.0, 1e-5)
    assert ok, msg


# ------------------------------------------------------------------------------------------------ attention
def attn_ref(q, k, v, mask, scale=8.0):
    sim = (q @ k.transpose(-1, -2)) * scale
    if mask is not None:
        km = F.pad(mask, (1, 0), value=True)[:, None, None, :]
        sim = sim.masked_fill(~km, O.NEG_MAX)
    return sim.softmax(-1) @ v


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32], ids=["bf16", "fp32"])
@pytest.mark.parametrize("bound", [0.0, 1.02], ids=["twopass", "singlepass"])
@pytest.mark.parametrize("Tq,Tk,masked", [(256, 257, False), (16, 17, False), (256, 33, True), (64, 81, True), (1024, 1025, False), (200, 290, True)])
def test_attention(dtype, Tq, Tk, masked, bound):
    b, heads = 2, 2
    if Tq == 1024:
        b = 1
    q = F.normalize(rnd("q", (b, heads, Tq, 64)), dim=-1)
    k = F.normalize(rnd("k", (b, heads, Tk, 64)), dim=-1)
    v = rnd("v", (b, heads, Tk, 64))
    if dtype == torch.bfloat16:
        q, k, v = (t.to(torch.bfloat16).float() for t in (q, k, v))
    mask = None
    if masked:
        mask = torch.from_numpy(synth.uniform("m", (b, Tk - 1))) > 0.4
        mask[0, :] = False                                            # one batch entry with every context key masked
    alloc = (Tk + 7) // 8 * 8
    kd = torch.zeros((b * heads, alloc, 64), device="cuda", dtype=dtype); kd[:, :Tk] = dev(k.reshape(b * heads, Tk, 64), dtype)
    vd = torch.zeros_like(kd); vd[:, :Tk] = dev(v.reshape(b * heads, Tk, 64), dtype)
    out = torch.empty((b * Tq, heads * 64), device="cuda", dtype=dtype)
    ops().attention(dev(q.reshape(b * heads, Tq, 64), dtype).contiguous(), kd, vd, out, b, heads, Tk,
                    key_mask=None if mask is None else dev(mask.to(torch.uint8)), logit_bound=bound)
    ref = attn_ref(q, k, v, mask).transpose(1, 2).reshape(b * Tq, heads * 64)
    ok, msg = close(out, ref, 2e-2 if dtype == torch.bfloat16 else 2e-5, 2e-2 if dtype == torch.bfloat16 else 1e-4)
    assert ok, msg
    if masked:   # fully masked context -> output is exactly the null value (SURVEY.md 8a T3)
        got0 = out.view(b, Tq, heads, 64)[0].float().cpu()
        if dtype == torch.bfloat16:
            assert torch.equal(got0, v[0, :, 0][None].expand(Tq, -1, -1))
        else:
            assert torch.allclose(got0, v[0, :, 0][None].expand(Tq, -1, -1), atol=1e-6)


# ------------------------------------------------------------------------------------------------ sampler
def test_remask():
    b, n, nm, mask_id = 4, 256, 97, 1000
    scores = torch.from_numpy(synth.uniform("sc", (b, n)))
    scores[1, 10:40] = 0.75                                            # ties across the boundary: lowest positions win
    ids = torch.from_numpy((synth.uniform("ids", (b, n)) * 1000).astype(np.int64))
    idd, sd = dev(ids.clone()), dev(scores.clone())
    mp = torch.empty((b, n), dtype=torch.int32, device="cuda")
    ops().remask(idd, sd, mp, nm, mask_id)
    order = torch.argsort(-scores, dim=-1, stable=True)[:, :nm]
    ref_set = torch.zeros((b, n), dtype=torch.bool).scatter_(1, order, True)
    got = idd.cpu() == mask_id
    assert torch.equal(got, ref_set)
    assert torch.equal(idd.cpu()[~ref_set], ids[~ref_set])
    assert float(sd.max()) == -1e5 and float(sd.min()) == -1e5
    pos = mp.cpu().view(-1)[:b * nm].view(b, nm).long()          # compact [B, num_masked] list
    assert torch.equal(pos, torch.sort(order, dim=-1).values)


def _sample_case(b, n, nm, V, temp, logits, u=None, seed=5):
    k = O.top_k_count(V, 0.9)
    g = torch.Generator().manual_seed(seed)
    mp = torch.stack([torch.sort(torch.randperm(n, generator=g)[:nm]).values for _ in range(b)]).int()
    ids = torch.full((b, n), V, dtype=torch.long)
    scores = torch.full((b, n), -1e5)
    idd, sd = dev(ids.clone()), dev(scores.clone())
    ops().logits_sample(dev(logits.reshape(b * nm, V).contiguous()), dev(mp), idd, sd, nm, k, temp, u=None if u is None else dev(u))
    return mp, idd.cpu(), sd.cpu(), k


def _oracle_rows(logits, u_rows, temp, k):
    """per-row reference: top-k filter (exactly k kept, ties by lowest index) + gumbel argmax + confidence."""
    R, V = logits.shape
    order = torch.argsort(-logits, dim=-1, stable=True)[:, :k]
    keep = torch.zeros((R, V), dtype=torch.bool).scatter_(1, order, True)
    filt = torch.where(keep, logits, torch.tensor(float("-inf")))
    pert = filt / max(temp, 1e-10) + O.gumbel_from_uniform(u_rows)
    pred = pert.argmax(-1)
    top2 = pert.topk(2, dim=-1).values
    p = logits.softmax(-1).gather(1, pred[:, None])[:, 0]
    return pred, 1 - p, top2[:, 0] - top2[:, 1]


@pytest.mark.parametrize("V,temp", [(65536, 1.0), (65536, 0.0), (1024, 0.5), (8192, 17 / 18), (512, 1.0)])
def test_logits_sample_injected_noise(V, temp):
    b, n, nm = 2, 16, 5
    logits = torch.from_numpy(synth.normal(f"lg{V}", (b, nm, V), 7, 0.58))
    u = torch.from_numpy(synth.uniform(f"u{V}", (b, n, V), 7))
    mp, ids, scores, k = _sample_case(b, n, nm, V, temp, logits, u)
    rows_u = torch.stack([u[bi, mp[bi, j]] for bi in range(b) for j in range(nm)])
    pred, sc, margin = _oracle_rows(logits.reshape(-1, V), rows_u, temp, k)
    got = torch.stack([ids[bi, mp[bi, j]] for bi in range(b) for j in range(nm)])
    gsc = torch.stack([scores[bi, mp[bi, j]] for bi in range(b) for j in range(nm)])
    bad = (got != pred) & (margin > 1e-4)
    assert not bad.any(), f"pred mismatch at rows {bad.nonzero().flatten().tolist()} got {got[bad].tolist()} want {pred[bad].tolist()}"
    same = got == pred
    assert same.float().mean() > 0.8
    assert torch.allclose(gsc[same], sc[same], atol=2e-6)
    untouched = torch.ones((b, n), dtype=torch.bool); untouched.scatter_(1, mp.long(), False)
    assert (ids[untouched] == V).all() and (scores[untouched] == -1e5).all()


def test_logits_sample_adversarial_rows():
    """rows that defeat the sampled threshold: constant rows (all ties), a heavy cluster, few distinct values."""
    b, n, nm, V = 1, 8, 4, 4096
    k = O.top_k_count(V, 0.9)
    base = torch.from_numpy(synth.normal("adv", (V,), 9))
    rows = [torch.zeros(V), torch.where(torch.arange(V) % 7 == 0, base, torch.full((V,), 0.25)),
            torch.round(base * 2) / 2, torch.cat((torch.full((V - 10,), -3.0), torch.arange(10).float()))]
    logits = torch.stack(rows)[None]
    u = torch.from_numpy(synth.uniform("uadv", (b, n, V), 9))
    mp, ids, scores, _ = _sample_case(b, n, nm, V, 1.0, logits, u)
    rows_u = torch.stack([u[0, mp[0, j]] for j in range(nm)])
    pred, sc, margin = _oracle_rows(logits.reshape(-1, V), rows_u, 1.0, k)
    got = torch.stack([ids[0, mp[0, j]] for j in range(nm)])
    assert torch.equal(got[margin > 1e-5], pred[margin > 1e-5]), (got.tolist(), pred.tolist())


def test_logits_sample_philox_is_shard_invariant():
    """in-kernel Philox noise is keyed on the GLOBAL row: a 2-shard run equals the 1-shard run bit for bit."""
    b, n, nm, V = 4, 16, 6, 2048
    k = O.top_k_count(V, 0.9)
    logits = torch.from_numpy(synth.normal("lgp", (b, nm, V), 11, 0.58))
    g = torch.Generator().manual_seed(1)
    mp = torch.stack([torch.sort(torch.randperm(n, generator=g)[:nm]).values for _ in range(b)]).int()

    def run(lo, hi):
        ids = torch.full((hi - lo, n), V, dtype=torch.long, device="cuda"); sc = torch.full((hi - lo, n), -1e5, device="cuda")
        ops().logits_sample(dev(logits[lo:hi].reshape(-1, V).contiguous()), dev(mp[lo:hi].contiguous()), ids, sc, nm, k, 1.0, seed=1234, step=3, row_offset=lo * n)
        return ids.cpu(), sc.cpu()
    full = run(0, b)
    a, c = run(0, 2), run(2, 4)
    assert torch.equal(full[0], torch.cat((a[0], c[0]))) and torch.equal(full[1], torch.cat((a[1], c[1])))
    assert (full[0][full[0] != V] < V).all()


# ------------------------------------------------------------------------------------------------ VQ
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32], ids=["bf16", "fp32"])
def test_vq_lfq_encode_bit_exact(dtype):
    """dyadic inputs: every partial sum is exact in fp32, so ids must be bit-identical in any summation order."""
    T, D, bits = 300, 2048, 16
    x = torch.from_numpy(synth.dyadic("vx", (T, D), bits=4, span=2.0))
    w = torch.from_numpy(synth.dyadic("vw", (bits, D), bits=4, span=1.0))
    bias = torch.from_numpy(synth.dyadic("vb", (bits,), bits=4, span=1.0))
    x[5] = 0.; bias_z = bias.clone()
    ids = torch.empty((T,), dtype=torch.int64, device="cuda")
    ops().vq_lfq_encode(dev(x, dtype), dev(w), dev(bias_z), ids, bits)
    proj = x @ w.t() + bias_z
    ref = ((proj > 0).long() * (2 ** torch.arange(bits - 1, -1, -1))).sum(-1)
    assert torch.equal(ids.cpu(), ref)
    # identity projection (D == bits)
    x2 = torch.from_numpy(synth.dyadic("vx2", (64, 10), bits=4)); x2[3, 4] = 0.
    ids2 = torch.empty((64,), dtype=torch.int64, device="cuda")
    ops().vq_lfq_encode(dev(x2), None, None, ids2, 10)
    assert torch.equal(ids2.cpu(), ((x2 > 0).long() * (2 ** torch.arange(9, -1, -1))).sum(-1))


def test_vq_l2_argmin_and_decode_codes():
    T, K, D = 100, 777, 96
    x = torch.from_numpy(synth.dyadic("ax", (T, D), bits=3, span=2.0))
    cb = torch.from_numpy(synth.dyadic("acb", (K, D), bits=3, span=2.0))
    cb[400] = cb[20]                                                   # exact duplicate: first index must win
    ids = torch.empty((T,), dtype=torch.int64, device="cuda")
    ops().vq_l2_argmin(dev(x), dev(cb), ids)
    assert torch.equal(ids.cpu(), O.vq_l2_argmin(x, cb))
    bits, Dd = 9, 512
    w, bb = rnd("pw", (Dd, bits)), rnd("pb", (Dd,))
    code_ids = torch.from_numpy((synth.uniform("cid", (50,)) * 512).astype(np.int64))
    out = torch.empty((50, Dd), device="cuda")
    ops().vq_decode_codes(dev(code_ids), dev(w), dev(bb), out, bits)
    ref = O.lfq_codes_from_ids({"quantizer.project_out.weight": w, "quantizer.project_out.bias": bb}, code_ids, bits)
    ok, msg = close(out, ref, 1e-5)
    assert ok, msg


# ------------------------------------------------------------------------------------------------ convolutions
def nhwc(t):
    return t.permute(0, 2, 3, 1).contiguous()


def pack_conv(w):
    return w.permute(0, 2, 3, 1).reshape(w.shape[0], -1).contiguous()


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32], ids=["bf16", "fp32"])
@pytest.mark.parametrize("kind,B,H,W,Cin,Cout", [(1, 2, 16, 16, 64, 128), (1, 5, 2, 2, 128, 64), (2, 2, 32, 32, 64, 128), (2, 3, 4, 4, 64, 64),
                                                  (0, 2, 8, 8, 128, 128), (1, 1, 16, 16, 16, 32), (2, 1, 256, 256, 64, 64)])
def test_conv2d(dtype, kind, B, H, W, Cin, Cout):
    ksz, stride, pad = {0: (1, 1, 0), 1: (3, 1, 1), 2: (4, 2, 1)}[kind]
    x = rnd("cx", (B, Cin, H, W), dtype)
    w = rnd("cw", (Cout, Cin, ksz, ksz), dtype, std=(Cin * ksz * ksz) ** -0.5)
    bias = rnd("cb", (Cout,))
    Ho, Wo = H // stride, W // stride
    out = torch.empty((B * Ho * Wo, Cout), device="cuda", dtype=torch.float32 if dtype == torch.float32 else torch.bfloat16)
    ops().conv2d(dev(nhwc(x), dtype).view(-1, Cin), dev(pack_conv(w), dtype), out, B, H, W, Cin, Cout, kind, bias=dev(bias), act=1)
    ref = nhwc(F.leaky_relu(F.conv2d(x, w, bias, stride=stride, padding=pad), 0.1)).reshape(-1, Cout)
    ok, msg = close(out, ref, 2e-2 if dtype == torch.bfloat16 else 2e-4, 1e-2 if dtype == torch.bfloat16 else 1e-3)
    assert ok, msg


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32], ids=["bf16", "fp32"])
def test_conv2d_glu_and_residual(dtype):
    B, H, W, C = 2, 16, 16, 64
    x = rnd("gx", (B, C, H, W), dtype)
    w = rnd("gw", (2 * C, C, 3, 3), dtype, std=(9 * C) ** -0.5)
    bias = rnd("gb", (2 * C,))
    idx = torch.arange(C).view(-1, 32)
    order = torch.cat((idx, idx + C), 1).reshape(-1)
    od = torch.float32 if dtype == torch.float32 else torch.bfloat16
    out = torch.empty((B * H * W, C), device="cuda", dtype=od)
    ops().conv2d(dev(nhwc(x), dtype).view(-1, C), dev(pack_conv(w)[order], dtype), out, B, H, W, C, 2 * C, 1, epilogue=ops().EPI_GLU, bias=dev(bias[order]))
    ref = nhwc(F.glu(F.conv2d(x, w, bias, padding=1), dim=1)).reshape(-1, C)
    tol = (2e-2, 1e-2) if dtype == torch.bfloat16 else (2e-4, 1e-3)
    ok, msg = close(out, ref, *tol)
    assert ok, msg
    w1 = rnd("rw", (C, C, 1, 1), dtype, std=C ** -0.5); b1 = rnd("rb", (C,))
    skip = rnd("rs", (B, C, H, W), dtype)
    out2 = torch.empty((B * H * W, C), device="cuda", dtype=od)
    ops().conv2d(dev(nhwc(x), dtype).view(-1, C), dev(pack_conv(w1), dtype), out2, B, H, W, C, C, 0, epilogue=ops().EPI_RESIDUAL, bias=dev(b1),
                 resid=dev(nhwc(skip), dtype).view(-1, C))
    ok, msg = close(out2, nhwc(F.conv2d(x, w1, b1) + skip).reshape(-1, C), *tol)
    assert ok, msg


def pack_convt(w):
    from muse_maskgit_pytorch_b200.vqgan_vae import CT_R
    packs = []
    for py in range(2):
        for px in range(2):
            packs.append(torch.cat([w[:, :, CT_R[py][a], CT_R[px][b]].t() for a in range(2) for b in range(2)], dim=1))
    return torch.stack(packs).contiguous()


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32], ids=["bf16", "fp32"])
@pytest.mark.parametrize("B,H,W,Cin,Cout", [(2, 16, 16, 128, 64), (3, 2, 2, 64, 64), (1, 128, 128, 64, 64), (1, 8, 8, 32, 16)])
def test_conv_transpose2d(dtype, B, H, W, Cin, Cout):
    x = rnd("tx", (B, Cin, H, W), dtype)
    w = rnd("tw", (Cin, Cout, 4, 4), dtype, std=(4 * Cin) ** -0.5)
    bias = rnd("tb", (Cout,))
    od = torch.float32 if dtype == torch.float32 else torch.bfloat16
    out = torch.empty((B * 4 * H * W, Cout), device="cuda", dtype=od)
    ops().conv_transpose2d(dev(nhwc(x), dtype).view(-1, Cin), dev(pack_convt(w), dtype), out, B, H, W, Cin, Cout, bias=dev(bias))
    ref = nhwc(F.leaky_relu(F.conv_transpose2d(x, w, bias, stride=2, padding=1), 0.1)).reshape(-1, Cout)
    tol = (2e-2, 1e-2) if dtype == torch.bfloat16 else (2e-4, 1e-3)
    ok, msg = close(out, ref, *tol)
    assert ok, msg


def test_conv_transpose2d_fused_rgb():
    B, H, W, Cin, Cout = 2, 32, 32, 64, 64
    x = rnd("fx", (B, Cin, H, W), torch.bfloat16)
    w = rnd("fw", (Cin, Cout, 4, 4), torch.bfloat16, std=(4 * Cin) ** -0.5)
    bias, rw, rb = rnd("fb", (Cout,)), rnd("frw", (3, Cout), std=Cout ** -0.5), rnd("frb", (3,))
    out = torch.empty((B, 3, 2 * H, 2 * W), device="cuda")
    ops().conv_transpose2d(dev(nhwc(x), torch.bfloat16).view(-1, Cin), dev(pack_convt(w), torch.bfloat16), out, B, H, W, Cin, Cout,
                           bias=dev(bias), rgb_w=dev(rw), rgb_b=dev(rb))
    ref = F.conv2d(F.leaky_relu(F.conv_transpose2d(x, w, bias, stride=2, padding=1), 0.1), rw[:, :, None, None], rb)
    ok, msg = close(out, ref, 5e-4)
    assert ok, msg


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32], ids=["bf16", "fp32"])
def test_groupnorm_and_conv_in(dtype):
    B, HW, C = 2, 64, 128
    x = rnd("nx", (B, HW, C), dtype) * 2 + 0.3
    g, be = 1 + 0.1 * rnd("ng", (C,)), 0.1 * rnd("nb", (C,))
    xd = dev(x, dtype).contiguous()
    ops().groupnorm_(xd, dev(g), dev(be), B, HW, C, 16, act=1)
    ref = F.leaky_relu(F.group_norm(x.permute(0, 2, 1), 16, g, be), 0.1).permute(0, 2, 1)
    ok, msg = close(xd, ref, 3e-2 if dtype == torch.bfloat16 else 2e-5, 1e-2)
    assert ok, msg
    img = torch.from_numpy(synth.uniform("im", (2, 3, 12, 20)))
    w, b = rnd("iw", (64, 3, 5, 5), std=75 ** -0.5), rnd("ib", (64,))
    out = torch.empty((2 * 12 * 20, 64), device="cuda", dtype=dtype)
    ops().conv_in(dev(img), dev(w), dev(b), out)
    ok, msg = close(out, nhwc(F.conv2d(img, w, b, padding=2)).reshape(-1, 64), 2e-2 if dtype == torch.bfloat16 else 1e-5, 1e-2)
    assert ok, msg


def test_linear_geglu_lnfold_pair():
    """inner LayerNorm folded through FF2: GEGLU epilogue accumulates per-row (sum, sumsq); LNFOLD_RESIDUAL applies
    rstd * (acc - mean * cvec) + resid  ==  resid + LN(h) W2^T   (ref: muse_maskgit_pytorch.py:83-89)."""
    M, K, Fu, Fp, dim = 300, 128, 341, 384, 128
    bf = torch.bfloat16
    a = rnd("a", (M, K), bf)
    wx, wg = rnd("wx", (Fu, K), bf, std=K ** -0.5), rnd("wg", (Fu, K), bf, std=K ** -0.5)
    wxp, wgp = torch.zeros((Fp, K)), torch.zeros((Fp, K)); wxp[:Fu], wgp[:Fu] = wx, wg
    w1 = torch.stack((wxp.view(-1, 32, K), wgp.view(-1, 32, K)), 1).reshape(2 * Fp, K)
    g3 = 1 + 0.1 * rnd("g3", (Fu,))
    w2 = rnd("w2", (dim, Fu), std=Fu ** -0.5)
    w2f = torch.zeros((dim, Fp)); w2f[:, :Fu] = w2 * g3
    w2f = w2f.to(bf)
    cvec = w2f.float().sum(1)
    x = rnd("x", (M, dim))
    h = torch.empty((M, Fp), device="cuda", dtype=bf)
    stats = torch.full((M, Fp // 32, 2), float("nan"), device="cuda")      # per-chunk partials: every slot is written, none accumulated
    xd = dev(x)
    ops().linear(dev(a, bf), dev(w1, bf), h, epilogue=ops().EPI_GEGLU, row_stats=stats)
    ops().linear(h, dev(w2f), xd, epilogue=ops().EPI_LNFOLD_RESIDUAL, bias=dev(cvec), resid=xd, row_stats=stats, ln_width=Fu)
    href = (a @ wg.t()) * F.gelu(a @ wx.t())
    # the statistics are those of the bf16-rounded outputs, chunk by chunk
    hq = h.float().cpu().view(M, Fp // 32, 32)
    assert torch.allclose(stats[..., 0].cpu(), hq.sum(-1), atol=1e-4, rtol=1e-5) and torch.allclose(stats[..., 1].cpu(), (hq * hq).sum(-1), atol=1e-4, rtol=1e-5)
    ok, msg = close(stats[..., 0].sum(-1), href.sum(-1), 5e-3 * float(href.sum(-1).abs().max()), 1e-2)     # bf16 rounding of 341 summands
    assert ok, "row sums: " + msg
    ref = x + F.layer_norm(href, (Fu,), g3, None) @ w2.t()
    ok, msg = close(xd, ref, 3e-2, 1e-2)
    assert ok, msg


def test_lfq_ids_gemm_epilogue_bit_exact():
    """tcgen05 path of the LFQ lookup: 3-way bf16 split of project_in + LFQ_IDS epilogue; dyadic data -> bit-identical ids."""
    T, D, bits = 1000, 2048, 16
    bf = torch.bfloat16
    x = torch.from_numpy(synth.dyadic("vx", (T, D), bits=4, span=2.0))
    w = torch.from_numpy(synth.dyadic("vw", (bits, D), bits=4, span=1.0)) + torch.from_numpy(synth.dyadic("vw2", (bits, D), bits=4, span=1.0)) * 2.0 ** -12
    bias = torch.from_numpy(synth.dyadic("vb", (bits,), bits=4, span=1.0))
    hi = w.to(bf); r1 = w - hi.float(); mid = r1.to(bf); lo = (r1 - mid.float()).to(bf)
    assert torch.equal(hi.float() + mid.float() + lo.float(), w)
    w3 = torch.zeros((64, D), dtype=bf); w3[:bits], w3[bits:2 * bits], w3[2 * bits:3 * bits] = hi, mid, lo
    ids = torch.empty((T,), dtype=torch.int64, device="cuda")
    ops().linear(dev(x, bf), dev(w3), ids, epilogue=ops().EPI_LFQ_IDS, bias=dev(bias), ln_width=bits)
    proj = x.double() @ w.double().t() + bias.double()
    ref = ((proj > 0).long() * (2 ** torch.arange(bits - 1, -1, -1))).sum(-1)
    assert torch.equal(ids.cpu(), ref)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32], ids=["bf16", "fp32"])
def test_argmin_gemm_epilogue(dtype):
    T, K, D = 200, 1024, 128
    x = torch.from_numpy(synth.dyadic("ax", (T, D), bits=3, span=2.0))
    cb = torch.from_numpy(synth.dyadic("acb", (K, D), bits=3, span=2.0))
    cb[700] = cb[33]
    best = torch.full((T,), -1, dtype=torch.int64, device="cuda")
    norms = (cb * cb).sum(-1)
    ops().linear(dev(x, dtype), dev(cb, dtype), best, epilogue=ops().EPI_ARGMIN, bias=dev(norms))
    assert torch.equal((best & 0xFFFFFFFF).cpu(), O.vq_l2_argmin(x, cb))


def test_logits_sample_philox_matches_oracle_stream():
    """In-kernel Philox4x32-10 draws exactly the uniforms oracle/philox.py produces for (seed, step, global row, v): the
    sampled ids equal the oracle's on that stream wherever the perturbed top-2 margin exceeds the fast-log error."""
    from oracle import philox
    b, n, nm, V, seed, step, off = 2, 16, 6, 8192, 987654321012, 5, 3 * 16
    k = O.top_k_count(V, 0.9)
    logits = torch.from_numpy(synth.normal("lgq", (b, nm, V), 13, 0.58))
    g = torch.Generator().manual_seed(4)
    mp = torch.stack([torch.sort(torch.randperm(n, generator=g)[:nm]).values for _ in range(b)]).int()
    ids = torch.full((b, n), V, dtype=torch.long, device="cuda"); sc = torch.full((b, n), -1e5, device="cuda")
    ops().logits_sample(dev(logits.reshape(-1, V).contiguous()), dev(mp), ids, sc, nm, k, 0.7, seed=seed, step=step, row_offset=off)
    rows_u = torch.stack([torch.from_numpy(philox.uniform(seed, step, off + bi * n + int(mp[bi, j]), V)) for bi in range(b) for j in range(nm)])
    pred, score, margin = _oracle_rows(logits.reshape(-1, V), rows_u, 0.7, k)
    got = torch.stack([ids.cpu()[bi, mp[bi, j]] for bi in range(b) for j in range(nm)])
    assert torch.equal(got[margin > 1e-3], pred[margin > 1e-3]), (got.tolist(), pred.tolist())
    assert (got == pred).float().mean() > 0.9


def test_ff_geglu_lnfold_bitwise_reproducible_at_block_width():
    """dim 512 / inner 1365 (44 statistic chunks per row, 11 column tiles, CTA pairs): the folded-LayerNorm FeedForward gives the same bits on
    every run — the row statistics are per-chunk partials added in a fixed order, not atomics."""
    M, K, Fu, Fp, dim = 4096, 512, 1365, 1408, 512
    bf = torch.bfloat16
    g = torch.Generator(device="cuda").manual_seed(3)
    a = torch.randn((M, K), device="cuda", generator=g).to(bf)
    w1 = (torch.randn((2 * Fp, K), device="cuda", generator=g) * K ** -0.5).to(bf)
    w2f = (torch.randn((dim, Fp), device="cuda", generator=g) * Fu ** -0.5).to(bf); w2f[:, Fu:] = 0
    cvec = w2f.float().sum(1).contiguous()
    x0 = torch.randn((M, dim), device="cuda", generator=g)
    outs = []
    for _ in range(4):
        h = torch.empty((M, Fp), device="cuda", dtype=bf); stats = torch.empty((M, Fp // 32, 2), device="cuda"); xd = x0.clone()
        ops().linear(a, w1, h, epilogue=ops().EPI_GEGLU, row_stats=stats)
        ops().linear(h, w2f, xd, epilogue=ops().EPI_LNFOLD_RESIDUAL, bias=cvec, resid=xd, row_stats=stats, ln_width=Fu)
        outs.append((h.clone(), stats.clone(), xd))
    for h, st, xd in outs[1:]:
        assert torch.equal(h, outs[0][0]) and torch.equal(st, outs[0][1])
        # the in-place residual is a TMA reduction (fp32 adds in L2, one per element): also order-independent
        assert torch.equal(xd, outs[0][2])


@pytest.mark.parametrize("N", [512, 128])
def test_linear_residual_with_fused_layernorm(N):
    """cluster-of-2 GEMM: x += a W^T (rows >= split also += add), ln_out = LN(x) * gamma (gamma_b for rows >= split),
    The two CTAs exchange (sum, sumsq) through distributed shared memory."""
    M, K, split = 700, 256, 384
    bf = torch.bfloat16
    a, w = rnd("a", (M, K), bf), rnd("w", (N, K), bf, std=K ** -0.5)
    x = rnd("x", (M, N)) * 2 + 0.3
    ga, gb, add = 1 + 0.1 * rnd("ga", (N,)), 1 + 0.1 * rnd("gb", (N,)), rnd("add", (N,))
    xd = dev(x); xn = torch.zeros((M, N), device="cuda", dtype=bf)
    gad, gbd, addd = dev(ga), dev(gb), dev(add)
    ops().linear(dev(a, bf), dev(w, bf), xd, epilogue=ops().EPI_RESIDUAL, resid=xd, ln_out=xn, ln_gamma=gad, ln_gamma_b=gbd, ln_add=addd, ln_split=split)
    ref = x + a @ w.t()
    ref[split:] += add
    ok, msg = close(xd, ref, 3e-4)
    assert ok, "x: " + msg
    lref = torch.cat((F.layer_norm(ref[:split], (N,), ga, None), F.layer_norm(ref[split:], (N,), gb, None)))
    ok, msg = close(xn, lref, 2e-2, 1e-2)
    assert ok, "ln_out: " + msg


@pytest.mark.parametrize("cfg_branch", [False, True])
def test_critic_score(cfg_branch):
    """mmg_critic_score vs torch: final LayerNorm + 1-wide head + CFG + annealed noise (ref: muse_maskgit_pytorch.py:590-600)."""
    from oracle import philox
    torch.manual_seed(3)
    rows, dim = 37, 128
    xc, xn = torch.randn(rows, dim) * 2 + 0.3, torch.randn(rows, dim)
    g, w = torch.rand(dim) + 0.5, torch.randn(dim) * 0.1
    u = torch.rand(rows)
    head = lambda x: torch.nn.functional.layer_norm(x, (dim,), g, None, 1e-5) @ w + 0.25
    want = head(xc)
    if cfg_branch:
        want = head(xn) + (want - head(xn)) * 3.0
    sc = torch.zeros(rows, device="cuda")
    ops().critic_score(xc.cuda(), xn.cuda() if cfg_branch else None, g.cuda(), w.cuda(), 0.25, 3.0, 0.6, sc, u=u.cuda())
    assert (sc.cpu() - (want + (u - 0.5) * 0.6)).abs().max() < 1e-5
    # Philox stream: counter (0xFFFFFFFF, step, global row), key = seed  -> same numbers as oracle/philox.py
    seed_dev = torch.tensor([11], dtype=torch.int64, device="cuda")
    ops().critic_score(xc.cuda(), xn.cuda() if cfg_branch else None, g.cuda(), w.cuda(), 0.25, 3.0, 0.6, sc, seed=1, seed_dev=seed_dev, step=4, row_offset=100)
    up = torch.tensor([float(philox.uniform_at(12, 4, 100 + r, 0xFFFFFFFF)) for r in range(rows)])
    assert (sc.cpu() - (want + (up - 0.5) * 0.6)).abs().max() < 1e-5


def test_linear_wide_tiles_tma_epilogues():
    """Shapes large enough for the 256-column tiles, whose fp32 epilogues leave through per-warp shared-memory tiles and TMA:
    a plain store (the logits GEMM's path) with a ragged last row block, and the in-place residual as a TMA reduction
    (x += a W^T with the adds performed in L2; the second call checks that nothing but the product is added)."""
    bf = torch.bfloat16
    M, N, K = 300, 25600, 64                      # 3 x 100 tiles, rows 256..299 of the last block only
    a, w = rnd("wa", (M, K), bf), rnd("ww", (N, K), bf, std=K ** -0.5)
    out = torch.full((M + 7, N), 7.0, device="cuda")
    ops().linear(dev(a, bf), dev(w, bf), out[:M])
    ok, msg = close(out[:M], a @ w.t(), 2e-4)
    assert ok, msg
    assert bool((out[M:] == 7.0).all()), "rows past M were written"
    M, N, K = 2000, 4096, 512                     # 128-column tiles (16 x 32): the fused tail's sample GEMM at 8 images per GPU
    a, w = rnd("sa", (M, K), bf), rnd("sw", (N, K), bf, std=K ** -0.5)
    out = torch.full((M + 3, N), 7.0, device="cuda")
    ops().linear(dev(a, bf), dev(w, bf), out[:M])
    ok, msg = close(out[:M], a @ w.t(), 2e-4)
    assert ok, msg
    assert bool((out[M:] == 7.0).all()), "rows past M were written"
    M, N, K = 2000, 5120, 64                      # 16 x 20 tiles
    a, w, x = rnd("ra", (M, K), bf), rnd("rw", (N, K), bf, std=K ** -0.5), rnd("rx", (M, N))
    xd = dev(x)
    ops().linear(dev(a, bf), dev(w, bf), xd, epilogue=ops().EPI_RESIDUAL, resid=xd)
    ok, msg = close(xd, x + a @ w.t(), 3e-4)
    assert ok, msg
    ops().linear(dev(a, bf), dev(w, bf), xd, epilogue=ops().EPI_RESIDUAL, resid=xd)
    ok, msg = close(xd, x + 2 * (a @ w.t()), 5e-4)
    assert ok, msg


@pytest.mark.parametrize("b,q_only", [(16, False), (32, False), (32, True)], ids=["bn128", "bn256", "q_only"])
def test_linear_qkv_epilogue_tma_tiles(b, q_only):
    """The QKV epilogue at shapes where it leaves through per-warp tiles + TMA stores (tokens % 32 == 0, M % 128 == 0, 128- or
    256-column tiles): same contract as test_linear_qkv_epilogue, incl. the null key/value row and untouched padding rows."""
    bf = torch.bfloat16
    n, heads, dim = 256, 8, 128
    inner = heads * 64
    nsec = 1 if q_only else 3
    x = rnd("xq", (b * n, dim), bf)
    w = rnd("wq3", (nsec * inner, dim), bf, std=dim ** -0.5)
    qs, ks = 1 + 0.1 * rnd("qs", (64,)), 1 + 0.1 * rnd("ks", (64,))
    nk, nv = rnd("nk8", (heads, 64), bf), rnd("nv8", (heads, 64), bf)
    q = torch.zeros((b * heads + 3, n, 64), device="cuda", dtype=bf)          # 3 guard blocks past the tensor the epilogue is told about
    k = torch.zeros((b * heads, n + 8, 64), device="cuda", dtype=bf)
    v = torch.zeros_like(k)
    qsd, ksd, nkd, nvd = dev(qs), dev(ks), dev(nk, bf), dev(nv, bf)
    if q_only:
        e = ops().qkv_epilogue(bf, heads, n, q=q[:b * heads], q_scale=qsd)
    else:
        e = ops().qkv_epilogue(bf, heads, n, q=q[:b * heads], k=k, v=v, q_scale=qsd, k_scale=ksd, key_off=1, null_k=nkd, null_v=nvd)
    ops().linear(dev(x, bf), dev(w, bf), None, epilogue=ops().EPI_QKV, epi=e)
    y = (x @ w.t()).view(b, n, nsec, heads, 64).permute(2, 0, 3, 1, 4)
    ok, msg = close(q[:b * heads].view(b, heads, n, 64), F.normalize(y[0], dim=-1) * qs, 2e-2, 1e-2)
    assert ok, "q: " + msg
    assert float(q[b * heads:].abs().max()) == 0.
    if not q_only:
        kk, vv = k.view(b, heads, n + 8, 64), v.view(b, heads, n + 8, 64)
        ok, msg = close(kk[:, :, 1:n + 1], F.normalize(y[1], dim=-1) * ks, 2e-2, 1e-2)
        assert ok, "k: " + msg
        ok, msg = close(vv[:, :, 1:n + 1], y[2], 2e-2, 1e-2)
        assert ok, "v: " + msg
        assert torch.equal(kk[:, :, 0].float().cpu(), nk.expand(b, -1, -1)) and torch.equal(vv[:, :, 0].float().cpu(), nv.expand(b, -1, -1))
        assert float(kk[:, :, n + 1:].abs().max()) == 0. and float(vv[:, :, n + 1:].abs().max()) == 0.


@pytest.mark.parametrize("thres,temp", [(0.8, 1.0), (0.5, 0.3), (0.0, 1.0)])
def test_logits_sample_any_topk_threshold(thres, temp):
    """topk_filter_thres below ~0.86 at V = 65536 keeps more logits than the candidate list holds (k > 9216): the row-walking kernel must
    give the reference's result (muse_maskgit_pytorch.py:413-418 accepts any threshold), including rows with many ties at the k-th value."""
    b, n, nm, V = 1, 8, 5, 65536
    k = O.top_k_count(V, thres)
    assert k > 9216
    base = torch.from_numpy(synth.normal("bigk", (nm, V), 21, 0.58))
    base[3] = torch.round(base[3] * 4) / 4                  # few distinct values: thousands of ties at the k-th largest
    base[4] = 0.                                            # constant row: every logit ties
    logits = base[None]
    u = torch.from_numpy(synth.uniform("ubigk", (b, n, V), 21))
    g = torch.Generator().manual_seed(3)
    mp = torch.sort(torch.randperm(n, generator=g)[:nm]).values.int()[None]
    ids = torch.full((b, n), V, dtype=torch.long, device="cuda"); sc = torch.full((b, n), -1e5, device="cuda")
    ops().logits_sample(dev(logits.reshape(nm, V).contiguous()), dev(mp), ids, sc, nm, k, temp, u=dev(u))
    rows_u = torch.stack([u[0, mp[0, j]] for j in range(nm)])
    pred, score, margin = _oracle_rows(logits.reshape(-1, V), rows_u, temp, k)
    got = torch.stack([ids.cpu()[0, mp[0, j]] for j in range(nm)])
    gsc = torch.stack([sc.cpu()[0, mp[0, j]] for j in range(nm)])
    ok = margin > 1e-4
    assert torch.equal(got[ok], pred[ok]), (got.tolist(), pred.tolist(), margin.tolist())
    assert torch.allclose(gsc[got == pred], score[got == pred], atol=2e-6)


# ------------------------------------------------------------------------------------------------ fp32 on the tensor cores (3-way bf16 split)
def test_split3_terms_reconstruct_fp32():
    """mmg_split3: hi + mid + lo == x to 2^-24 relative, every term a bf16 value, operand orders as documented in include/mmg.h."""
    x = rnd("s3", (70, 192)) * torch.from_numpy(synth.normal("s3e", (70, 192), 5, 3.0)).exp()       # wide dynamic range
    for side, order in ((0, "LHMMHH"), (1, "HLMHMH")):
        s = ops().split3(dev(x), side).float().cpu().view(70, 6, 192)
        hi = x.to(torch.bfloat16).float(); r1 = x - hi; mid = r1.to(torch.bfloat16).float(); lo = (r1 - mid).to(torch.bfloat16).float()
        terms = {"H": hi, "M": mid, "L": lo}
        for t, ch in enumerate(order):
            assert torch.equal(s[:, t], terms[ch]), (side, t)
        assert ((hi + mid + lo - x).abs() <= x.abs() * 2.0 ** -23).all()


@pytest.mark.parametrize("M,N,K", [(256, 512, 512), (300, 192, 128), (1024, 2816, 512), (512, 512, 1408)])
def test_linear_fp32_tensor_core_split_vs_fp64(M, N, K):
    """precision='fp32' products run as 6K-wide bf16 products on tcgen05: error vs an fp64 reference at the level of the fp32 CUDA-core kernel."""
    a, w = rnd(f"a{M}{K}", (M, K)), rnd(f"w{N}{K}", (N, K), std=K ** -0.5)
    ref = (a.double() @ w.double().t())
    o = ops()
    was = o.fp32_tc()
    try:
        errs = {}
        for mode in (True, False):
            o.fp32_tc(mode)
            out = torch.empty((M, N), device="cuda", dtype=torch.float32)
            o.linear(dev(a), dev(w), out)
            errs[mode] = float((out.cpu().double() - ref).abs().max())
    finally:
        o.fp32_tc(was)
    print(f"max |err| vs fp64: tensor-core split {errs[True]:.3e}, CUDA-core fp32 {errs[False]:.3e}")
    assert errs[True] <= max(4 * errs[False], 2e-6), errs


def test_conv2d_fp32_tensor_core_split_vs_fp64():
    B, H, W, Cin, Cout = 2, 16, 16, 64, 128
    x, wt, bias = rnd("cx", (B, Cin, H, W)), rnd("cw", (Cout, Cin, 3, 3), std=(9 * Cin) ** -0.5), rnd("cb", (Cout,))
    ref = F.conv2d(x.double(), wt.double(), bias.double(), padding=1).permute(0, 2, 3, 1).reshape(-1, Cout)
    o = ops()
    xh = dev(x.permute(0, 2, 3, 1).contiguous())
    wp = dev(wt.permute(0, 2, 3, 1).reshape(Cout, -1).contiguous())
    was = o.fp32_tc()
    try:
        errs = {}
        for mode in (True, False):
            o.fp32_tc(mode)
            out = torch.empty((B * H * W, Cout), device="cuda", dtype=torch.float32)
            o.conv2d(xh, wp, out, B, H, W, Cin, Cout, 1, bias=dev(bias))
            errs[mode] = float((out.cpu().double() - ref).abs().max())
    finally:
        o.fp32_tc(was)
    print(f"max |err| vs fp64: tensor-core split {errs[True]:.3e}, CUDA-core fp32 {errs[False]:.3e}")
    # the tensor core adds into its fp32 accumulator with truncation (up to ~1 ulp per K = 16 step, 216 steps here) where the CUDA-core kernel
    # rounds to nearest: the bound is in ulps of the output range, not relative to the CUDA-core error
    assert errs[True] <= 3e-5 * float(ref.abs().max()), errs
