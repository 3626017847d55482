"""bench.py — images/sec of MaskGit.generate() 256x256, 18 steps, CFG=3 (BASELINE.json metric, config C3), batch 64
sharded over N GPUs of one node (STRONG scaling: the global batch is fixed at 64, per-GPU batch = 64/N).

  python bench.py --gpus N --steps K --warmup W            # our arm (libmmg.so through the drop-in classes + parallel.generate_sharded)
  python bench.py --impl reference --gpus N --steps K ...  # the UNMODIFIED reference's MaskGit.generate() on the host cores (baseline/_ref)
  python bench.py --config C2|C4|C5                        # secondary configs of BASELINE.json (one JSON line each; C3 is the default)
  python bench.py ... --dump-outputs DIR                   # C3: also write the last timed step's images to DIR/images.npy

One "step" = one full generate() call over the rank's shard (18 decode steps + VAE decode + (N>1) one NCCL all-gather of
the decoded images).  `value` is timed with the text embeddings already resident in HBM; `e2e` times the same public call
with the embeddings coming from pinned host memory and the images copied back to the host inside the timed region.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

GLOBAL_BATCH = 64
IMAGE, TIMESTEPS, COND_SCALE, TEXT_LEN = 256, 18, 3.0, 32
TR_CFG = dict(num_tokens=65536, seq_len=256, dim=512, depth=8, dim_head=64, heads=8, ff_mult=4)
TR_SR_CFG = dict(num_tokens=65536, seq_len=1024, dim=512, depth=2, dim_head=64, heads=8, ff_mult=4)
VAE_CFG = dict(dim=256, codebook_size=65536)
# algorithmic dense work (SURVEY.md 8d / BASELINE.md 3), GFLOP per image
GFLOP_PER_IMAGE = 1378.7            # C3: 36 forwards x 33.70 + decode 165.47
ATTN_GFLOP_PER_IMAGE = 1.216 * 36
GFLOP_C2_FORWARD = 33.70
GFLOP_C4_IMAGE = 4026.0
GFLOP_C5_IMAGE = 1178.9
METRIC = "images/sec MaskGit.generate() 256x256 18-step CFG=3"
REF_BATCH = 4                       # BASELINE.md section 4: the CPU arm runs B_cpu = 4 (CPU throughput is flat in B)
DUMP_BYTES = 64 << 20               # --dump-outputs writes at most this much (the 64 images of C3 are 50 MB in fp32)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(tflops=d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1400.0)), hbm=d.get("hbm_gbs", 6650.0), src="measured")
    return dict(tflops=1400.0, hbm=6650.0, src="fallback")


def text_embeddings(batch, seed=1):
    g = torch.Generator().manual_seed(seed)
    te = torch.randn((batch, TEXT_LEN, 512), generator=g)
    te[1::2, 24:] = 0.                      # padded positions on odd rows (exercises the context mask)
    return te


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    def __init__(self, index):
        super().__init__(daemon=True)
        self.rows, self.proc, self.index = [], None, index

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc:
            self.proc.terminate()
        out = dict(sm_mhz=None, sm_max_mhz=None, reasons=[])
        try:
            sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
            if sm:
                out["sm_mhz"] = sm[len(sm) // 2]
                out["sm_max_mhz"] = float(self.rows[0][1])
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            out["reasons"] = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        except Exception:
            pass
        return out


def build_models(device, precision="bf16", superres=False):
    import muse_maskgit_pytorch_b200 as M
    from muse_maskgit_pytorch_b200 import t5
    t5.T5_CONFIGS["synth-512"] = {"d_model": 512}
    torch.manual_seed(0)
    vae = M.VQGanVAE(precision=precision, **VAE_CFG)
    if superres:
        tr = M.MaskGitTransformer(t5_name="synth-512", precision=precision, **TR_SR_CFG)
        return M.MaskGit(image_size=512, cond_image_size=256, transformer=tr.to(device), vae=vae.to(device)).to(device)
    tr = M.MaskGitTransformer(t5_name="synth-512", precision=precision, **TR_CFG)
    return M.MaskGit(image_size=IMAGE, transformer=tr.to(device), vae=vae.to(device)).to(device)


def dist_setup():
    import torch.distributed as dist
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    return dist, rank, world, local, device


def timed_loop(dist, world, device, fn, steps, flush=None):
    """EXACTLY `steps` calls of fn bracketed by barrier + synchronize, CUDA events on the launching stream, MAX over ranks."""
    from muse_maskgit_pytorch_b200 import _lib
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    l0 = _lib.launch_count()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(steps):
        if flush is not None:
            flush()
        fn()
    t1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([t0.elapsed_time(t1)], device=device)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        dist.barrier()
    return float(ms) / steps, (_lib.launch_count() - l0) // steps


# ================================================================================================ C3 (the headline)
def run_ours(args):
    dist, rank, world, local, device = dist_setup()
    assert GLOBAL_BATCH % world == 0
    b = GLOBAL_BATCH // world
    from muse_maskgit_pytorch_b200 import parallel
    mg = build_models(device)
    mg.sampler_seed = 2
    te_all_host = text_embeddings(GLOBAL_BATCH).pin_memory()
    lo, hi = parallel.shard_bounds(GLOBAL_BATCH, rank, world)
    te_host = te_all_host[lo:hi].contiguous().pin_memory()              # this rank's rows (what a data loader would hand it)
    te_dev = te_host.to(device)
    texts = [""] * GLOBAL_BATCH
    host_out = torch.empty((GLOBAL_BATCH, 3, IMAGE, IMAGE)).pin_memory() if rank == 0 else None
    gen_kw = dict(timesteps=TIMESTEPS, cond_scale=COND_SCALE, temperature=1., topk_filter_thres=0.9)

    def step(e2e):
        # the product's own multi-GPU entry point: shard by global row, generate, ONE all-gather of the decoded images
        shard = te_host.to(device, non_blocking=True) if e2e else te_dev
        images = parallel.generate_sharded(mg, texts, text_embeds_shard=shard, seed=2, **gen_kw)
        if e2e and rank == 0:
            host_out.copy_(images, non_blocking=True)                    # the step's result is read back on rank 0
        return images

    for _ in range(max(args.warmup, 3)):
        step(False)
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    last = {}

    def timed_step():
        last["images"] = step(False)
    ms, launches = timed_loop(dist, world, device, timed_step, args.steps)
    clocks = sampler.stop() if sampler else None
    step(True)
    ms_e2e, _ = timed_loop(dist, world, device, lambda: step(True), args.steps)

    line = None
    if rank == 0:
        pk = peaks()
        mg.row_offset = lo
        roof = kernel_roofline(mg, [""] * b, te_dev, pk)
        value = GLOBAL_BATCH / (ms / 1e3)
        line = {
            "metric": METRIC, "value": round(value, 2), "unit": "images/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": round(ms, 3),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "C3: MaskGit.generate() 256x256, 18 steps, cond_scale=3, top-k 0.9, global batch 64 "
                                   "(batch-sharded, one NCCL all-gather of images per call); transformer dim512 depth8 V65536, VQGanVAE dim256; "
                                   "random-init weights, pre-computed T5 embeddings (32 positions)",
                       "global_batch": GLOBAL_BATCH, "per_gpu_batch": b, "parallelism": f"dp{world}",
                       "l2": "inputs larger than L2: every decode step streams the 67 MB logits weight and > 1 GB of activations / candidates"},
            "e2e": {"value": round(GLOBAL_BATCH / (ms_e2e / 1e3), 2), "unit": "images/s",
                    "h2d_bytes_per_step": te_host.numel() * 4 * world, "d2h_bytes_per_step": host_out.numel() * 4},
            "gpu_launches": (launches if launches > 0 else roof["launches_per_step_all_kernels"]) * args.steps,   # graph replays re-issue the captured kernel nodes
            "launches_per_decode_step": round(roof["launches_per_step_all_kernels"] / TIMESTEPS, 1),
            "simt_fallbacks": __import__("muse_maskgit_pytorch_b200")._lib.simt_fallback_count(),      # bf16 products that left the tcgen05 path (must be 0 here)
            "clocks": clocks,
            "roofline": roof,
            "dense_flop_frac_of_peak": round(value * GFLOP_PER_IMAGE / 1e3 / world / pk["tflops"], 4),
            "attention_gemm_roofline_frac": round(value * ATTN_GFLOP_PER_IMAGE / 1e3 / world / pk["tflops"], 5),
            "peaks": pk,
            "parity_note": "bf16 operands / fp32 accumulation: token ids are a flip-rate bound vs the fp32 reference (see `parity`), identical in "
                           "precision='fp32'; top-k keeps the LOWEST vocabulary index among logits equal to the k-th, re-mask the lowest position",
        }
        if world == 1 and not args.no_extras:
            line["hbm_kernels"] = hbm_kernels(mg, pk)
            line["parity"] = teacher_forced_flip_rate(mg)
            line["gpu_eager_baseline"] = gpu_eager_baseline(device)
            line["cpu_baseline"] = cpu_baseline()
        if args.dump_outputs:
            dump_images(args.dump_outputs, last["images"])
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        print(json.dumps(line))


def dump_images(directory, images):
    """--dump-outputs: the images the timed generate() returned in its last timed step, as float32 DIR/images.npy, so that two builds run with
    the same arguments (hence the same seeded weights, text embeddings and sampler seed) can be compared output for output.  A batch larger
    than DUMP_BYTES (--global-batch) is cut to a fixed, seeded sample of whole images."""
    import numpy as np
    a = images.detach().float().cpu().numpy()
    if a.nbytes > DUMP_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(a.shape[0], DUMP_BYTES // a[0].nbytes, replace=False))
        a = a[keep]
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "images.npy"), a)


def _gemm_flops(name, a):
    if name == "mmg_linear":
        return 2.0 * a.M * a.N * a.K
    if name == "mmg_conv2d":
        taps = {0: 1, 1: 9, 2: 16, 3: 25}[a.kind]
        s = 2 if a.kind == 2 else 1
        return 2.0 * a.B * (a.H // s) * (a.W // s) * a.Cout * taps * a.Cin
    if name == "mmg_conv_transpose2d":
        return 2.0 * a.B * a.H * a.W * a.Cout * 16 * a.Cin
    if name == "mmg_logits_fused":
        return 2.0 * a.s.B * a.s.num_masked * a.s.V * a.K
    return 0.0


def kernel_roofline(mg, texts, te_dev, pk):
    """Per-entry-point device time of ONE generate(): every libmmg call is bracketed by CUDA events.  Preferred: the events are
    captured INTO a CUDA graph of the call (external event-record nodes) and read after a replay, so the durations are the in-situ ones
    of the replayed graph; fallback: an eager pass (launch gaps then contaminate small kernels).  The dominant kernel is the tcgen05 GEMM
    (mmg_linear / mmg_conv* / the fused logits-sampling GEMM): algorithmic FLOPs / its summed duration vs the measured bf16 peak."""
    from muse_maskgit_pytorch_b200 import _lib
    rec = []
    orig = _lib.call
    state = {"external": False}

    def prof_call(name, a, stream=None):
        kw = dict(enable_timing=True)
        if state["external"]:
            kw["external"] = True
        e0, e1 = torch.cuda.Event(**kw), torch.cuda.Event(**kw)
        e0.record()
        orig(name, a, stream)
        e1.record()
        rec.append((name, e0, e1, _gemm_flops(name, a)))

    graph_mode, check_mode = mg.use_cuda_graph, mg.check_fused_tail
    mg.check_fused_tail = False                                # its 4-byte host read is not capturable
    mg.transformer.encode_text = lambda t: te_dev
    kw = dict(timesteps=TIMESTEPS, cond_scale=COND_SCALE)
    how = "eager"
    try:
        mg.use_cuda_graph = False
        if os.environ.get("MMG_ROOFLINE_EAGER", "0") != "1":
            try:
                state["external"] = True
                mg.generate(texts, **kw)                       # warm (workspaces, packing) outside the capture
                torch.cuda.synchronize()
                _lib.call = prof_call
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    mg.generate(texts, **kw)
                _lib.call = orig
                g.replay(); torch.cuda.synchronize()
                g.replay(); torch.cuda.synchronize()
                _ = rec[0][1].elapsed_time(rec[0][2])
                how = "graph-replay"
            except Exception as ex:                            # torch without external events / capture refused: eager pass
                _lib.call = orig
                how = f"eager ({type(ex).__name__})"
                rec.clear()
                state["external"] = False
                torch.cuda.synchronize()
        if not rec:
            _lib.call = prof_call
            mg.generate(texts, **kw)
            torch.cuda.synchronize()
    finally:
        _lib.call = orig
        mg.use_cuda_graph, mg.check_fused_tail = graph_mode, check_mode
    tot = {}
    for name, e0, e1, fl in rec:
        d = tot.setdefault(name, [0.0, 0.0, 0])
        d[0] += e0.elapsed_time(e1); d[1] += fl; d[2] += 1
    all_ms = sum(v[0] for v in tot.values())
    traffic, tsrc, fused_share = None, None, 1.0
    tp = os.path.join(ROOT, "profiles", "r2_traffic.json")
    if os.path.exists(tp):                                      # dram bytes per launch of the dominant kernel, from the committed ncu capture
        tj = json.load(open(tp))
        traffic, tsrc = tj.get("tc_gemm_dram_bytes_per_launch"), tj.get("source")
        fused_share = float(tj.get("logits_fused_gemm_share", 1.0))
    # mmg_logits_fused is one entry point = GEMMs + threshold / finisher kernels: only its GEMM share (ncu launch list of the same build) counts as
    # tcgen05 GEMM time; its FLOPs are the logits GEMM's (the 1/16 sample GEMM is not counted)
    if "mmg_logits_fused" in tot:
        tot["mmg_logits_fused (GEMM share)"] = [tot["mmg_logits_fused"][0] * fused_share, tot["mmg_logits_fused"][1], tot["mmg_logits_fused"][2]]
    gemm = [tot[k] for k in ("mmg_linear", "mmg_conv2d", "mmg_conv_transpose2d", "mmg_logits_fused (GEMM share)") if k in tot]
    g_ms, g_fl, g_n = sum(v[0] for v in gemm), sum(v[1] for v in gemm), sum(v[2] for v in gemm)
    tot.pop("mmg_logits_fused (GEMM share)", None)
    achieved = g_fl / (g_ms * 1e-3) / 1e12 if g_ms > 0 else 0.0
    return {"bound": "tensor", "kernel": "tc_gemm_kernel (tcgen05; mmg_linear + mmg_conv2d + mmg_conv_transpose2d + fused logits/sampling GEMM)",
            "achieved": round(achieved, 1), "peak": pk["tflops"], "unit": "TFLOP/s", "frac": round(achieved / pk["tflops"], 4),
            "traffic": traffic, "traffic_source": tsrc, "flop_per_launch": round(g_fl / max(g_n, 1)),
            "launches": g_n, "launches_per_step_all_kernels": len(rec), "avg_launch_us": round(1e3 * g_ms / max(g_n, 1), 2),
            "share_of_step": round(g_ms / max(all_ms, 1e-9), 3), "timing": how, "logits_fused_gemm_share": fused_share,
            "by_entry_point_ms": {k: round(v[0], 3) for k, v in sorted(tot.items(), key=lambda kv: -kv[1][0])}, "peak_source": pk["src"]}


def hbm_kernels(mg, pk):
    """Achieved HBM GB/s of the VQ codebook lookup (the HBM-bound kernel north_star names) at the C5 per-GPU size (16 images x 32 x 32 tokens x
    2048 channels, bf16) and at 8x that.  Inputs larger than L2: the launches rotate over enough distinct read-only token buffers (> 2x the
    126 MB L2) that every launch streams its tokens from HBM, CUDA-event timed over the back-to-back sequence.  (Flushing by WRITING a buffer
    between launches, as the GEMM microbenchmarks do, leaves the L2 full of dirty lines whose write-back is then charged to this read-only
    kernel byte for byte: `flushed_by_write_us` keeps that figure.)"""
    from muse_maskgit_pytorch_b200 import ops
    vae = mg.vae
    P = vae._packed()
    out = {}
    flush = torch.empty((256 << 20,), dtype=torch.uint8, device="cuda")
    for name, T in (("vq_lookup_c5_per_gpu", 16384), ("vq_lookup_c5_global", 131072)):
        nbytes = T * (2048 * 2 + 8)
        nbuf = max(2, -(-(300 << 20) // nbytes))
        xs = [torch.randn((T, 2048), device="cuda").to(torch.bfloat16) for _ in range(nbuf)]
        ids = torch.empty((T,), dtype=torch.int64, device="cuda")
        call = lambda x: ops.vq_lfq_encode(x, P["pin_w"], P["pin_b"], ids, 16, w_split=P["pin_w3"])
        for x in xs:
            call(x)
        reps = 3
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(reps):
            for x in xs:
                call(x)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / (reps * nbuf)
        ts = []
        for _ in range(5):
            flush.zero_()
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record(); call(xs[0]); f1.record()
            torch.cuda.synchronize()
            ts.append(f0.elapsed_time(f1))
        gbs = nbytes / (ms * 1e-3) / 1e9
        out[name] = {"tokens": T, "bytes": nbytes, "us": round(ms * 1e3, 2), "achieved_gbs": round(gbs, 1), "frac_of_hbm_peak": round(gbs / pk["hbm"], 4),
                     "l2": f"inputs larger than L2: {nbuf} read-only token buffers of {nbytes >> 20} MB in rotation, launches back to back",
                     "flushed_by_write_us": round(sorted(ts)[len(ts) // 2] * 1e3, 2)}
        del xs
    return out


def teacher_forced_flip_rate(mg, b=2):
    """Token-id parity of the timed (bf16, tcgen05) path at the C3 model config: every decode step is fed the fp32 oracle's ids and noise;
    flip = a sampled token that differs from the oracle's.  (The oracle is the CHECKER here, tests/test_gpu_full_config.py holds the same test.)"""
    from oracle import muse_oracle as O
    tr = mg.transformer
    sd = {k: v.detach().float().cpu() for k, v in tr.state_dict().items()}
    n, V = 256, TR_CFG["num_tokens"]
    te = text_embeddings(GLOBAL_BATCH)[:b]
    g = torch.Generator().manual_seed(2)
    torch.set_num_threads(cpu_threads())

    class Trace(list):
        def append(self, st):
            st = dict(st); st.pop("logits", None); st.pop("embed", None)
            super().append(st)
    trace = Trace()
    t0 = time.perf_counter()
    O.generate_ids(sd, dict(heads=8, depth=8), te, n, V, lambda step, shape: torch.rand(shape, generator=g), timesteps=TIMESTEPS, cond_scale=COND_SCALE, trace=trace)
    t_or = time.perf_counter() - t0
    ctx = tr._prepare_context(te.cuda(), None, [False, True])
    tail = mg._tail_buffers(b, n, n, V, torch.device("cuda"), math.ceil(0.1 * V))
    flips = total = 0
    for step, st in enumerate(trace):
        ids_in = st["ids_in"].cuda()
        nm = st["num_masked"]
        mp = torch.stack([torch.nonzero(ids_in[i] == V).flatten() for i in range(b)]).int().contiguous()
        x = tr._run_blocks(ids_in, ctx, 2)
        ids = ids_in.clone(); sc = torch.full((b, n), -1e5, device="cuda")
        mg._sample_tail(x, 2, mp, nm, ids, sc, float(st["temperature"]), step, st["u"].cuda().contiguous(), COND_SCALE, math.ceil(0.1 * V), tail)
        is_mask = st["ids_in"] == V
        flips += int(((ids.cpu() != st["ids_out"]) & is_mask).sum()); total += int(is_mask.sum())
    return {"teacher_forced_flip_rate": round(flips / max(total, 1), 5), "flips": flips, "tokens": total, "sequences": b, "steps": TIMESTEPS,
            "vs": "fp32 torch-CPU oracle (pinned to the unmodified reference), same injected noise", "oracle_seconds": round(t_or, 1),
            "bound": "<= 0.08 (the reference's own bf16-vs-fp32 argmax disagreement is 3-5 %)"}


# ================================================================================================ the reference, unmodified
def cpu_threads():
    return min(os.cpu_count() or 1, int(os.environ.get("MMG_CPU_THREADS", "32")))


def build_reference(device="cpu", flash=True):
    """The UNMODIFIED reference package (baseline/_ref, pip-installed from /root/reference in the build container) with its own default
    init under torch.manual_seed(0) at the C3 config; four absent third-party packages are stood in for by tests/golden/_shims."""
    from baseline import ref_loader
    ref = ref_loader.load(512)
    torch.manual_seed(0)
    vae = ref.VQGanVAE(**VAE_CFG)
    tr = ref.MaskGitTransformer(t5_name="synth-512", flash=flash, **TR_CFG)
    mg = ref.MaskGit(image_size=IMAGE, transformer=tr, vae=vae).to(device).eval()
    return mg


def reference_generate(mg, te, timesteps=TIMESTEPS):
    mg.transformer.encode_text = lambda texts: te
    with torch.no_grad():
        return mg.generate(texts=[""] * te.shape[0], timesteps=timesteps, cond_scale=COND_SCALE, temperature=1., topk_filter_thres=0.9)


def reference_available():
    from baseline import ref_loader
    return ref_loader.available()


def cpu_baseline():
    """BASELINE.md section 4: the unmodified reference's MaskGit.generate() on this box's host cores, B_cpu = 4, full 18 steps, fp32 —
    one 2-step warm-up call, one timed call (a bounded sample of the 64-image workload: CPU throughput is flat in B)."""
    cores = cpu_threads()
    torch.set_num_threads(cores)
    if not reference_available():
        return cpu_baseline_port(cores)
    mg = build_reference("cpu")
    te = text_embeddings(GLOBAL_BATCH)[:REF_BATCH]
    torch.manual_seed(2)
    reference_generate(mg, te, timesteps=2)
    t0 = time.perf_counter()
    reference_generate(mg, te)
    dt = time.perf_counter() - t0
    return {"value": round(REF_BATCH / dt, 5), "unit": "images/s", "cores": cores, "kind": "reference",
            "sample": f"unmodified reference MaskGit.generate(), {REF_BATCH} of the 64 images, full config (18 steps, CFG=3, V=65536, 256x256, fp32), "
                      f"one timed call = {dt:.1f} s on {cores} torch threads"}


def cpu_baseline_port(cores):
    """Fallback when baseline/_ref is absent: the oracle port, 2 of 18 decode steps + the VAE decode of one image."""
    from oracle import muse_oracle as O
    import muse_maskgit_pytorch_b200 as M
    from muse_maskgit_pytorch_b200 import t5
    t5.T5_CONFIGS["synth-512"] = {"d_model": 512}
    torch.manual_seed(0)
    vae = M.VQGanVAE(**VAE_CFG)
    tr = M.MaskGitTransformer(t5_name="synth-512", **TR_CFG)
    sd = {k: v.detach().float() for k, v in tr.state_dict().items()}
    vsd = {k: v.detach().float() for k, v in vae.state_dict().items()}
    te = text_embeddings(GLOBAL_BATCH)[:1]
    g = torch.Generator().manual_seed(2)
    with torch.no_grad():
        t0 = time.perf_counter()
        ids = O.generate_ids(sd, dict(heads=8, depth=8), te, 256, 65536, lambda s, shape: torch.rand(shape, generator=g), timesteps=TIMESTEPS,
                             cond_scale=COND_SCALE, max_steps=2)
        t1 = time.perf_counter()
        O.vae_decode_from_ids(vsd, ids.clamp(max=65535).view(1, 16, 16), 16)
        t2 = time.perf_counter()
    total = TIMESTEPS * (t1 - t0) / 2 + (t2 - t1)
    return {"value": round(1.0 / total, 5), "unit": "images/s", "cores": cores, "kind": "port",
            "sample": "baseline/_ref missing: oracle port, 1 image, 2 of 18 decode steps + VAE decode timed, images/s = 1 / (18 x step + decode)"}


def gpu_eager_baseline(device):
    """The unmodified reference modules on this B200 in eager PyTorch (SURVEY.md 8d, BASELINE.md 4.4): fp32 and autocast(bf16), both through
    the reference-owned attention branch (flash=False, attend.py:123-138; the flash branch belongs to an un-vendored third-party package), global
    batch 64, one warm-up + one timed generate() each.  None of this repo's kernels run here."""
    out = {}
    if not reference_available():
        return {"unavailable": "baseline/_ref missing"}
    te = text_embeddings(GLOBAL_BATCH).to(device)
    for name, flash, autocast in (("fp32", False, False), ("autocast_bf16", False, True)):
        try:
            mg = build_reference(device, flash=flash)
            torch.manual_seed(2)
            ctx = torch.autocast("cuda", dtype=torch.bfloat16) if autocast else torch.autocast("cuda", enabled=False)
            with ctx:
                reference_generate(mg, te, timesteps=2)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                reference_generate(mg, te)
                e1.record()
                torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            out[name] = {"value": round(GLOBAL_BATCH / (ms / 1e3), 2), "unit": "images/s", "ms_per_generate": round(ms, 1), "batch": GLOBAL_BATCH}
            del mg
        except Exception as ex:
            out[name] = {"error": f"{type(ex).__name__}: {str(ex)[:160]}"}
        torch.cuda.empty_cache()
    out["note"] = "unmodified reference (baseline/_ref + stand-ins for its 4 absent third-party packages), eager PyTorch on one B200"
    return out


def run_reference(args):
    """`--impl reference`: the unmodified reference's own MaskGit.generate() (stock code path: its Transformer / Attend / VQGanVAE modules,
    its sampling tail) on the host cores.  One bench step = one full generate() of REF_BATCH images (18 steps, CFG = 3), a bounded sample of the
    64-image workload (BASELINE.md section 4).  A wall budget (MMG_REF_BUDGET_S, default 270 s) caps the number of timed steps."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    cores = cpu_threads()
    torch.set_num_threads(cores)
    base = {"impl": "reference", "metric": METRIC, "unit": "images/s", "n_gpus": args.gpus, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic"}
    if not reference_available():
        cb = cpu_baseline_port(cores)
        base.update({"value": cb["value"], "steps": 1, "warmup": 0, "ms_per_step": round(1e3 / cb["value"], 1), "cpu_baseline": cb,
                     "config": {"workload": "C3 on host cores: oracle port (baseline/_ref missing)", "global_batch": 1, "parallelism": "cpu"},
                     "e2e": {"value": cb["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
        print(json.dumps(base))
        return
    budget = float(os.environ.get("MMG_REF_BUDGET_S", "270"))
    mg = build_reference("cpu")
    te = text_embeddings(GLOBAL_BATCH)[:REF_BATCH]
    torch.manual_seed(2)
    t_start = time.perf_counter()
    warm = 1 if args.warmup > 0 else 0
    if warm:
        reference_generate(mg, te, timesteps=2)                      # allocator / thread-pool warm-up (2 of the 18 steps)
    times = []
    for i in range(args.steps):
        t0 = time.perf_counter()
        reference_generate(mg, te)
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_start + times[-1] > budget:      # the next step would overrun the wall budget
            break
    dt = sum(times) / len(times)
    v = REF_BATCH / dt
    sample = (f"unmodified reference MaskGit.generate() (baseline/_ref), {REF_BATCH} images per step, full config (18 steps, CFG=3, V=65536, 256x256, fp32), "
              f"{len(times)} timed calls of {dt:.1f} s on {cores} torch threads" + ("" if len(times) == args.steps else f" (of {args.steps} requested: wall budget {budget:.0f} s)"))
    base.update({"value": round(v, 5), "steps": len(times), "steps_requested": args.steps, "warmup": warm, "ms_per_step": round(1e3 * dt, 1),
                 "config": {"workload": "C3: MaskGit.generate() 256x256, 18 steps, cond_scale=3, top-k 0.9 — the reference's own implementation on the host cores; "
                                        "transformer dim512 depth8 V65536, VQGanVAE dim256; random-init weights, pre-computed T5 embeddings (32 positions); "
                                        f"batch {REF_BATCH} per call (a bounded sample of the 64-image workload; CPU throughput is flat in the batch size)",
                            "global_batch": REF_BATCH, "parallelism": "cpu"},
                 "cpu_baseline": {"value": round(v, 5), "unit": "images/s", "cores": cores, "kind": "reference", "sample": sample},
                 "e2e": {"value": round(v, 5), "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
    print(json.dumps(base))


# ================================================================================================ secondary configs
def _secondary_line(metric, unit, value, ms, world, args, workload, extra):
    pk = peaks()
    line = {"metric": metric, "value": round(value, 2), "unit": unit, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": round(ms, 3), "higher_is_better": True, "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": workload}, "peaks": pk}
    line.update(extra)
    return line


def run_c2(args):
    """C2: MaskGitTransformer dim 512, depth 8, seq 256, bf16 — one conditional forward (ids -> logits [B, 256, 65536] fp32), B = 64 per GPU."""
    dist, rank, world, local, device = dist_setup()
    mg = build_models(device)
    tr = mg.transformer
    B = args.batch or 64
    ids = torch.randint(0, 65537, (B, 256), device=device, generator=torch.Generator(device=device).manual_seed(3 + rank))
    te = text_embeddings(B).to(device)
    fn = lambda: tr(ids, text_embeds=te)
    for _ in range(max(args.warmup, 3)):
        fn()
    ms, launches = timed_loop(dist, world, device, fn, args.steps)
    if rank == 0:
        v = B * world / (ms / 1e3)
        pk = peaks()
        print(json.dumps(_secondary_line("sequences/sec MaskGitTransformer forward (n=256, V=65536)", "sequences/s", v, ms, world, args,
              f"C2: MaskGitTransformer dim512 depth8 seq256 bf16 conditional forward incl. to_logits on all 256 positions, batch {B} per GPU (weak scaling), eager launches",
              {"scaling": "weak", "gpu_launches": launches * args.steps,
               "dense_flop_frac_of_peak": round(v * GFLOP_C2_FORWARD / 1e3 / world / pk["tflops"], 4),
               "l2": "logits output 4.3 GB per call > L2"})))
    if world > 1:
        dist.barrier(); dist.destroy_process_group()


def run_c4(args):
    """C4: super-resolution MaskGit 512x512 (seq 1024, depth 2) conditioned on 256x256 images, global batch 32, batch-sharded."""
    dist, rank, world, local, device = dist_setup()
    from muse_maskgit_pytorch_b200 import parallel
    G = args.batch or 32
    mg = build_models(device, superres=True)
    lo, hi = parallel.shard_bounds(G, rank, world)
    te = text_embeddings(G)[lo:hi].to(device)
    cond = torch.rand((G, 3, 256, 256), generator=torch.Generator().manual_seed(4))[lo:hi].to(device)
    texts = [""] * G
    fn = lambda: parallel.generate_sharded(mg, texts, text_embeds_shard=te, cond_images_shard=cond, seed=2, timesteps=TIMESTEPS, cond_scale=COND_SCALE)
    for _ in range(max(args.warmup, 3)):
        fn()
    ms, launches = timed_loop(dist, world, device, fn, args.steps)
    if rank == 0:
        v = G / (ms / 1e3)
        pk = peaks()
        print(json.dumps(_secondary_line("images/sec super-res MaskGit.generate() 512x512 18-step CFG=3", "images/s", v, ms, world, args,
              f"C4: super-res MaskGit 512x512, seq 1024, depth 2, cond image 256 (256 conditioning tokens), 18 steps, CFG 3, global batch {G} batch-sharded; "
              "cond-VAE encode + token loop + 512x512 VAE decode + one all-gather per call",
              {"scaling": "strong", "gpu_launches": launches * args.steps,
               "dense_flop_frac_of_peak": round(v * GFLOP_C4_IMAGE / 1e3 / world / pk["tflops"], 4)})))
    if world > 1:
        dist.barrier(); dist.destroy_process_group()


def run_c5(args):
    """C5: VQGanVAE dim 256, codebook 65536: encode + VQ lookup + decode of 512x512 images, 16 per GPU (global 128 on 8 GPUs)."""
    dist, rank, world, local, device = dist_setup()
    import muse_maskgit_pytorch_b200 as M
    torch.manual_seed(0)
    vae = M.VQGanVAE(precision="bf16", **VAE_CFG).to(device)
    B = args.batch or 16
    img = torch.rand((B, 3, 512, 512), device=device, generator=torch.Generator(device=device).manual_seed(5 + rank))
    fn = lambda: vae(img)
    for _ in range(max(args.warmup, 3)):
        fn()
    ms, launches = timed_loop(dist, world, device, fn, args.steps)
    if rank == 0:
        v = B * world / (ms / 1e3)
        pk = peaks()
        print(json.dumps(_secondary_line("images/sec VQGanVAE encode+VQ+decode 512x512", "images/s", v, ms, world, args,
              f"C5: VQGanVAE dim256 codebook65536 (LFQ) forward on 512x512 images, {B} per GPU (weak scaling), eager launches",
              {"scaling": "weak", "gpu_launches": launches * args.steps,
               "dense_flop_frac_of_peak": round(v * GFLOP_C5_IMAGE / 1e3 / world / pk["tflops"], 4),
               "l2": "activations of 16 images at 512x512x256 bf16 = 2.1 GB per layer > L2"})))
    if world > 1:
        dist.barrier(); dist.destroy_process_group()


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C3", choices=["C2", "C3", "C4", "C5"])
    ap.add_argument("--batch", type=int, default=0, help="secondary configs: override the batch")
    ap.add_argument("--no-extras", "--no-cpu-baseline", dest="no_extras", action="store_true",
                    help="skip cpu_baseline / parity / gpu_eager_baseline / hbm_kernels (N=1 extras)")
    ap.add_argument("--global-batch", type=int, default=GLOBAL_BATCH, help="experiments only; the benchmark config is 64")
    ap.add_argument("--dump-outputs", metavar="DIR", help="C3: write the images of the last timed step to DIR/images.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.config != "C3"):
        ap.error("--dump-outputs applies to the C3 benchmark of this implementation")
    GLOBAL_BATCH = args.global_batch
    if args.impl == "reference":
        run_reference(args)
    else:
        with torch.no_grad():
            {"C3": run_ours, "C2": run_c2, "C4": run_c4, "C5": run_c5}[args.config](args)
