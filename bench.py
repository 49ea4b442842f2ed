#!/usr/bin/env python
"""Benchmark of the VisRAG-Ret hot path on B200 (contract: see the task statement / DESIGN.md §Measurement).

  python bench.py --gpus N --steps K --warmup W            # our CUDA path (one JSON line from rank 0)
  python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on the host cores (oracle port)

Workload = BASELINE.json configs[2]: full VisRAG-Ret (SigLIP-so400m 26 blocks + Resampler + MiniCPM-2B 40 layers,
random-init weights of that architecture) encoding synthetic 448x448 pages, plus 1 k text queries scored top-10
against a 10 k-page corpus. One step = one batch of `--pages` pages through the whole encode path.
  value : pages/s, inputs (uint8 pixels + packed token arrays) already resident in HBM, CUDA-event timed, max over ranks
  e2e   : pages/s through the reference-facing encode loop (inference.encode_stream over DRModelForInference) with HOST inputs (PIL pages):
          host prep + pinned H2D + kernels + D2H of the embeddings, every step
N > 1: one process per GPU (torchrun); every rank encodes its own `--pages` pages per step (weak scaling, no collective
in the encode path); the retrieval figure shards the corpus by page and merges partial top-k with one all-gather.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "page-images encoded/sec"
UNIT = "pages/s"


def _env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1429.0), d.get("hbm_gbs", 6585.8), "measured (MEASURED_PEAKS.json, sustained bf16)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


def burst_peak_tf():
    """Tensor peak for a kernel timed ALONE (the score filter): the burst figure; the sustained one is for the long step."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)).get("bf16_tflops", 1693.1)
    return 1700.0


class ClockSampler:
    """nvidia-smi sampling DURING the timed region (recipe in B200_PROFILING.md)."""

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, f"/tmp/vr_clocks_{os.getpid()}.csv"

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for line in open(self.path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "samples": len(sm), "reasons": sorted(reasons)}


def algorithmic_gemm_flops_per_page(n_patches: int, lm_tokens: int) -> float:
    """Dense-contraction FLOPs one page needs (SURVEY.md Appendix B), GEMMs only (attention excluded), UNPADDED dims."""
    vit = 793_046_016.0 * n_patches                       # patch-embed + 26 x (qkv, proj, fc1, fc2)
    rs = (5_308_416.0 + 21_233_664.0) * n_patches + 2 * 2 * 64 * 2304 * 2304  # kv_proj, Wk, Wv per token; out-proj + proj on 64 rows
    lm = 4_883_742_720.0 * lm_tokens
    return vit + rs + lm


def total_flops_per_page(n_patches: int, lm_tokens: int) -> float:
    return (793_046_016.0 * n_patches + 119_808.0 * n_patches ** 2 + 27_131_904.0 * n_patches + 2.0385e9
            + 4_883_742_720.0 * lm_tokens + 184_320.0 * lm_tokens ** 2)


def workload_name(a) -> str:
    """Both arms measure the same thing: pages/s of this workload (BASELINE.json configs[2])."""
    return (f"BASELINE configs[2]: full VisRAG-Ret (SigLIP-so400m x26 + Resampler + MiniCPM-2B x40) encode of synthetic "
            f"{a.page_px}x{a.page_px} pages")


# --------------------------------------------------------------------------------------------- our arm
def run_ours(a):
    import numpy as np
    import torch
    import torch.distributed as dist
    from PIL import Image

    from visrag_b200 import _lib as L
    from visrag_b200 import ops, retriever
    from visrag_b200.config import VisRAGConfig
    from visrag_b200.host import prepare_batch
    from visrag_b200.modeling import DRModelForInference, VisRAGRetB200
    from visrag_b200.tokenizer_stub import StubTokenizer
    from visrag_b200.weights import random_state_dict_device

    rank, world, local = _env_int("RANK", 0), _env_int("WORLD_SIZE", 1), _env_int("LOCAL_RANK", 0)
    if world != a.gpus and world > 1:
        raise SystemExit(f"--gpus {a.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    if world > 1:
        # NCCL writes its "NCCL version ..." banner to STDOUT when the first communicator is created (whenever NCCL_DEBUG
        # is set, as it is on the GPU boxes); stdout must carry exactly one JSON line, so the banner is sent to stderr
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device(dev))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    cfg = VisRAGConfig.full() if a.model == "full" else VisRAGConfig.tiny()
    tok = StubTokenizer(cfg.vocab)
    t0 = time.time()
    sd = random_state_dict_device(cfg, 2024 + rank, dev)
    lm = VisRAGRetB200(cfg, sd, dev)
    eng = lm.engine
    model = DRModelForInference(lm_q=lm, pooling="wmean", normalize=True)
    if not (rank == 0 and world == 1 and (a.cpu_baseline or a.torch_baseline)):
        del sd
    torch.cuda.empty_cache()
    setup_s = time.time() - t0

    # ---- synthetic pages: uint8 448x448 noise (single slice, 1024 patches, 68 LM tokens)
    P = a.pages
    rs = np.random.RandomState(1000 + rank)
    page_arrays = rs.randint(0, 256, (P, a.page_px, a.page_px, 3), dtype=np.uint8)
    pages = [Image.fromarray(x) for x in page_arrays]
    items = {"id": [f"d{i}" for i in range(P)], "text": [""] * P, "image": pages}
    pb = prepare_batch(items["text"], pages, tok, cfg, 2048)
    groups, src, pos, cu = eng.upload(pb)
    max_len = int(pb.seq_lens.max())
    n_patches = (a.page_px // 14) ** 2 if a.page_px % 14 == 0 else None
    lm_tokens = float(pb.seq_lens.mean())

    def step_device():
        return eng.encode_device(groups, pb.group_row0, pb.n_slices, src, pos, cu, max_len)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- (1) device-resident throughput
    for _ in range(a.warmup):
        step_device()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = L.LAUNCHES
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(a.steps):
        reps = step_device()
    e1.record()
    barrier()
    launches = L.LAUNCHES - launches0
    dumped = {"page_reps": reps.float().cpu().numpy()} if a.dump_outputs else None
    clocks = sampler.stop() if rank == 0 else None
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    value = world * a.steps * P / (ms_total / 1e3)

    # ---- (2) end to end through the reference-facing encode loop: host PIL pages -> device -> embeddings on host.
    # `encode_stream` is the core of distributed_parallel_embedding_inference (reference inference.py:53-172): every batch
    # is prepared on the host (slicing, resampling, tokenising), uploaded from pinned memory, encoded and read back; the
    # host preparation of batch i+1 overlaps the kernels of batch i. The fill (first batch's preparation) is inside the
    # timed region. `blocking` is the same work through one synchronous model(passage=...) call per step.
    from visrag_b200.inference import encode_stream
    kw = {"tokenizer": tok, "max_inp_length": 2048}
    stream_items = dict(items, id=[str(i) for i in range(P)])
    for _ in encode_stream([stream_items] * max(2, a.warmup - 1), model, kw):
        pass
    barrier()
    e0.record()
    marks = [time.perf_counter()]
    for _, host_np in encode_stream([stream_items] * a.steps, model, kw):
        marks.append(time.perf_counter())  # batch i's embeddings are on the host
    e1.record()
    barrier()
    e2e_ms = max_over_ranks(e0.elapsed_time(e1))
    intervals = [round((b - a_) * 1e3, 1) for a_, b in zip(marks, marks[1:])]  # first one includes the pipeline fill
    e2e_value = world * a.steps * P / (e2e_ms / 1e3)
    host_reps = torch.from_numpy(host_np)
    if dumped is not None:
        dumped["e2e_page_reps"] = host_np.astype(np.float32)
    e0.record()
    for _ in range(a.steps):
        model(passage=items, tokenizer=tok, max_inp_length=2048).p_reps.cpu()
    e1.record()
    barrier()
    blocking_ms = max_over_ranks(e0.elapsed_time(e1))
    blocking_value = world * a.steps * P / (blocking_ms / 1e3)
    pb_e2e = model.prepare(stream_items, **kw)  # what the e2e path really uploads (raw RGBX pages with the device front-end)
    h2d = int(pb_e2e.pixel_bytes() + pb_e2e.token_src.nbytes + pb_e2e.positions.nbytes + pb_e2e.cu_seqlens.nbytes)
    d2h = int(host_reps.numel() * 4)
    assert torch.isfinite(host_reps).all()

    # ---- (3) roofline pass: CUDA events around every launch (separate from the timed regions above)
    ops.profile_begin()
    for _ in range(2):
        step_device()
    prof = ops.profile_end()
    peak_tf, peak_hbm, peak_src = load_peaks()
    gemm_classes = {k: v for k, v in prof.items() if k.startswith("gemm:")}
    gemm_n = sum(v[0] for v in gemm_classes.values())
    gemm_ms = sum(v[1] for v in gemm_classes.values())
    gemm_padded_flops = sum(v[2] for v in gemm_classes.values())
    all_ms = sum(v[1] for v in prof.values())
    roofline, shares = None, {}
    if gemm_n and n_patches:
        alg = algorithmic_gemm_flops_per_page(n_patches, lm_tokens) * P * 2  # two profiled steps
        achieved = alg / (gemm_ms / 1e3) / 1e12
        # the single heaviest launch class (same kernel template, one shape + epilogue)
        top_k, (top_n, top_ms, top_fl) = max(gemm_classes.items(), key=lambda kv: kv[1][1])
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "gemm_traffic.json")
        if os.path.exists(tpath):
            traffic = json.load(open(tpath)).get(top_k)
        roofline = {"bound": "tensor", "kernel": "gemm_tcgen05_kernel (all launches of the step; epilogue variants bias/GELU/resid/RoPE/SwiGLU)",
                    "achieved": round(achieved, 1), "peak": peak_tf, "unit": "TFLOP/s", "frac": round(achieved / peak_tf, 4),
                    "traffic": traffic, "peak_source": peak_src, "launches_per_step": gemm_n // 2,
                    "avg_launch_ms": round(gemm_ms / gemm_n, 4), "padded_tflops": round(gemm_padded_flops / (gemm_ms / 1e3) / 1e12, 1),
                    "heaviest_class": {"shape": top_k, "launches_per_step": top_n // 2, "avg_launch_ms": round(top_ms / top_n, 4),
                                       "tflops": round(top_fl / (top_ms / 1e3) / 1e12, 1), "share_of_gemm_time": round(top_ms / gemm_ms, 3)},
                    # every launch class of the step: [launches/step, avg ms, padded TFLOP/s, share of GEMM time]
                    "classes": {k: [v[0] // 2, round(v[1] / v[0], 4), round(v[2] / (v[1] / 1e3) / 1e12, 1), round(v[1] / gemm_ms, 3)]
                                for k, v in sorted(gemm_classes.items(), key=lambda kv: -kv[1][1])}}
        shares = {}
        for k, v in prof.items():
            kk = "gemm" if k.startswith("gemm:") else k
            shares[kk] = round(shares.get(kk, 0.0) + v[1] / all_ms, 4)

    # ---- (4) queries: encode text queries + exact top-10 over a page-sharded corpus.
    # Corpus sharded by page (rank r holds pages shard_range(nd*world, r, world)); the query ENCODE is sharded by rank as in
    # the reference (dense_retriever.py:48-50): rank r encodes queries shard_range(nq, r, world), ONE all-gather of the
    # [nq/world, 2304] fp32 embeddings makes them global, every rank scores all queries against its shard, ONE all-gather
    # of [nq, 10] (score, id) pairs + a k-way merge finishes (retriever.gather_queries / sharded_topk).
    nq, nd = a.queries, a.corpus
    from visrag_b200.synth import synth_queries
    qtexts = synth_queries(nq, 7)
    g = torch.Generator(device=dev).manual_seed(5 + rank)
    lo, hi = retriever.shard_range(nd * world, rank, world)
    corpus = torch.nn.functional.normalize(torch.randn(hi - lo, cfg.hidden, device=dev, generator=g), dim=1)
    index = retriever.build_index(corpus)
    qb = a.query_batch
    qlo, qhi = retriever.shard_range(nq, rank, world)
    my_q = qtexts[qlo:qhi]

    def encode_my_queries():
        outs = [eng.encode(my_q[i:i + qb], [None] * len(my_q[i:i + qb]), tok) for i in range(0, len(my_q), qb)]
        local = torch.cat(outs) if outs else torch.zeros((0, cfg.hidden), dtype=torch.float32, device=dev)
        return retriever.gather_queries(local, nq)

    def queries_step():
        qe = encode_my_queries()
        s, ids = retriever.sharded_topk(qe, index, 10, lo)
        return s.cpu(), ids.cpu(), qe

    queries_step()
    barrier()
    e0.record()
    for _ in range(a.query_reps):
        s_top, i_top, qe_all = queries_step()
    e1.record()
    barrier()
    q_ms = max_over_ranks(e0.elapsed_time(e1)) / a.query_reps
    if dumped is not None:
        dumped.update(query_reps=qe_all.float().cpu().numpy(), query_top10_scores=s_top.float().numpy(),
                      query_top10_ids=i_top.numpy().astype(np.float64))  # ids are exact in float64
    qe = torch.nn.functional.normalize(torch.randn(nq, cfg.hidden, device=dev, generator=torch.Generator(device=dev).manual_seed(77)), dim=1)
    retriever.sharded_topk(qe, index, 10, lo)
    barrier()
    e0.record()
    for _ in range(a.query_reps):
        retriever.sharded_topk(qe, index, 10, lo)
    e1.record()
    barrier()
    r_ms = max_over_ranks(e0.elapsed_time(e1)) / a.query_reps

    def check_against_torch(q_all, idx, lo_, k=10, n_check=64):
        """Correctness under NCCL, outside every timed region: the sharded result of `n_check` queries vs an independent
        route - torch.matmul + torch.topk on every rank's fp32 shard, all_gather of those partial lists, torch.topk merge.
        Raises on any id mismatch (scores within 2e-6)."""
        sub = q_all[:n_check].contiguous()
        got_s, got_i = retriever.sharded_topk(sub, idx, k, lo_)
        ref = torch.topk(sub @ idx.emb.T, k, dim=1)
        ref_s, ref_i = ref.values.contiguous(), (ref.indices + lo_).contiguous()
        if world > 1:
            all_s = [torch.empty_like(ref_s) for _ in range(world)]
            all_i = [torch.empty_like(ref_i) for _ in range(world)]
            dist.all_gather(all_s, ref_s)
            dist.all_gather(all_i, ref_i)
            cs, ci = torch.cat(all_s, dim=1), torch.cat(all_i, dim=1)
            top = torch.topk(cs, k, dim=1)
            ref_s, ref_i = top.values, torch.gather(ci, 1, top.indices)
        ok = bool(torch.equal(got_i, ref_i)) and float((got_s - ref_s).abs().max()) <= 2e-6
        if not ok:
            raise SystemExit(f"rank {rank}: sharded_topk disagrees with the torch fp32 route under world={world}")
        return n_check

    checked = check_against_torch(qe, index, lo)
    # every rank must hold the same global query embeddings after gather_queries (bitwise)
    if world > 1:
        ref_q = qe_all.clone()
        dist.broadcast(ref_q, 0)
        if not torch.equal(ref_q, qe_all):
            raise SystemExit(f"rank {rank}: gathered query embeddings differ from rank 0's")

    # ---- (4b) BASELINE configs[3] retrieval at its stated size: `--big-corpus` pages per GPU (125 000 x 8 = 1 M) resident as
    # fp32 + fp16, `--big-queries` queries, top-10, staged timing (filter / rescore / all-gather / merge)
    big = None
    if a.big_corpus > 0:
        del index, corpus
        torch.cuda.empty_cache()
        blo, bhi = retriever.shard_range(a.big_corpus * world, rank, world)
        gen = torch.Generator(device=dev).manual_seed(900 + rank)
        bc = torch.empty((bhi - blo, cfg.hidden), dtype=torch.float32, device=dev)
        for r0 in range(0, bhi - blo, 32768):
            x = torch.randn((min(32768, bhi - blo - r0), cfg.hidden), device=dev, generator=gen)
            bc[r0:r0 + x.shape[0]] = torch.nn.functional.normalize(x, dim=1)
        barrier()
        e0.record()
        bindex = retriever.build_index(bc)
        e1.record()
        barrier()
        build_ms = max_over_ranks(e0.elapsed_time(e1))
        bq = torch.nn.functional.normalize(torch.randn(a.big_queries, cfg.hidden, device=dev,
                                                       generator=torch.Generator(device=dev).manual_seed(901)), dim=1)
        st = {}
        retriever.sharded_topk(bq, bindex, 10, blo, stats=st)
        barrier()
        st = {"stages": {}}
        e0.record()
        for _ in range(a.query_reps):
            retriever.sharded_topk(bq, bindex, 10, blo, stats=st)
        e1.record()
        barrier()
        big_ms = max_over_ranks(e0.elapsed_time(e1)) / a.query_reps
        stages = {k: round(v / a.query_reps, 3) for k, v in retriever.resolve_stages(st).items()}
        filt_tf = 2.0 * a.big_queries * (bhi - blo) * cfg.hidden / (stages.get("filter", float("inf")) / 1e3) / 1e12
        checked_big = check_against_torch(bq, bindex, blo)
        big = {"workload": "BASELINE configs[3]: synthetic unit-norm corpus sharded by page, index build (fp32 -> fp16 copy + row norms) + "
                           "top-10 of every query over the FULL corpus with the partial-top-k all-gather",
               "corpus_pages": a.big_corpus * world, "pages_per_gpu": bhi - blo, "queries": a.big_queries, "k": 10,
               "index_build_ms": round(build_ms, 2), "ms_per_query_batch": round(big_ms, 3),
               "queries_per_s": round(a.big_queries / (big_ms / 1e3), 1), "stages_ms_rank0": stages,
               "filter_tflops_fp16_per_gpu": round(filt_tf, 1), "filter_frac_of_tensor_peak": round(filt_tf / burst_peak_tf(), 3),
               "filter_peak": "burst dense bf16/fp16 figure of MEASURED_PEAKS.json (a kernel timed alone, not inside the encode step)",
               "flagged": st.get("flagged"), "checked_queries_vs_torch_fp32": checked_big}

    # ---- (4c) the reference's own operating point (eval.sh: per-device batch 16) and the demo's single query, blocking API
    small = None
    if a.small_batch > 0 and P >= a.small_batch:
        sb_items = {k: v[: a.small_batch] for k, v in items.items()}
        for _ in range(3):
            model(passage=sb_items, tokenizer=tok, max_inp_length=2048).p_reps.cpu()
        barrier()
        e0.record()
        for _ in range(10):
            model(passage=sb_items, tokenizer=tok, max_inp_length=2048).p_reps.cpu()
        e1.record()
        barrier()
        sb_ms = max_over_ranks(e0.elapsed_time(e1)) / 10
        q1 = {"id": ["q"], "text": [qtexts[0]], "image": [None]}
        idx1 = retriever.build_index(torch.nn.functional.normalize(
            torch.randn(nd, cfg.hidden, device=dev, generator=torch.Generator(device=dev).manual_seed(3)), dim=1))

        def one_query():
            qv = model(query=q1, tokenizer=tok, max_inp_length=2048).q_reps
            return retriever.score_topk(qv, idx1, 10)[1].cpu()

        for _ in range(3):
            one_query()
        barrier()
        t_q = time.perf_counter()
        for _ in range(20):
            one_query()
        torch.cuda.synchronize()
        q_lat_ms = (time.perf_counter() - t_q) / 20 * 1e3
        small = {"pages_per_s_batch": a.small_batch, "pages_per_s": round(world * a.small_batch / (sb_ms / 1e3), 1),
                 "ms_per_batch": round(sb_ms, 2), "api": "DRModelForInference.forward(passage=...).p_reps.cpu(), host PIL pages in",
                 "single_query_encode_plus_top10_ms": round(q_lat_ms, 2), "single_query_corpus_pages": nd}
        del idx1

    # ---- (4d) context arm: the same step in stock PyTorch on this GPU (bf16, cuBLAS linears, SDPA attention, batched over the
    # pages; tools/torch_gpu_baseline.py - none of this repo's kernels), pixels and tokens resident like `value`. Outside
    # every timed region above; reported beside the CPU arm so the hand-written kernels are also placed against cuBLAS + FA.
    torch_arm = None
    if rank == 0 and world == 1 and a.torch_baseline and n_patches and bool((pb.seq_lens == max_len).all()):
        from tools.torch_gpu_baseline import TorchPageEncoder
        tenc = TorchPageEncoder(sd, cfg)
        px_dev = torch.from_numpy(page_arrays).to(dev)
        src_dev = torch.from_numpy(np.asarray(pb.token_src)).to(dev)
        for _ in range(2):
            t_reps = tenc.encode(px_dev, src_dev, max_len)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(3):
            t_reps = tenc.encode(px_dev, src_dev, max_len)
        e1.record()
        torch.cuda.synchronize()
        t_ms = e0.elapsed_time(e1) / 3
        cos = torch.nn.functional.cosine_similarity(t_reps.float(), reps.float(), dim=1)
        torch_arm = {"value": round(P / (t_ms / 1e3), 1), "unit": UNIT, "ms_per_step": round(t_ms, 2),
                     "impl": f"plain PyTorch {torch.__version__} on the same GPU: bf16 weights and activations, F.linear (cuBLAS), "
                             "F.scaled_dot_product_attention, F.layer_norm, batched over all pages, inputs resident",
                     "cosine_vs_engine_min": round(float(cos.min()), 5), "engine_speedup": round(value / (P / (t_ms / 1e3)), 2)}
        del tenc, px_dev, t_reps
        torch.cuda.empty_cache()

    # ---- (5) CPU baseline: the oracle port of the reference algorithm on the host cores (rank 0, N = 1 only)
    cpu_baseline = None
    if rank == 0 and world == 1 and a.cpu_baseline:
        cpu_baseline = cpu_port_baseline(cfg, {k: v.float().cpu() for k, v in sd.items()}, tok, pages[: a.cpu_pages], a.page_px)
    sd = None

    if rank == 0:
        line = {
            "metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": round(ms_total / a.steps, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": workload_name(a), "queries": f"{nq} text queries top-10 over {nd * world} pages",
                       "size": a.model, "pages_per_step_per_gpu": P, "global_batch": P * world, "patches_per_page": n_patches,
                       "lm_tokens_per_page": lm_tokens, "parallelism": f"dp{world} (pages sharded, no encode collective)",
                       "weights": "random-init, bf16", "l2": "working set (6.3 GB weights + >1 GB activations per step) >> 126 MB L2"},
            "e2e": {"value": round(e2e_value, 2), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": round(e2e_ms / a.steps, 3), "batch_intervals_ms": intervals,
                    "api": "inference.encode_stream (loop body of distributed_parallel_embedding_inference) over DRModelForInference",
                    "inputs": "the same 128 host PIL pages every step: nothing in the prep path caches per image (only the placeholder "
                              "string is memoised), but Pillow's zero-copy row export always finds the pages warm in the host caches",
                    "blocking": {"value": round(blocking_value, 2), "ms_per_step": round(blocking_ms / a.steps, 3),
                                 "api": "DRModelForInference.forward(passage=..., tokenizer=...).p_reps.cpu() per step"}},
            "gpu_launches": launches, "clocks": clocks,
            "roofline": roofline, "kernel_time_share": shares,
            "model_tflops": round(total_flops_per_page(n_patches, lm_tokens) * value / 1e12 / world, 1) if n_patches else None,
            "queries": {"queries_per_s_encode_plus_top10": round(nq / (q_ms / 1e3), 1), "retrieve_only_queries_per_s": round(nq / (r_ms / 1e3), 1),
                        "n_queries": nq, "corpus_pages": nd * world, "k": 10,
                        "lm_tokens_per_query": round(sum(len(tok.encode(t)) for t in qtexts[:64]) / max(1, len(qtexts[:64])), 1),
                        "tokenizer": "character-level stub (no SentencePiece model ships with the reference): ~4x the tokens a real one gives", "query_encode": f"sharded by rank ({qhi - qlo} of {nq} on rank 0)",
                        "collectives": (["all_gather_into_tensor of [ceil(nq/world), 2304] fp32 query embeddings",
                                         "all_gather_into_tensor of [nq, 10] (score, id) pairs"] if world > 1 else []),
                        "checked_vs_torch_fp32_under_nccl": checked},
            "retrieval_configs3": big, "small_batch": small,
            "cpu_baseline": cpu_baseline, "torch_gpu_baseline": torch_arm, "setup_s": round(setup_s, 1),
        }
        print(json.dumps(line), flush=True)
        if dumped is not None:
            dump_outputs(a.dump_outputs, dumped)
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir, arrays):
    """Writes what the timed paths returned in their last step as out_dir/<name>.npy (rank 0's share when N > 1):
    page_reps       [pages, 2304] embeddings of the device-resident step (`value`)
    e2e_page_reps   [pages, 2304] embeddings the host received from the last step of the e2e loop
    query_reps      [queries, 2304] encoded text queries, query_top10_scores / _ids [queries, 10] their top-10.
    All inputs are seeded, so runs with the same arguments compare output for output. Above 64 MB in all, every array
    keeps the same fraction of its rows, chosen with a fixed seed (the same rows in every run with these arguments)."""
    import numpy as np

    limit = 64 << 20
    total = sum(x.nbytes for x in arrays.values())
    os.makedirs(out_dir, exist_ok=True)
    for name, x in arrays.items():
        assert x.dtype in (np.float32, np.float64), (name, x.dtype)
        if total > limit:
            keep = max(1, len(x) * limit // total)
            x = x[np.sort(np.random.RandomState(0).choice(len(x), keep, replace=False))]
        np.save(os.path.join(out_dir, f"{name}.npy"), x)


def cpu_port_baseline(cfg, sd_cpu, tok, pages, page_px):
    """Times oracle/restated.py (the CPU port of the reference algorithm) on a bounded sample of the same workload."""
    import torch

    from oracle import restated as O

    threads = pick_cpu_threads()
    torch.set_num_threads(threads)
    t0, done = time.time(), 0
    for pg in pages:  # bounded sample: stop after ~25 s of CPU work
        O.encode(sd_cpu, cfg, tok, [""], [pg])
        done += 1
        if time.time() - t0 > 25.0:
            break
    dt = time.time() - t0
    # the reference's retrieval step on the same host cores (SURVEY 8d): fp32 Q.D^T + top-10, 1 000 queries x 10 000 pages
    import numpy as np
    rs = np.random.RandomState(3)
    Dh = rs.randn(10000, cfg.hidden).astype(np.float32)
    Qh = rs.randn(1000, cfg.hidden).astype(np.float32)
    O.score_topk(Qh[:64], Dh, 10)
    t1 = time.time()
    O.score_topk(Qh, Dh, 10)
    rt = time.time() - t1
    cpu_model = ""
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                cpu_model = ln.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    return {"value": round(done / dt, 4), "unit": UNIT, "cores": threads, "host_cpus": os.cpu_count(), "cpu_model": cpu_model, "kind": "port",
            "sample": f"{done} pages {page_px}x{page_px}, {'full' if cfg.layers == 40 else 'reduced'} model, fp32, oracle/restated.py", "seconds": round(dt, 1),
            "retrieval": {"queries_per_s": round(1000 / rt, 1), "sample": "1000 queries x 10000 pages x 2304, fp32 matmul + top-10 (oracle.score_topk)",
                          "seconds": round(rt, 2)}}


def pick_cpu_threads():
    """All host threads is not the fastest setting for these GEMM sizes on a many-core box (oversubscription): time a
    ViT-block-sized matmul at a few thread counts and keep the best, so the baseline is the CPU's best case."""
    import torch

    n = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 64, n) if c <= n})
    a, b = torch.randn(1024, 1152), torch.randn(1152, 4304)
    best, best_t = n, float("inf")
    for c in cands:
        torch.set_num_threads(c)
        torch.mm(a, b)
        t0 = time.time()
        for _ in range(5):
            torch.mm(a, b)
        dt = time.time() - t0
        if dt < best_t:
            best, best_t = c, dt
    return best


# --------------------------------------------------------------------------------------------- reference arm
def run_reference(a):
    """The reference's algorithm on the host cores. The reference itself is pure Python over PyTorch and cannot travel to
    the GPU box (/root/reference is absent there), so this runs its oracle port (validated against the real reference in the
    build container, tests/golden). Each step = ONE page through the full model; rank 0 only."""
    rank = _env_int("RANK", 0)
    if rank != 0:
        return
    import numpy as np
    import torch
    from PIL import Image

    from oracle import restated as O
    from visrag_b200.config import VisRAGConfig
    from visrag_b200.tokenizer_stub import StubTokenizer
    from visrag_b200.weights import random_state_dict, random_state_dict_device

    cfg = VisRAGConfig.full() if a.model == "full" else VisRAGConfig.tiny()
    tok = StubTokenizer(cfg.vocab)
    if torch.cuda.is_available():  # draw the 3.1 B weights on the GPU (seconds) and move them to the host; compute stays on the CPU
        sd = {k: v.float().cpu() for k, v in random_state_dict_device(cfg, 2024, "cuda:0").items()}
    else:
        sd = random_state_dict(cfg, 2024)
    threads = pick_cpu_threads()
    torch.set_num_threads(threads)
    rs = np.random.RandomState(1000)
    n = a.steps + a.warmup
    pages = [Image.fromarray(rs.randint(0, 256, (a.page_px, a.page_px, 3), dtype=np.uint8)) for _ in range(n)]
    budget_s = 150.0  # the whole arm must end within a few minutes whatever K the driver passes
    t_w = time.time()
    for i in range(a.warmup):
        O.encode(sd, cfg, tok, [""], [pages[i]])
        if time.time() - t_w > 30.0:
            break
    t0, done = time.time(), 0
    for i in range(a.warmup, n):
        O.encode(sd, cfg, tok, [""], [pages[i]])
        done += 1
        if time.time() - t0 > budget_s:
            break
    dt = time.time() - t0
    a.steps = done
    v = done / dt
    sample = f"{a.steps} steps x 1 page {a.page_px}x{a.page_px}, full model fp32 on host cores"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": round(v, 4), "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": round(dt / a.steps * 1e3, 1), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(a), "size": a.model, "pages_per_step_per_gpu": 1,
                   "sample": "each step is ONE page of the workload through the full model on the host cores"},
        "cpu_baseline": {"value": round(v, 4), "unit": UNIT, "cores": threads, "host_cpus": os.cpu_count(), "kind": "port", "sample": sample},
        "e2e": {"value": round(v, 4), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="full", choices=["full", "tiny"])
    ap.add_argument("--pages", type=int, default=128, help="pages per step per GPU")
    ap.add_argument("--page-px", type=int, default=448)
    ap.add_argument("--queries", type=int, default=1000)
    ap.add_argument("--corpus", type=int, default=10000, help="corpus pages per GPU for the retrieval figure")
    ap.add_argument("--big-corpus", type=int, default=-1,
                    help="pages per GPU of the configs[3] retrieval leg (default: 125000 when N > 1, off at N = 1; 0 = off)")
    ap.add_argument("--big-queries", type=int, default=10000)
    ap.add_argument("--small-batch", type=int, default=16, help="pages per call of the small-batch figure (0 = off)")
    ap.add_argument("--query-batch", type=int, default=500)
    ap.add_argument("--query-reps", type=int, default=3)
    ap.add_argument("--cpu-pages", type=int, default=2)
    ap.add_argument("--no-cpu-baseline", dest="cpu_baseline", action="store_false")
    ap.add_argument("--no-torch-baseline", dest="torch_baseline", action="store_false",
                    help="skip the stock-PyTorch-on-this-GPU context arm (N = 1 only)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the outputs of their last step to DIR/<name>.npy (see dump_outputs)")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs is only implemented for --impl ours")
    if a.warmup < 3 and a.impl == "ours":
        a.warmup = 3
    if a.big_corpus < 0:
        a.big_corpus = 125000 if a.gpus > 1 else 0
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
