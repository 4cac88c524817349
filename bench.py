#!/usr/bin/env python
"""Headline benchmark: SEAL constrained beam-search decode, queries/sec at beam 15 on a synthetic
10 M-token FM-index with BART-large (BASELINE.json metric / configs[1]; SURVEY.md §8d).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --steps K --warmup W    # the reference's algorithm on host cores
    python bench.py ... --dump-outputs DIR                   # also save the last timed step's records as DIR/*.npy

One "step" = one full pass of the hot path (encoder, 9 constrained decode steps, hypothesis records, the
single gather of the records to rank 0) over the 1 000-query batch.  With N GPUs the SAME 1 000 queries are
sharded in contiguous blocks (strong scaling, BASELINE.json configs[3]); `--scaling weak` gives every GPU its
own 1 000.  Prints ONE JSON line (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "queries/sec at beam=15, 1k queries, 10M-token index; rank-kernel HBM GB/s"
BEAM, MIN_LEN, MAX_LEN, LP = 15, 10, 10, 0.0          # SEALSearcher body defaults (retrieval.py:70-83)
# dram__bytes_read.sum + dram__bytes_write.sum per launch of the fc1-shaped GEMM (M=15000, N=4096, K=1024) from
# `ncu --set full` (profiles/r01_ncu_2cta_fc1_raw.csv); algorithmic bytes of that launch: A halves 61 MB + W halves
# 17 MB + C halves 246 MB = 324 MB, of which the activations/weights mostly hit L2.
TRAFFIC_PER_LAUNCH = {2: 438.3e6, 3: 290.8e6, 5: 296.5e6}      # 5: profiles/r02_c_ncu_2cta_fc1_raw.csv (86.5 MB read + 210.0 MB written)
TOL = 1e-4                                             # BASELINE.json north_star: beam scores within 1e-4


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), float(p["bf16_tflops"]), float(p.get("bf16_tflops_sustained", p["bf16_tflops"])), "measured"
    except Exception:
        return 6650.0, 1590.0, 1400.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) < 9:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def build_inputs(n_queries, seed):
    from seal_b200.synthetic import make_corpus, make_queries        # pure numpy: does not load libsealb200.so
    docs = make_corpus()                                     # 100 000 docs x 100 tokens, seed 1234
    ids, mask = make_queries(n_queries, seed=seed)
    return docs, ids, mask


def make_model(freq_bias=None):
    import torch
    from transformers import BartConfig, BartForConditionalGeneration
    cfg = BartConfig()                                       # defaults == facebook/bart-large
    cfg.forced_bos_token_id = None                           # seal/retrieval.py:566,580
    torch.manual_seed(0)
    model = BartForConditionalGeneration(cfg).eval().float()
    with torch.no_grad():
        if freq_bias is not None:                            # regime "freq": SURVEY.md 8d (retrieval.py:584-588 edits this buffer)
            model.final_logits_bias[0, :] = torch.from_numpy(freq_bias)
        for t in (cfg.pad_token_id, cfg.bos_token_id, cfg.vocab_size - 1):
            model.final_logits_bias[0, t] = float("-inf")    # seal/retrieval.py:584-588
    return model


def unigram_log_freq(docs, vocab):
    """final_logits_bias = log(unigram corpus frequency) (tokens absent from the corpus: the smallest present one)."""
    cnt = np.bincount(docs.reshape(-1), minlength=vocab).astype(np.float64)
    lf = np.log(np.maximum(cnt, 1.0) / cnt.sum())
    return lf.astype(np.float32)


def decode_trace(rec, max_triples=1 << 22):
    """(symbol, lo, hi_inclusive) LF triples of the decode itself, rebuilt from the hypothesis records: a record of
    length n extends the record of its first n-1 tokens (its parent beam) by one backward-search step."""
    lens, toks, valid, lo, hi = rec["lens"], rec["tokens"], rec["valid"], rec["lo"], rec["hi"]
    sym, plo, phi = [], [], []
    Q, H = lens.shape
    for q in range(Q):
        ranges = {}
        for h in range(H):
            if valid[q, h]:
                ranges[tuple(toks[q, h, :lens[q, h]])] = (int(lo[q, h]), int(hi[q, h]))
        for key, _ in ranges.items():
            par = ranges.get(key[:-1])
            if par is not None and par[1] > par[0]:
                sym.append(key[-1] + 10); plo.append(par[0]); phi.append(par[1] - 1)
        if len(sym) >= max_triples:
            break
    return np.asarray(sym, dtype=np.int64), np.asarray(plo, dtype=np.int64), np.asarray(phi, dtype=np.int64)


# ------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    import ctypes as C
    from seal_b200._lib import lib, check
    from seal_b200.beam_search import (SealBartEngine, DeviceRecords, generate_records_device, generate_records,
                                       sharded_generate_records)
    from seal_b200.index import FMIndex
    from seal_b200.sharding import RecordLayout, shard_bounds, gather_buffers, merge_gathered
    from seal_b200.synthetic import corpus_symbols

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    strong = args.scaling == "strong"
    Qtot = args.queries if strong else args.queries * world
    docs, ids_all, mask_all = build_inputs(args.queries, seed=4321 if strong else 4321 + rank)
    if strong:
        q_lo, q_hi = shard_bounds(args.queries, world, rank)
        n_max = max(shard_bounds(args.queries, world, r)[1] - shard_bounds(args.queries, world, r)[0] for r in range(world))
    else:
        q_lo, q_hi, n_max = 0, args.queries, args.queries
    ids_np = np.ascontiguousarray(ids_all[q_lo:q_hi]); mask_np = np.ascontiguousarray(mask_all[q_lo:q_hi])
    Q = q_hi - q_lo
    # build straight from the symbol stream (same result as FMIndex.initialize, without 100k Python lists)
    from seal_b200.cpp_modules.fm_index import FMIndex as RawFM
    index = FMIndex()
    RawFM.initialize(index, corpus_symbols(docs))
    index.beginnings = list(range(0, docs.size + 1, docs.shape[1]))
    index._sync_beginnings()
    index.to_device(local)
    index.occurring_distinct, index.occurring_counts = index.get_distinct_count(0, len(index))
    freq = unigram_log_freq(docs, 50265) if args.regime == "freq" else None
    model = make_model(freq)
    eng = SealBartEngine.from_hf(model, device=local, gemm_mode=args.gemm_mode)
    cfg = model.config
    del model
    kw = dict(min_length=MIN_LEN, max_length=MAX_LEN, length_penalty=LP, num_beams=BEAM, forced_bos_token_id=None)
    H = (MAX_LEN - 1) * 2 * BEAM + BEAM
    layout = RecordLayout(max(n_max, 1), H, MAX_LEN)
    rec = DeviceRecords(layout, dev)
    ids = torch.from_numpy(ids_np).to(dev); mask = torch.from_numpy(mask_np).to(dev)
    src_tokens = int(mask_np.sum())                          # right-padded by construction (seal_b200.synthetic)
    stream = torch.cuda.Stream(device=dev)
    gathered = None

    def step_device(gather=True):
        nonlocal gathered
        with torch.cuda.stream(stream):
            if Q:
                generate_records_device(eng, index, ids, mask, out=rec, src_tokens=src_tokens, stream=stream, **kw)
            if world > 1 and gather:                     # the single collective: every rank's record buffer to rank 0
                gathered = gather_buffers(rec.buf, dst=0)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step_device()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    barrier()
    prof_range = bool(os.environ.get("SEAL_PROFILE_RANGE"))   # ncu --profile-from-start off: capture the timed steps only
    if prof_range:
        torch.cuda.profiler.start()
    e0.record(stream)
    for _ in range(args.steps):
        step_device()
    e1.record(stream)
    barrier()
    if prof_range:
        torch.cuda.profiler.stop()
    ms = e0.elapsed_time(e1)
    used_graph = int(lib.sealbart_get_stat(eng._h, b"last_used_graph"))
    launches = eng.last_launch_count() * args.steps
    if world > 1:
        t = torch.tensor([ms], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); ms = float(t.item())
    clocks = sampler.stop() if rank == 0 else None
    value = Qtot * args.steps / (ms * 1e-3)
    # the records of the timed run, on rank 0: all ranks' blocks in query order
    full = merge_gathered(gathered, layout) if (world > 1 and rank == 0) else (rec.host() if world == 1 else None)
    errs = rec.host()["errors"] if Q else np.zeros(4, dtype=np.int32)
    assert not errs.any(), f"generate raised error flags {errs.tolist()} (include/sealdec.h)"
    if args.dump_outputs and full is not None:
        dump_outputs(full, args.dump_outputs)

    # ---- end to end through the public host-array API: H2D of the inputs, decode, the gather, D2H of the records ----
    e2e_steps = max(1, min(args.steps, 3))
    if world > 1:
        e2e_call = lambda: sharded_generate_records(eng, index, ids_all if strong else ids_np, mask_all if strong else mask_np, **kw)
        api = "seal_b200.beam_search.sharded_generate_records (host arrays -> sealdec_generate_dx -> one NCCL gather -> host records on rank 0)"
    else:
        e2e_call = lambda: generate_records(eng, index, ids_np, mask_np, MIN_LEN, MAX_LEN, LP, BEAM, forced_bos_token_id=None)
        api = "sealdec_generate (host buffers)"
    for _ in range(min(args.warmup, 3)):
        e2e_call()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_call()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); e2e_s = float(t.item())
    W32 = (50265 + 31) // 32
    rec_bytes = Qtot * H * (4 + 4 + 4 * MAX_LEN + 1 + 16)
    e2e = {"value": Qtot * e2e_steps / e2e_s, "unit": "queries/s",
           "h2d_bytes_per_step": int(Qtot * ids_all.shape[1] * 16 + W32 * 4 * (1 if world == 1 else 0)),
           "d2h_bytes_per_step": int(rec_bytes + 16), "api": api,
           "gathered_bytes_per_step": int(layout.nbytes * (world - 1)) if world > 1 else 0}

    weak = None
    if world > 1 and strong and args.weak_too:               # second curve: every GPU its own 1 000 queries (round 1's figure)
        _, ids_w, mask_w = build_inputs(args.queries, seed=4321 + rank)
        lw = RecordLayout(args.queries, H, MAX_LEN); rw = DeviceRecords(lw, dev)
        idw = torch.from_numpy(ids_w).to(dev); mkw = torch.from_numpy(mask_w).to(dev); stw = int(mask_w.sum())

        def step_w():
            with torch.cuda.stream(stream):
                generate_records_device(eng, index, idw, mkw, out=rw, src_tokens=stw, stream=stream, **kw)
                gather_buffers(rw.buf, dst=0)
        for _ in range(2):
            step_w()
        barrier()
        a0 = torch.cuda.Event(enable_timing=True); a1 = torch.cuda.Event(enable_timing=True)
        a0.record(stream)
        for _ in range(e2e_steps):
            step_w()
        a1.record(stream); barrier()
        t = torch.tensor([a0.elapsed_time(a1)], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX)
        weak = {"value": world * args.queries * e2e_steps / (float(t.item()) * 1e-3), "unit": "queries/s",
                "ms_per_step": float(t.item()) / e2e_steps, "queries_per_gpu": args.queries}

    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    hbm, tf_burst, tf_sus, which = peaks()
    # ---- roofline of the dominant kernel (the decoder/encoder/lm_head GEMM), measured live: one extra
    # pass (eager launches, no CUDA graph) with every GEMM launch bracketed by CUDA events on its stream --------
    eng.profile_gemm(True)
    step_device(gather=False); torch.cuda.synchronize()
    prof = eng.profile_gemm(False)
    phases = eng.last_phase_us()
    gemm_s = prof["total_us"] * 1e-6
    passes = 3
    ach = prof["flops"] / gemm_s / 1e12
    roof = {"bound": "tensor", "kernel": {2: "umma_gemm_tf32x3_persistent_kernel", 3: "umma_gemm_f16x3_persistent_kernel",
                                          5: "umma_gemm_f16x3_2cta_kernel"}[args.gemm_mode],
            "achieved": ach, "peak": tf_sus, "unit": "TFLOP/s", "frac": ach / tf_sus,
            "traffic": TRAFFIC_PER_LAUNCH.get(args.gemm_mode),
            "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({which}; the kernel runs inside a long step)",
            "avg_launch_us": prof["total_us"] / max(prof["launches"], 1), "launches_per_step": prof["launches"],
            "share_of_step": gemm_s / (phases["total"] * 1e-6),
            "tensor_pipe_TFLOPs": ach * passes, "tensor_pipe_frac": ach * passes / tf_sus,
            "note": "achieved = algorithmic 2MNK flops (fp32-equivalent) of all GEMM launches of one step / their summed "
                    "CUDA-event durations; the kernel issues 3 half-precision tensor-core passes per product "
                    "(error-compensated split, DESIGN.md section 4), so the tensor pipe itself runs at tensor_pipe_TFLOPs; "
                    "traffic = dram bytes read+written per launch of the fc1-shaped GEMM (ncu, profiles/)"}
    rank_kernel = rank_kernel_report(index, full, dev, hbm, phases, args)
    cpu = cpu_baseline_and_parity(args, full, q_lo) if world == 1 else None
    out = {"metric": METRIC, "value": value, "unit": "queries/s", "n_gpus": world, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": args.scaling,
           "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": "configs[1]/[3]: synthetic 10M-token corpus (100k docs x 100 tok, seed 1234), "
                                  + (f"{args.queries} queries (seed 4321) sharded over {world} GPU(s)" if strong else f"{args.queries} queries/GPU (seed 4321+rank)")
                                  + f", beam {BEAM}, min=max_length {MAX_LEN}, BART-large random init seed 0, fp32"
                                  + (", final_logits_bias = log unigram frequency" if args.regime == "freq" else ""),
                      "queries_total": Qtot, "queries_this_rank": Q, "beam": BEAM, "decode_steps": MAX_LEN - 1, "regime": args.regime,
                      "parallelism": f"query-sharded x{world}, index+weights replicated, one NCCL gather of the record buffers "
                                     f"({layout.nbytes} B per rank)",
                      "l2": "per-step working set (KV cache + logits > 10 GB at 1000 queries) exceeds L2; no explicit flush",
                      "cuda_graph": bool(used_graph),
                      "exact_work_elision": "results identical to the full computation (parity tests): the first decode step runs on one "
                                            "row per query (its beams are identical rows) [SEALB200_COMPACT_FIRST=%s]; the step whose scores "
                                            "ForcedEOS overwrites entirely (the 9th) has no model forward [SEALB200_SKIP_DEAD_STEP=%s]; "
                                            "all 9 select/record steps run; the encoder runs on the real (unpadded) source tokens [SEALB200_PACK_ENCODER=%s]"
                                            % (os.environ.get("SEALB200_COMPACT_FIRST", "1"), os.environ.get("SEALB200_SKIP_DEAD_STEP", "1"),
                                               os.environ.get("SEALB200_PACK_ENCODER", "1"))},
           "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
           "roofline": roof, "rank_kernel": rank_kernel, "phases_us_last_step": phases,
           "cpu_baseline": cpu["cpu_baseline"] if cpu else None,
           "parity_check": cpu["parity_check"] if cpu else None}
    if weak:
        out["weak"] = weak
    print(json.dumps(out))


DUMP_LIMIT = 64 << 20


def dump_outputs(rec, out_dir, limit=DUMP_LIMIT):
    """Writes the hypothesis records of the last timed step (what the caller of the timed path receives) as
    out_dir/<name>.npy: SA bounds as float64, everything else as float32 (token ids, lengths and flags are exact there).
    A slot without a hypothesis has score -inf in the records; the dump marks such slots 0 in present.npy and stores
    score 0 there, so every written value is finite.
    If the records exceed `limit` bytes, a fixed seeded sample of queries is written, their indices in query_index.npy."""
    rec = dict(rec)
    present = ~np.isneginf(rec["scores"])                      # a NaN stays in the dump: it would be a fault
    rec["present"] = present.astype(np.uint8)
    rec["scores"] = np.where(present, rec["scores"], np.float32(0))
    per_dtype = {k: (np.float64 if v.dtype in (np.uint64, np.int64) else np.float32) for k, v in rec.items()}
    Q = rec["scores"].shape[0]
    row_bytes = sum(np.dtype(per_dtype[k]).itemsize * rec[k][0].size for k in rec if k != "errors") if Q else 0
    rows = None
    if Q and Q * row_bytes > limit - 4096:                     # 4 KB left for the .npy headers
        n = (limit - 4096) // (row_bytes + 8)
        rows = np.sort(np.random.default_rng(0).choice(Q, size=n, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for k, v in rec.items():
        if rows is not None and k != "errors":
            v = v[rows]
        np.save(os.path.join(out_dir, k + ".npy"), v.astype(per_dtype[k]))
    if rows is not None:
        np.save(os.path.join(out_dir, "query_index.npy"), rows.astype(np.float64))


def rank_kernel_report(index, full, dev, hbm, phases, args):
    """The metric's rank kernel: batched LF-mapping (backward_search_step).  (1) on this 10 M-token index with the
    decode's own (symbol, lo, hi) trace -- the 27 MB index is L2-resident, so that rate is L2-, not HBM-bound; (2) on
    a beyond-L2 index (2e8 random tokens, 610 MB on the device) with random triples: the HBM figure."""
    import torch
    from seal_b200.index import FMIndex
    from seal_b200.cpp_modules.fm_index import FMIndex as RawFM

    def time_lf(idx, sym, lo_t, hi_t, reps=10):
        for _ in range(3):
            idx.lf_step_tensors(sym, lo_t, hi_t)
        ea = torch.cuda.Event(enable_timing=True); eb = torch.cuda.Event(enable_timing=True)
        ea.record()
        for _ in range(reps):
            idx.lf_step_tensors(sym, lo_t, hi_t)
        eb.record(); torch.cuda.synchronize()
        return ea.elapsed_time(eb) * 1e-3 / reps

    sym_np, lo_np, hi_np = decode_trace(full)
    n_trace = len(sym_np)
    reps = max(1, (1 << 22) // max(n_trace, 1))
    sym = torch.from_numpy(np.tile(sym_np, reps)).to(dev); lo_t = torch.from_numpy(np.tile(lo_np, reps)).to(dev)
    hi_t = torch.from_numpy(np.tile(hi_np, reps)).to(dev)
    N1 = int(sym.numel())
    s1 = time_lf(index, sym, lo_t, hi_t)
    out = {"kernel": "lf_step_kernel", "bytes_per_lf_step": 48 * 16,
           "decode_trace_10M": {"triples": N1, "distinct_trace_triples": n_trace, "us": s1 * 1e6, "steps_per_s": N1 / s1,
                                "algorithmic_GBps": N1 * 768 / s1 / 1e9, "bound": "L2 (27 MB index resident in the 126 MB L2; "
                                "not an HBM fraction)"},
           "note": "48*L B per LF step (SURVEY 8d); select+expand phase of the step: %.1f ms of %.1f ms"
                   % (phases["select_expand"] / 1e3, phases["total"] / 1e3)}
    if not args.no_big_index:
        try:
            n_big = args.big_index_tokens
            rng = np.random.Generator(np.random.PCG64(99))
            text = rng.integers(14, 50275, size=n_big, dtype=np.int64).astype(np.uint64)
            big = FMIndex(); RawFM.initialize(big, text); del text
            big.to_device(dev.index)
            g = torch.Generator(device=dev); g.manual_seed(1)
            Nlf = 1 << 22
            sy = torch.randint(14, 50275, (Nlf,), device=dev, generator=g)
            lo2 = torch.randint(0, big.size() // 2, (Nlf,), device=dev, generator=g)
            hi2 = lo2 + torch.randint(1, big.size() // 2, (Nlf,), device=dev, generator=g)
            s2 = time_lf(big, sy, lo2, hi2)
            gbs = Nlf * 768 / s2 / 1e9
            # for scale: the rate of UNIFORM random 32-byte sector reads over a buffer of the index's size (no locality at all,
            # sealfm_debug_sector_probe) -- ~0.2 of the copy peak on this part; an LF step reads 2 sectors per tree level and
            # beats that rate where its two rank chains and the top tree levels have locality
            import ctypes as C
            from seal_b200._lib import lib, check
            us = C.c_double(0)
            n_loads = Nlf * 32
            check(lib.sealfm_debug_sector_probe(int(big.device_bytes()), n_loads, 5, C.byref(us)))
            ceil_sectors = n_loads / (us.value * 1e-6)
            lf_sectors = Nlf * 32 / s2
            out["hbm_index"] = {"index_tokens": n_big, "device_bytes": int(big.device_bytes()), "triples": Nlf, "us": s2 * 1e6,
                                "algorithmic_GBps": gbs, "hbm_peak_GBps": hbm, "frac_of_hbm_peak": gbs / hbm,
                                "sector_GBps": lf_sectors * 32 / 1e9, "uniform_random_sector_GBps": ceil_sectors * 32 / 1e9,
                                "ratio_to_uniform_random_sector_rate": lf_sectors / ceil_sectors,
                                "bound": "HBM, isolated 32-byte sectors (index 5x the L2): uniform random sector reads reach only "
                                         "uniform_random_sector_GBps on this part; the LF kernel's sectors have some locality"}
            del big
        except Exception as ex:  # pragma: no cover
            out["hbm_index"] = {"error": repr(ex)}
    return out


# ------------------------------------------------------------------------------------------------
def reference_setup(n_queries, seed=4321, regime="random"):
    """The reference algorithm on host cores: CPU restatement of seal/beam_search.py (oracle/
    decode_oracle.py) on transformers' eager fp32 BART + the reference FM-index (oracle/_ref, the
    unmodified seal/cpp_modules/fm_index.cpp on sdsl-lite; the C port if _ref was not shipped).
    The queries are the SAME batch the GPU arm decodes (seed 4321, generated as a batch of `n_queries`)."""
    import torch
    from oracle.fm_oracle import OracleIndex, RefFM, PortFM, ref_available
    from seal_b200.synthetic import corpus_symbols
    docs, ids, mask = build_inputs(n_queries, seed)
    fm = RefFM(corpus_symbols(docs)) if ref_available() else PortFM(corpus_symbols(docs))
    idx = OracleIndex(_raw=fm)
    idx.beginnings = list(range(0, docs.size + 1, docs.shape[1]))
    idx.occurring_distinct, idx.occurring_counts = idx.get_distinct_count(0, len(idx))
    model = make_model(unigram_log_freq(docs, 50265) if regime == "freq" else None)
    return idx, model, torch.from_numpy(ids), torch.from_numpy(mask), ("reference" if ref_available() else "port")


def pick_threads(idx, model, ids, mask):
    """torchrun exports OMP_NUM_THREADS=1 and the box's default is one thread per hardware thread; the decoder GEMMs of
    a KV-cached step are 120-row matrices, which scale badly past a few dozen threads.  Time a 2-query decode at a few
    thread counts and keep the fastest: the baseline gets the best configuration of the box's cores."""
    import torch
    n_cpu = os.cpu_count() or 1
    best, best_t = None, None
    for th in sorted({t for t in (8, 16, 32, 64, n_cpu) if t <= n_cpu}):
        torch.set_num_threads(th)
        t0 = time.perf_counter()
        reference_step(idx, model, ids, mask, 0, 2)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = th, dt
    torch.set_num_threads(best)
    return best


def reference_step(idx, model, ids, mask, lo, n):
    from oracle.decode_oracle import fm_index_generate_oracle
    return fm_index_generate_oracle(model, idx, ids[lo:lo + n], mask[lo:lo + n], min_length=MIN_LEN, max_length=MAX_LEN,
                                    length_penalty=LP, num_beams=BEAM, use_cache=True)


def cpu_baseline_and_parity(args, full, q_lo):
    """Rank 0, N = 1: the reference algorithm decodes the first n queries of the SAME batch on the host cores --
    timed (cpu_baseline) and compared with the GPU records of the timed run (parity_check): identical hypothesis
    token sets after the caller's get_count > 0 filter (SURVEY.md H4), |dscore| <= 1e-4, SA ranges == get_range."""
    if args.no_cpu_baseline:
        return None
    try:
        import torch
        n = args.ref_queries
        idx, model, ids, mask, kind = reference_setup(args.queries, regime=args.regime)
        pick_threads(idx, model, ids, mask)
        t0 = time.perf_counter()
        exp = reference_step(idx, model, ids, mask, 0, n)
        dt = time.perf_counter() - t0
        base = {"value": n / dt, "unit": "queries/s", "cores": torch.get_num_threads(), "kind": kind,
                "sample": f"first {n} of the 1000 queries, full 9-step constrained decode (HF BART eager fp32 with KV cache on "
                          f"the host cores + {'sdsl-lite FM-index (oracle/_ref)' if kind == 'reference' else 'C port of the FM-index'}), {dt:.1f} s"}
        worst, n_hyp, n_rng, bad = 0.0, 0, 0, []
        for q in range(n):
            keep = lambda t: idx.get_count(list(t[1:])) > 0
            fb = sorted((tuple(t), s) for s, t, _ in exp[q] if keep(t))
            fa = []
            for h in range(full["scores"].shape[1]):
                s = float(full["scores"][q - q_lo, h])
                if s > float("-inf"):
                    t = tuple(int(x) for x in full["tokens"][q - q_lo, h, :full["lens"][q - q_lo, h]])
                    if keep(t):
                        fa.append((t, s))
                        if full["valid"][q - q_lo, h] == 1:
                            n_rng += 1
                            if (int(full["lo"][q - q_lo, h]), int(full["hi"][q - q_lo, h])) != idx.get_range(list(t[1:])):
                                bad.append(("range", q, t))
            fa.sort()
            if [x[0] for x in fa] != [x[0] for x in fb]:
                bad.append(("tokens", q, len(fa), len(fb)))
                continue
            for (ta, sa), (tb, sb) in zip(fa, fb):
                worst = max(worst, abs(sa - sb)); n_hyp += 1
        # SURVEY 8(d)-2: the reference algorithm with eager fp32 BART ON THIS GPU (what README.md:76-83 recommends) + sdsl on
        # the host cores, at the reference's batch size of 20 -- one warm-up batch, one timed batch
        gpu_eager = None
        if not args.no_gpu_eager_baseline:
            try:
                mg = model.to("cuda")
                from oracle.decode_oracle import fm_index_generate_oracle
                kwb = dict(min_length=MIN_LEN, max_length=MAX_LEN, length_penalty=LP, num_beams=BEAM, use_cache=True)
                fm_index_generate_oracle(mg, idx, ids[20:40].cuda(), mask[20:40].cuda(), **kwb)
                torch.cuda.synchronize(); t1 = time.perf_counter()
                fm_index_generate_oracle(mg, idx, ids[:20].cuda(), mask[:20].cuda(), **kwb)
                torch.cuda.synchronize(); dtg = time.perf_counter() - t1
                gpu_eager = {"value": 20 / dtg, "unit": "queries/s", "batch": 20, "s_per_batch": dtg,
                             "what": "reference algorithm (oracle decode loop) with eager fp32 HF BART + KV cache on this B200, "
                                     "sdsl-lite FM-index on the host cores"}
                del mg
            except Exception as ex:  # pragma: no cover
                gpu_eager = {"error": repr(ex)}
        base["gpu_eager_bart_batch20"] = gpu_eager
        ok = not bad and worst <= TOL
        par = {"queries": n, "hypotheses_compared": n_hyp, "sa_ranges_compared": n_rng, "worst_dscore": worst, "tol": TOL,
               "ok": bool(ok), "mismatches": [str(b) for b in bad[:4]],
               "rule": "GPU records of the timed 1000-query batch vs the reference algorithm (oracle) on the same first queries: "
                       "identical token sets after the get_count>0 filter, |dscore| <= tol, [lo,hi) == oracle get_range"}
        return {"cpu_baseline": base, "parity_check": par}
    except Exception as ex:  # pragma: no cover
        return {"cpu_baseline": {"value": None, "unit": "queries/s", "error": repr(ex)}, "parity_check": {"ok": False, "error": repr(ex)}}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    n = args.ref_queries
    idx, model, ids, mask, kind = reference_setup(args.queries, regime=args.regime)
    pick_threads(idx, model, ids, mask)
    k = 0
    for _ in range(args.warmup):
        reference_step(idx, model, ids, mask, k % (args.queries - n + 1), n); k += n
    t0 = time.perf_counter()
    for _ in range(args.steps):
        reference_step(idx, model, ids, mask, k % (args.queries - n + 1), n); k += n
    dt = time.perf_counter() - t0
    v = n * args.steps / dt
    base = {"value": v, "unit": "queries/s", "cores": torch.get_num_threads(), "kind": kind,
            "sample": f"{n} queries per step (bounded sample of the 1000-query batch), 9 decode steps, beam {BEAM}, KV-cached eager fp32 BART"}
    print(json.dumps({"impl": "reference", "metric": METRIC, "value": v, "unit": "queries/s",
                      "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": args.steps, "warmup": args.warmup,
                      "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
                      "dtype": "f32", "data": "synthetic",
                      "config": {"workload": "configs[1] sample: synthetic 10M-token corpus, beam 15, min=max_length 10, "
                                             "BART-large random init seed 0, fp32, host cores only", "queries_per_step": n,
                                 "regime": args.regime},
                      "cpu_baseline": base,
                      "e2e": {"value": v, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--queries", type=int, default=1000)
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="strong: --queries in total, sharded over the GPUs (configs[3]); weak: --queries per GPU")
    ap.add_argument("--weak-too", type=int, default=1, help="at N>1 also time the weak-scaling variant (reported under 'weak')")
    ap.add_argument("--regime", default="random", choices=["random", "freq"],
                    help="freq: final_logits_bias = log unigram frequency, beams follow frequent continuations (SURVEY 8d)")
    ap.add_argument("--ref-queries", type=int, default=8, help="queries per step of the CPU reference sample / parity check")
    ap.add_argument("--gemm-mode", type=int, default=int(os.environ.get("SEALB200_GEMM", "5")))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-big-index", action="store_true")
    ap.add_argument("--no-gpu-eager-baseline", action="store_true")
    ap.add_argument("--big-index-tokens", type=int, default=200_000_000)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the hypothesis records of the last timed step as DIR/<name>.npy (at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
