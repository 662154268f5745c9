#!/usr/bin/env python
"""bench.py — queries/sec of the dense-retrieval hot path (embed -> brute-force top-k -> cross-encoder
rerank) on a 10M x 384 synthetic corpus, BASELINE.json's metric.

One "step" = one batch of Q queries through the whole path:
  1. embed      Q query token sequences  -> MiniLM-L6-shaped encoder -> [Q, 384] unit vectors
  2. top-k      exact top-R (R=100) of every query over this rank's shard of the 10M x 384 fp32 corpus
  3. merge      (N>1) ONE all-gather of the per-shard [Q, R] candidates over NCCL + on-device merge
  4. rerank     (query, doc) token pairs of the R candidates -> ms-marco-MiniLM-L-6-shaped cross-encoder
                -> logits; pairs are split across ranks for N>1 and all-gathered
  5. select     stable sort by logit, keep top-10 (ScoredCrossEncoderReranker semantics)

`value`   : queries/sec with the step's inputs (query tokens, corpus, doc token table) resident in HBM.
`e2e`     : same step through the host-buffer C-ABI entry points (rmu_encoder_embed_host,
            rmu_index_search_host, rmu_encoder_classify_host): token ids / vectors / logits cross PCIe
            inside the timed region.  Host string tokenisation (HF `tokenizers`, unchanged from the
            reference) is outside both numbers and outside the CPU arm.
`--impl reference`: the reference's own CPU path (oracle restatement: torch-CPU fp32 BERT, fp32
            brute-force top-k, fp32 cross-encoder) on the host cores, bounded sample per step.

Weights are seeded random-init of the named architectures and the corpus is seeded synthetic
(no network in the image); strong scaling: the corpus is 10M rows in total for every N.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from dataclasses import asdict

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

TOPN = 10
Q_TOK = 16                                      # query tokens (without specials)
D_TOK = 128                                     # doc tokens
PAIR_LEN = Q_TOK + D_TOK + 3                    # [CLS] q [SEP] d [SEP] = 147
DOC_TABLE = 65536                               # distinct synthetic documents' token rows
CHUNK = 250_000                                 # corpus generation granularity (seed per global chunk)
CE_CHUNK = int(os.environ.get("BENCH_CE_CHUNK", 800))      # rerank pairs per encoder call (117.6k tokens, ~2 GB of activations)
PARITY_ROWS = 1_000_000                         # corpus block the in-run CPU-oracle parity check searches
DUMP_BYTES = 64 << 20                           # cap on what --dump-outputs writes

# BASELINE.json `configs` (SURVEY.md §8a: C2..C5) + the headline the metric is quoted on.  Every config runs on any
# number of GPUs: the corpus is row-sharded over the ranks (strong scaling), rerank pairs are split over the ranks.
CONFIGS = {
    #            corpus rows, dim, queries, candidates, rerank, embedding model (shape preset)
    "headline": dict(n=10_000_000, dim=384, q=64, r=100, rerank=True, emb="all-MiniLM-L6-v2"),
    "c2": dict(n=1_000_000, dim=384, q=64, r=10, rerank=False, emb="all-MiniLM-L6-v2"),
    "c3": dict(n=10_000_000, dim=384, q=256, r=10, rerank=False, emb="all-MiniLM-L6-v2"),
    "c4": dict(n=1_000_000, dim=384, q=64, r=100, rerank=True, emb="all-MiniLM-L6-v2"),
    "c5": dict(n=5_000_000, dim=768, q=64, r=50, rerank=True, emb="bge-base-en-v1.5"),
}
CE_MODEL = "ms-marco-MiniLM-L-6-v2"


class Workload:
    def __init__(self, name: str):
        c = dict(CONFIGS[name])
        self.name = name
        self.n = int(os.environ.get("BENCH_N", c["n"]))
        self.dim = c["dim"]
        self.q = int(os.environ.get("BENCH_Q", c["q"]))
        self.r = int(os.environ.get("BENCH_R", c["r"]))
        self.rerank = c["rerank"]
        self.emb = c["emb"]
        self.metric = os.environ.get("BENCH_METRIC", "cosine")
        self.n -= self.n % CHUNK

    def describe(self, q_len: int) -> str:
        tail = (f" -> cross-encoder rerank of {self.r} pairs x {PAIR_LEN} tokens -> top-{TOPN}" if self.rerank else "")
        return (f"[{self.name}] {self.n}x{self.dim} fp32 corpus ({self.metric}), {self.emb}-shaped encoder, batch {self.q} "
                f"queries x {q_len} tokens, top-{self.r}" + tail)

    @property
    def metric_name(self) -> str:
        stages = "embed+top-k+rerank" if self.rerank else "embed+top-k"
        return f"queries/sec ({stages}) on {self.n // 1_000_000}M x {self.dim} corpus"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops", 1590.0), d.get("bf16_tflops_sustained", 1400.0), "measured"
    return 6650.0, 1590.0, 1400.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def wait_rows(self, n: int, timeout: float) -> None:
        """nvidia-smi takes a good part of a second to print its first row: wait until it is really sampling"""
        t0 = time.perf_counter()
        while self.proc is not None and len(self.rows) < n and time.perf_counter() - t0 < timeout:
            time.sleep(0.01)

    def mark(self) -> None:
        self.first = len(self.rows)                     # rows from here on belong to the timed region

    def stop(self):
        rows = self.rows[getattr(self, "first", 0):]
        if self.proc is not None:
            self.proc.terminate()
        sm = [float(r[1]) for r in rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in rows:
            if len(r) >= 8:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------- synthetic data
def corpus_chunk(torch, dev, c: int, dim: int):
    g = torch.Generator(device=dev).manual_seed(1000 + c)
    x = torch.randn(CHUNK, dim, generator=g, device=dev, dtype=torch.float32)
    return torch.nn.functional.normalize(x, dim=1)


def host_inputs(vocab_size: int, nq: int):
    rng = np.random.default_rng(4321)
    q_tok = rng.integers(104, vocab_size, (nq, Q_TOK)).astype(np.int32)
    doc_tab = np.random.default_rng(7).integers(104, vocab_size, (DOC_TABLE, D_TOK)).astype(np.int32)
    return q_tok, doc_tab


def query_batch(q_tok: np.ndarray):
    """[CLS] q [SEP] ragged batch (all the same length here) -> ids, type_ids, cu_seqlens (int32)."""
    n = q_tok.shape[0]
    ids = np.concatenate([np.full((n, 1), 101, np.int32), q_tok, np.full((n, 1), 102, np.int32)], 1)
    cu = (np.arange(n + 1) * ids.shape[1]).astype(np.int32)
    return ids.reshape(-1), np.zeros(ids.size, np.int32), cu, ids.shape[1]


PAIR_TYPES = np.concatenate([np.zeros(Q_TOK + 2, np.int32), np.ones(D_TOK + 1, np.int32)])


def models(W):
    from ragmeup_b200.weights import PRESETS, BertConfig, synthetic_bert_weights
    ecfg = BertConfig(**asdict(PRESETS[W.emb][0]))
    ccfg = BertConfig(**asdict(PRESETS[CE_MODEL][0]))
    ew = synthetic_bert_weights(ecfg, seed=0)
    cw = synthetic_bert_weights(ccfg, seed=1, with_head=True, scale=4.0)
    return ecfg, ccfg, ew, cw, PRESETS[W.emb][1]


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Write the row-aligned [Q, k] result arrays as out_dir/<name>.npy.  Above DUMP_BYTES a fixed seeded sample
    of rows is written, the same rows for the same arguments, so that two builds can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    n = len(next(iter(arrays.values())))
    row_bytes = sum(a[0].nbytes for a in arrays.values())
    rows = np.arange(n)
    if n * row_bytes > DUMP_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(n, DUMP_BYTES // row_bytes, replace=False))
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a[rows])


def assemble_pairs_np(q_tok: np.ndarray, doc_tab: np.ndarray, ids: np.ndarray):
    """[Q, R] candidate ids -> [Q * R, PAIR_LEN] token rows `[CLS] q [SEP] d [SEP]` (synthetic document table)."""
    nq, r = ids.shape
    docs = doc_tab[ids % DOC_TABLE]
    pairs = np.concatenate([np.full((nq, r, 1), 101, np.int32), np.broadcast_to(q_tok[:, None, :], (nq, r, Q_TOK)),
                            np.full((nq, r, 1), 102, np.int32), docs, np.full((nq, r, 1), 102, np.int32)], 2)
    return pairs.reshape(nq * r, PAIR_LEN)


# ---------------------------------------------------------------------------------------- GPU arm
def run_gpu(args):
    import torch
    import torch.distributed as dist
    from ragmeup_b200 import _lib
    from ragmeup_b200.encoder import BertEncoder
    from ragmeup_b200.index import FlatIndex
    from ragmeup_b200.sharded import ShardedFlatIndex

    W = Workload(args.config)
    Q, R, DIM = W.q, W.r, W.dim
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    hbm_peak, tf_burst, tf_sust, peak_src = peaks()

    ecfg, ccfg, ew, cw, pool = models(W)
    emb = BertEncoder(ecfg, ew, with_head=False, device=local)
    ce = BertEncoder(ccfg, cw, with_head=True, device=local) if W.rerank else None

    # corpus shard: global chunks [c0, c1)
    nchunks = W.n // CHUNK
    c0, c1 = rank * nchunks // world, (rank + 1) * nchunks // world
    index = FlatIndex(DIM, W.metric, device=local)
    index.reserve((c1 - c0) * CHUNK)
    for c in range(c0, c1):
        index.add(corpus_chunk(torch, dev, c, DIM))
    sh = ShardedFlatIndex(index)
    sh.sync_offsets()
    torch.cuda.synchronize()

    q_tok_h, doc_tab_h = host_inputs(ecfg.vocab_size, Q)
    q_ids_h, q_typ_h, q_cu_h, q_len = query_batch(q_tok_h)
    q_ids = torch.from_numpy(q_ids_h).to(dev)
    q_typ = torch.from_numpy(q_typ_h).to(dev)
    q_cu = torch.from_numpy(q_cu_h).to(dev)
    q_tok = torch.from_numpy(q_tok_h).to(dev)
    doc_tab = torch.from_numpy(doc_tab_h).to(dev)
    npairs = Q * R
    p0, p1 = rank * npairs // world, (rank + 1) * npairs // world
    pair_cu = (torch.arange(p1 - p0 + 1, device=dev, dtype=torch.int32) * PAIR_LEN)
    pair_typ = torch.from_numpy(PAIR_TYPES).to(dev).repeat(p1 - p0)
    # pair rows are assembled in place: the constant columns ([CLS], query tokens, [SEP]s) are written once,
    # a step only gathers the document tokens of its candidates into the middle of each row
    pair_buf = torch.empty((Q, R, PAIR_LEN), dtype=torch.int32, device=dev)
    pair_buf[:, :, 0] = 101
    pair_buf[:, :, 1:1 + Q_TOK] = q_tok[:, None, :]
    pair_buf[:, :, 1 + Q_TOK] = 102
    pair_buf[:, :, PAIR_LEN - 1] = 102
    pair_docs = pair_buf[:, :, 2 + Q_TOK:PAIR_LEN - 1]
    pair_rows = pair_buf.view(npairs, PAIR_LEN)
    all_logits = torch.empty(npairs, dtype=torch.float32, device=dev)      # one preallocated gather target
    even_split = npairs % world == 0

    def rerank_device(ids):
        pair_docs.copy_(doc_tab[(ids % DOC_TABLE)])                      # [Q, R, D_TOK]
        mine = pair_rows[p0:p1]
        my_logits = all_logits[p0:p1] if even_split or world == 1 else torch.empty(p1 - p0, dtype=torch.float32, device=dev)
        for s_ in range(0, p1 - p0, CE_CHUNK):                             # bounded activation workspace per call
            n_ = min(CE_CHUNK, p1 - p0 - s_)
            my_logits[s_:s_ + n_] = ce.classify_tokens(mine[s_:s_ + n_].reshape(-1), pair_typ[: n_ * PAIR_LEN], pair_cu[: n_ + 1], PAIR_LEN)[:, 0]
        if world > 1:
            if even_split:
                dist.all_gather_into_tensor(all_logits, my_logits)
            else:
                parts = [torch.empty(((r_ + 1) * npairs // world - r_ * npairs // world,), dtype=torch.float32, device=dev) for r_ in range(world)]
                dist.all_gather(parts, my_logits)
                all_logits.copy_(torch.cat(parts))
        lg = all_logits.view(Q, R)
        order = torch.sort(lg, dim=1, descending=True, stable=True).indices[:, :TOPN]
        return torch.gather(ids, 1, order), torch.gather(lg, 1, order)

    state = {}

    def step_device():
        q_emb = emb.embed_tokens(q_ids, q_typ, q_cu, q_len, pool, True)
        scores, ids = sh.search(q_emb, R)                              # [Q, R] global ids, best first
        state["q_emb"] = q_emb
        if not W.rerank:
            return ids, scores
        return rerank_device(ids)

    host_t = {"embed": 0.0, "search": 0.0, "assemble": 0.0, "classify": 0.0, "select": 0.0}
    my_typ_h = np.tile(PAIR_TYPES, p1 - p0)
    my_cu_h = (np.arange(p1 - p0 + 1) * PAIR_LEN).astype(np.int32)

    def step_host():
        """the same step through the HOST-buffer C-ABI entry points: token ids, vectors, candidates and
        logits cross PCIe in both directions inside the call.  For N > 1 every rank searches its shard with
        rmu_index_search_host and the per-shard candidates / logits are exchanged with the same collectives."""
        t = time.perf_counter()
        q_emb = emb.embed_host(q_ids_h, q_typ_h, q_cu_h, pool, True)
        t1 = time.perf_counter(); host_t["embed"] += t1 - t
        sc, ids = index.search_host(q_emb, R, id_offset=sh.offset)
        if world > 1:
            s_d, i_d = torch.from_numpy(sc).to(dev), torch.from_numpy(ids).to(dev)
            s_m, i_m = sh.merge_gathered(s_d, i_d)
            sc, ids = s_m.cpu().numpy(), i_m.cpu().numpy()
        t2 = time.perf_counter(); host_t["search"] += t2 - t1
        if not W.rerank:
            return ids, sc
        flat = np.ascontiguousarray(assemble_pairs_np(q_tok_h, doc_tab_h, ids)[p0:p1].reshape(-1))
        t3 = time.perf_counter(); host_t["assemble"] += t3 - t2
        logits = ce.classify_host(flat, my_typ_h, my_cu_h)[:, 0]
        if world > 1:
            l_d = torch.from_numpy(logits).to(dev)
            parts = [torch.empty(((r_ + 1) * npairs // world - r_ * npairs // world,), dtype=torch.float32, device=dev) for r_ in range(world)]
            dist.all_gather(parts, l_d)
            logits = torch.cat(parts).cpu().numpy()
        t4 = time.perf_counter(); host_t["classify"] += t4 - t3
        order = np.argsort(-logits.reshape(Q, R), axis=1, kind="stable")[:, :TOPN]
        out = np.take_along_axis(ids, order, 1), np.take_along_axis(logits.reshape(Q, R), order, 1)
        host_t["select"] += time.perf_counter() - t4
        return out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- timed region: device-resident step
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        out_ids, out_scores = step_device()
    if rank == 0:
        sampler.wait_rows(1, 3.0)          # nvidia-smi is really sampling before anybody starts the timed region
    barrier()
    launches0 = _lib.launch_count()
    _lib.profile_reset()
    _lib.profile_enable(True)
    # the clock sampler is started during the warm-up (nvidia-smi needs ~1 s before its first row) and only the rows it
    # prints between here and the end of the timed steps are kept; short steps are repeated (untimed region extended
    # AFTER ev1) until at least a few samples fell inside GPU work of the same kind
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if rank == 0:
        sampler.mark()
    ev0.record()
    for _ in range(args.steps):
        out_ids, out_scores = step_device()
    ev1.record()
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"ids": out_ids.cpu().numpy().astype(np.float64), "scores": out_scores.cpu().numpy()})
    ms = torch.tensor([ev0.elapsed_time(ev1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    total_ms = float(ms.item())
    _lib.profile_enable(False)
    prof = _lib.profile_read()
    launches = _lib.launch_count() - launches0
    # short steps: keep the same load running (outside the timed events, the same count on every rank) until the sampler
    # has seen ~0.3 s of it
    extra = min(400, max(0, int(np.ceil(300.0 / max(total_ms / args.steps, 1e-3))) - args.steps))
    for _ in range(extra):
        step_device()
    barrier()
    clocks = sampler.stop() if rank == 0 else None

    # ---------------- e2e through host buffers (every rank runs its part; max over ranks)
    light = os.environ.get("BENCH_LIGHT") == "1"       # launch-list captures under ncu only: no e2e warm-up, no CPU arm
    for _ in range(0 if light else max(1, min(args.warmup, 2))):
        h_ids, h_scores = step_host()
    barrier()
    for k_ in host_t:
        host_t[k_] = 0.0
    t0 = time.perf_counter()
    n_e2e = max(1, min(args.steps, 5))
    for _ in range(n_e2e):
        h_ids, h_scores = step_host()
    torch.cuda.synchronize()
    e2e_t = torch.tensor([(time.perf_counter() - t0) * 1e3 / n_e2e], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_ms = float(e2e_t.item())
    same = bool((h_ids == out_ids.cpu().numpy()).all())
    my_pairs = (p1 - p0) if W.rerank else 0
    h2d = q_ids_h.nbytes * 2 + q_cu_h.nbytes + Q * DIM * 4 + my_pairs * PAIR_LEN * 4 * 2 + (my_cu_h.nbytes if W.rerank else 0)
    d2h = Q * DIM * 4 + Q * R * 12 + my_pairs * 4
    if world > 1:
        h2d += Q * R * 12 + my_pairs * 4
        d2h += Q * R * 12 + (npairs * 4 if W.rerank else 0)
    api = "rmu_encoder_embed_host + rmu_index_search_host" + (" + rmu_encoder_classify_host" if W.rerank else "")
    e2e = {"value": Q / (e2e_ms * 1e-3), "unit": "queries/s", "ms_per_step": e2e_ms, "h2d_bytes_per_step": int(h2d),
           "d2h_bytes_per_step": int(d2h), "bytes_are": "per rank", "ids_equal_device_path": same,
           "host_ms_per_step": {k_: round(v_ * 1e3 / n_e2e, 2) for k_, v_ in host_t.items()}, "api": api}

    if rank != 0:
        if world > 1:
            dist.barrier()                                  # rank 0 finishes the parity check before the group is torn down
            dist.destroy_process_group()
        return

    # ---------------- in-run parity vs the CPU oracle on the SAME corpus block and queries (rank 0's first rows)
    parity, cpu = None, None
    if not light:
        parity, cpu = parity_and_cpu_arm(W, torch, dev, index, emb, ce, pool, state["q_emb"], q_tok_h, doc_tab_h, q_ids_h, q_len,
                                         ecfg, ccfg, ew, cw, time_cpu=(world == 1))

    ms_per_step = total_ms / args.steps
    n_local = (c1 - c0) * CHUNK
    # rooflines: with a rerank stage the dominant kernel of the step is the cross-encoder GEMM (tensor bound);
    # the top-k scan is the HBM-bound kernel BASELINE.json quotes separately (and the dominant one without rerank).
    tok_rerank = (p1 - p0) * PAIR_LEN if W.rerank else 0
    tok_embed = Q * q_len
    per_tok = lambda c_: 2 * c_.layers * (4 * c_.hidden * c_.hidden + 2 * c_.hidden * c_.ffn)
    gemm_flops_step = per_tok(ccfg) * tok_rerank + per_tok(ecfg) * tok_embed
    gemm_ms, gemm_n = prof["gemm"]
    scan_ms, scan_n = prof["scan"]
    fin_ms, fin_n = prof["finalize"]
    traffic = {}
    tpath = os.path.join(ROOT, "profiles", "traffic.json")          # dram bytes per launch from the committed ncu captures
    if os.path.exists(tpath):
        with open(tpath) as f:
            traffic = json.load(f)
    roof_gemm = None
    if gemm_n:
        ach = gemm_flops_step * args.steps / (gemm_ms * 1e-3) / 1e12
        roof_gemm = {"kernel": "gemm_f16x3_kernel + gemm_f16x3_ln_kernel (all encoder projections)", "bound": "tensor", "achieved": ach, "peak": tf_sust, "unit": "TFLOP/s",
                     "frac": ach / tf_sust, "traffic": traffic.get("gemm_dram_bytes_per_launch"),
                     "peak_source": peak_src + " bf16 sustained (timed inside a long step)",
                     "launches": gemm_n, "avg_launch_ms": gemm_ms / gemm_n,
                     "hw_tflops": 3 * ach, "hw_frac": 3 * ach / tf_sust,
                     "algorithmic_flops_per_launch": gemm_flops_step * args.steps / gemm_n,
                     "note": "achieved = algorithmic fp32-equivalent flops; every K step issues 3 fp16 MMAs (hi*hi+lo*hi+hi*lo) "
                             "to hold 1e-3 fp32 parity, so frac <= 1/3; hw_tflops = the fp16 MMA rate actually issued"}
    roof_scan = None
    if scan_n:
        bytes_per_launch = 4.0 * n_local * DIM            # one scan launch reads the corpus shard exactly once
        ach = bytes_per_launch / (scan_ms / scan_n * 1e-3) / 1e9
        ms_per_search = (scan_ms + fin_ms) / args.steps   # scan + selection / exact re-score / certificate
        roof_scan = {"kernel": "scan_rows_kernel", "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s",
                     "frac": ach / hbm_peak, "traffic": traffic.get("scan_dram_bytes_per_launch") if W.name == "headline" and world == 1 else None,
                     "peak_source": peak_src,
                     "launches": scan_n, "avg_launch_ms": scan_ms / scan_n, "bytes_per_launch": bytes_per_launch,
                     "ms_per_search_incl_select": ms_per_search, "launches_per_search": scan_n / args.steps,
                     "gbps_per_search_incl_select": bytes_per_launch * (scan_n / args.steps) / (ms_per_search * 1e-3) / 1e9,
                     "frac_per_search_incl_select": bytes_per_launch * (scan_n / args.steps) / (ms_per_search * 1e-3) / 1e9 / hbm_peak,
                     "k": R, "candidates_rescored": 256 if R > 42 else (128 if R > 21 else 64)}
    kernel_ms = {k: round(v[0] / args.steps, 4) for k, v in prof.items() if v[1]}
    par = f"row-sharded corpus x{world}" + (f", rerank pairs split x{world}" if W.rerank else "") if world > 1 else "single GPU"
    line = {
        "metric": W.metric_name, "value": Q / (ms_per_step * 1e-3),
        "unit": "queries/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32 (fp16 hi/lo split MMA, fp32 accumulate; TF32 coarse scan + exact fp32 re-score)",
        "data": f"synthetic (seeded unit-norm corpus, seeded token ids, random-init {W.emb}-shaped encoder" + (f" and {CE_MODEL}-shaped cross-encoder)" if W.rerank else ")"),
        "config": {"workload": W.describe(q_len), "name": W.name,
                   "corpus_rows_per_gpu": n_local, "parallelism": par,
                   "l2_flush": "not needed: corpus shard (>= 0.19 GB streamed with evict-first) and activations exceed the 126 MB L2"},
        "roofline": roof_gemm if W.rerank else roof_scan, "roofline_topk": roof_scan, "kernel_ms_per_step": kernel_ms,
        "parity": parity, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
    }
    print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def parity_and_cpu_arm(W, torch, dev, index, emb, ce, pool, q_emb_gpu, q_tok_h, doc_tab_h, q_ids_h, q_len, ecfg, ccfg, ew, cw,
                       time_cpu: bool, sample_queries: int = 2):
    """The CPU oracle and the GPU path on the SAME data inside this run: rank 0's first PARITY_ROWS corpus rows are
    copied to the host; (1) the oracle embeds the first queries -> compared with the GPU embeddings; (2) the oracle's
    exact fp32 top-R of ALL Q GPU-embedded queries over the block is compared with a GPU search of the same block
    (ids identical, scores within 1e-3); (3) the oracle reranks the candidates of `sample_queries` queries -> logits
    compared with the GPU cross-encoder's, final top-10 ids compared.  The timed CPU arm (cpu_baseline, N = 1 only)
    is the same oracle code on the same block, one query per search call as the reference does."""
    from oracle import bert_ref, flat_ref
    from ragmeup_b200.index import FlatIndex
    Q, R = W.q, W.r
    rows = min(PARITY_ROWS, len(index))
    x_gpu = index.data()[:rows]
    x_h = x_gpu.cpu()
    sub = FlatIndex(W.dim, W.metric, device=dev.index)
    sub.add(x_gpu)
    g_s, g_i = sub.search(q_emb_gpu, R, want_stats=True)
    flagged = int(sub.last_stats[0])
    g_s, g_i = g_s.cpu().numpy(), g_i.cpu().numpy()
    q_emb_h = q_emb_gpu.cpu().numpy()

    threads = min(usable_cores(), 32)
    torch.set_num_threads(threads)
    st = cpu_state(W, ecfg, ccfg, ew, cw, q_tok_h, doc_tab_h, q_ids_h, q_len, x_h)
    if time_cpu:
        threads = calibrate_threads(st)
    # (1) embeddings
    ne = min(Q, 8)
    with torch.no_grad():
        h = bert_ref.bert_encoder_forward(st["ew"], st["ecfg"], st["q_ids"][:ne], st["q_mask"][:ne])
        e_ref = bert_ref.l2_normalize(bert_ref.pool(h, st["q_mask"][:ne], pool)).numpy()
    embed_err = float(np.abs(e_ref - q_emb_h[:ne]).max())
    # (2) top-R of all Q queries over the block
    o_s, o_i = flat_ref.flat_search_blocked(q_emb_h, x_h.numpy(), R, W.metric)
    ids_same = bool((o_i == g_i).all())
    sets_same = all(set(o_i[r].tolist()) == set(g_i[r].tolist()) for r in range(Q))
    score_err = float(np.abs(o_s - g_s).max())
    # rows ordered differently only where the oracle's own fp32 scores are within 1e-6 of each other (BLAS vs fmaf order)
    order_ok = True
    for r in range(Q):
        diff = np.nonzero(o_i[r] != g_i[r])[0]
        for j in diff:
            pos = np.nonzero(g_i[r] == o_i[r, j])[0]
            if len(pos) == 0 or abs(float(o_s[r, j]) - float(o_s[r, pos[0]])) > 1e-6:
                order_ok = False
    parity = {"corpus_block_rows": rows, "queries": Q, "k": R, "topk_ids_identical": ids_same, "topk_id_sets_identical": sets_same,
              "topk_order_identical_where_oracle_gap_gt_1e-6": order_ok, "topk_max_abs_score_err": score_err,
              "embed_max_abs_err": embed_err, "embed_queries_checked": ne, "queries_sent_to_exact_fallback": flagged,
              "oracle": "oracle/bert_ref.py + oracle/flat_ref.py (torch-CPU / numpy fp32)", "tolerance": 1e-3}
    ok = sets_same and order_ok and score_err <= 1e-3 and embed_err <= 1e-3
    # (3) rerank of the first queries' candidates
    if W.rerank:
        sq = min(sample_queries, Q)
        pairs = assemble_pairs_np(q_tok_h[:sq], doc_tab_h, o_i[:sq])
        l_ref = cpu_rerank(st, torch.from_numpy(pairs.astype(np.int64))).numpy()
        n_p = pairs.shape[0]
        flat = torch.from_numpy(np.ascontiguousarray(pairs.reshape(-1))).to(dev)
        typ = torch.from_numpy(np.tile(PAIR_TYPES, n_p)).to(dev)
        cu = torch.arange(n_p + 1, device=dev, dtype=torch.int32) * PAIR_LEN
        l_gpu = ce.classify_tokens(flat, typ, cu, PAIR_LEN)[:, 0].cpu().numpy()
        logit_err = float(np.abs(l_ref - l_gpu).max())
        o_top = np.argsort(-l_ref.reshape(sq, R), axis=1, kind="stable")[:, :TOPN]
        g_top = np.argsort(-l_gpu.reshape(sq, R), axis=1, kind="stable")[:, :TOPN]
        final_same = bool((np.take_along_axis(o_i[:sq], o_top, 1) == np.take_along_axis(g_i[:sq], g_top, 1)).all())
        parity.update({"rerank_pairs_checked": int(n_p), "rerank_logit_max_abs_err": logit_err, "final_top10_ids_identical": final_same})
        ok = ok and logit_err <= 1e-3 and final_same
    parity["ok"] = bool(ok)
    cpu = None
    if time_cpu:
        cpu_step(W, 1, st)                                  # warm
        total, t = cpu_step(W, sample_queries, st)
        cpu = {"value": sample_queries / total, "unit": "queries/s", "cores": threads, "host_cores_usable": usable_cores(), "kind": "port",
               "sample": cpu_sample_text(W, sample_queries, rows), "seconds": {k: round(v, 4) for k, v in t.items()}}
    return parity, cpu


# ---------------------------------------------------------------------------------------- CPU arm
def cpu_rerank(st, pairs):
    """CrossEncoder.predict restated: batches of 32 in input order, fp32 (oracle/bert_ref.py)."""
    import torch
    from oracle import bert_ref
    typ = torch.from_numpy(PAIR_TYPES.astype(np.int64))[None].expand(pairs.shape[0], PAIR_LEN)
    mask = torch.ones_like(pairs)
    logits = []
    with torch.no_grad():
        for s in range(0, pairs.shape[0], 32):
            hh = bert_ref.bert_encoder_forward(st["cw"], st["ccfg"], pairs[s:s + 32], mask[s:s + 32], typ[s:s + 32])
            logits.append(bert_ref.classifier_head(st["cw"], hh)[:, 0])
    return torch.cat(logits)


def cpu_sample_text(W, sample_queries: int, rows: int) -> str:
    scale = W.n / rows
    tail = f" + rerank of {sample_queries * W.r} pairs x {PAIR_LEN} tokens" if W.rerank else ""
    return (f"{sample_queries} queries: embed + top-{W.r} over a {rows} x {W.dim} block (one query per call, as the reference searches) "
            f"timed and scaled x{scale:g} to {W.n} rows (brute force is linear in rows){tail}, torch-CPU fp32 oracle")


def cpu_step(W, sample_queries: int, st: dict):
    """One bounded sample of the reference CPU path: embed + top-R over the corpus block (scaled to the full
    corpus, brute force is linear in rows) + cross-encoder rerank, all fp32 on the host cores."""
    import torch
    from oracle import bert_ref
    t = {}
    t0 = time.perf_counter()
    with torch.no_grad():
        h = bert_ref.bert_encoder_forward(st["ew"], st["ecfg"], st["q_ids"][:sample_queries], st["q_mask"][:sample_queries])
        q_emb = bert_ref.l2_normalize(bert_ref.pool(h, st["q_mask"][:sample_queries], st["pool"]))
    t["embed"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    ids = []
    for i in range(sample_queries):                       # the reference searches one query per call
        sc = st["xblock"] @ q_emb[i]
        ids.append(torch.topk(sc, W.r).indices)
    t["topk_block"] = time.perf_counter() - t0
    ids = torch.stack(ids)
    t["rerank"] = 0.0
    if W.rerank:
        t0 = time.perf_counter()
        pairs = torch.from_numpy(assemble_pairs_np(st["q_tok"][:sample_queries], st["doc_tab"], ids.numpy()).astype(np.int64))
        cpu_rerank(st, pairs)
        t["rerank"] = time.perf_counter() - t0
    scale = W.n / st["xblock"].shape[0]
    total = t["embed"] + t["topk_block"] * scale + t["rerank"]
    return total, t


def usable_cores() -> int:
    """host cores this process may really use: affinity mask capped by the cgroup CPU quota"""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except Exception:
        pass
    return n


def calibrate_threads(st) -> int:
    """pick the torch thread count that makes the CPU arm fastest (more threads than real cores, or
    than the small GEMMs can use, slows torch down by orders of magnitude)"""
    import torch
    from oracle import bert_ref
    cores = usable_cores()
    cands = sorted({c for c in (4, 8, 16, 32, 64, cores) if c <= cores} | {min(cores, 8)})
    ids = torch.randint(104, 30000, (32, PAIR_LEN))
    mask = torch.ones_like(ids)
    best, best_t = cands[0], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        with torch.no_grad():
            bert_ref.bert_encoder_forward(st["cw"], st["ccfg"], ids[:4], mask[:4])
            t0 = time.perf_counter()
            bert_ref.bert_encoder_forward(st["cw"], st["ccfg"], ids, mask)
            dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best


def cpu_state(W, ecfg, ccfg, ew, cw, q_tok_h, doc_tab_h, q_ids_h, q_len, xblock):
    import torch
    from oracle import bert_ref
    return {"ecfg": bert_ref.BertCfg(**asdict(ecfg)), "ccfg": bert_ref.BertCfg(**asdict(ccfg)),
            "ew": {k: torch.from_numpy(v) for k, v in ew.items()}, "cw": {k: torch.from_numpy(v) for k, v in cw.items()},
            "q_ids": torch.from_numpy(q_ids_h.reshape(W.q, q_len).astype(np.int64)), "q_mask": torch.ones(W.q, q_len, dtype=torch.long),
            "q_tok": q_tok_h, "doc_tab": doc_tab_h, "xblock": xblock, "pool": PRESET_POOL(W)}


def PRESET_POOL(W):
    from ragmeup_b200.weights import PRESETS
    return PRESETS[W.emb][1]


def run_reference(args):
    """--impl reference: the reference's CPU path (oracle port) on the host cores, bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    W = Workload(args.config)
    torch.set_num_threads(min(usable_cores(), 32))
    ecfg, ccfg, ew, cw, _ = models(W)
    q_tok_h, doc_tab_h = host_inputs(ecfg.vocab_size, W.q)
    q_ids_h, _, _, q_len = query_batch(q_tok_h)
    rows = min(PARITY_ROWS, W.n)
    g = torch.Generator().manual_seed(5)
    xblock = torch.nn.functional.normalize(torch.randn(rows, W.dim, generator=g), dim=1)
    st = cpu_state(W, ecfg, ccfg, ew, cw, q_tok_h, doc_tab_h, q_ids_h, q_len, xblock)
    calibrate_threads(st)
    sample = 2
    for _ in range(min(args.warmup, 1)):
        cpu_step(W, 1, st)
    tot = 0.0
    for _ in range(args.steps):
        s, _ = cpu_step(W, sample, st)
        tot += s
    v = sample * args.steps / tot
    cb = {"value": v, "unit": "queries/s", "cores": torch.get_num_threads(), "kind": "port",
          "sample": "each step = " + cpu_sample_text(W, sample, rows)}
    print(json.dumps({
        "impl": "reference", "metric": W.metric_name, "value": v, "unit": "queries/s",
        "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": tot / args.steps * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": {"workload": W.describe(q_len) + " (CPU oracle port of the reference path)", "name": W.name},
        "cpu_baseline": cb, "e2e": {"value": v, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="headline", choices=sorted(CONFIGS),
                    help="BASELINE.json workload: headline (10M x 384, top-100, rerank), c2, c3, c4, c5")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps write the last step's result to DIR: ids.npy (float64 corpus row ids, "
                         "best first) and scores.npy (float32 rerank logits, or top-k scores without rerank), both [Q, k]")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of --impl b200")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
