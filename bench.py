#!/usr/bin/env python
"""Benchmark of the SSE hot path: queries/sec for encode + cosine top-k (BASELINE.json metric), train-step/s secondary.

Default workload = the north_star headline: cross-lingual style dual LSTM encoder (V=32000, We=H=E=256, T=50), an index of
1M target SSE vectors resident in HBM -- BUILT BY THE TARGET ENCODER from synthetic REAL-regime target tokens
(`config.index = "encoded"`) -- query batches of 600 token rows (sse_evaluator.py:104); one "step" = one query batch
through the source encoder and the cosine top-10 of the whole index.  The headline number uses FULL-length query rows
(one leading PAD, T-2 real tokens: every one of the T LSTM steps is executed, pad-prefix skipping off) so that roofline
fractions count the work the reference executes; the REAL regime (queries ~3 tokens, pad-prefix start on) is reported
next to it under "regimes".

    python bench.py --gpus N --steps K --warmup W               (B200 arm)
    python bench.py --impl reference --gpus N --steps K --warmup W
        the reference's own CPU path (numpy restatement of the TF1 encoder + the reference's np.dot / full-argsort
        ranking) on the host cores, bounded sample; inputs are built ONCE, only encode + dot + sort are timed.
    python bench.py --config c1|c2|c3|c4|c5                      the other BASELINE.json configs (see CONFIGS)

N > 1 (torchrun, one rank per GPU): the index is sharded by rows (N/G per rank); a step carries G x 600 queries: each
rank encodes its own 600, an NCCL all-gather distributes the [600,E] encodings, every rank scans its shard for all
G x 600 and writes ONE packed [G*600, 2k] block, an NCCL all-to-all hands every rank the G per-shard blocks of ITS OWN
600 queries, and the merge kernel reduces G*k candidates to k for those 600 rows.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
for p in (REPO, os.path.join(REPO, "sequence-semantic-embedding_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

K_TOP = 10
L2_BYTES = 126e6

# BASELINE.json configs (SURVEY 8d "Concrete configs").  targets = TOTAL index rows at the GPU count the config names.
CONFIGS = {
    "headline": dict(mode="dual-encoder", V=32000, We=256, H=256, E=256, T=50, targets=1_000_000, queries=600,
                     name="cross-lingual retrieval: dual LSTM V=32000 We=H=E=256 T=50, 1M-target index (north_star headline)"),
    "c1": dict(mode="source-encoder-only", V=32000, We=50, H=128, E=64, T=80, targets=20_000, queries=600,
               name="BASELINE config 1 (synthetic variant): source-encoder-only LSTM h=128, We=50 E=64 T=80, 20k-row target table"),
    "c2": dict(mode="dual-encoder", V=32000, We=256, H=256, E=256, T=50, targets=100_000, queries=600,
               name="BASELINE config 2: cross-lingual dual LSTM h=256 T=50, 100k-target index"),
    "c3": dict(mode="dual-cnn", V=32000, We=256, H=0, E=256, T=50, targets=1_000_000, queries=600, cnn_k=(3, 4, 5), cnn_f=(256, 256, 256),
               name="BASELINE config 3: search-ranking dual CNN (3/4/5-gram x 256 filters) We=E=256 T=50, 1M targets"),
    "c4": dict(mode="dual-encoder", V=32000, We=256, H=256, E=256, T=50, targets=100_000, queries=600, train_rows=1536,
               name="BASELINE config 4: training step, 256-d dual LSTM, 512 positives + 1024 negatives = 1536 pair rows"),
    "c5": dict(mode="shared-encoder", V=32000, We=512, H=512, E=512, T=50, targets=5_000_000, queries=600, targets_at_gpus=8,
               name="BASELINE config 5: QnA shared LSTM We=H=E=512 T=50, 5M-target index sharded 8 x 625k"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="headline", choices=sorted(CONFIGS))
    ap.add_argument("--targets", type=int, default=0, help="TOTAL index rows (sharded by rows over the GPUs); 0 = the config's")
    ap.add_argument("--queries", type=int, default=0, help="query rows per step PER GPU (sse_evaluator.py:104 batch); 0 = the config's")
    ap.add_argument("--index", default="encoded", choices=["encoded", "gaussian"],
                    help="encoded: index built by the target encoder from synthetic REAL-regime target tokens (default); "
                         "gaussian: isotropic unit vectors (best case for the sampled-threshold filter)")
    ap.add_argument("--repeats", type=int, default=5, help="the K-step timed region is repeated this many times; the median is reported")
    ap.add_argument("--search", type=int, default=0, help="0 auto (tcgen05), 1 fp32 SIMT, 2 tcgen05")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-pipeline", action="store_true", help="run encode and search of a step back to back on one stream "
                    "(default: 2-stage software pipeline over steps: encoder of batch s+1 overlaps the scan of batch s)")
    ap.add_argument("--search-ctas", type=int, default=-1, help="scan grid cap when pipelining (the remaining SMs run the encoder clusters); "
                    "-1 = auto: 108 (= 148 - 5 clusters x 8 CTAs) up to 4 GPUs, uncapped beyond, 0 = uncapped")
    ap.add_argument("--cluster-rows", type=int, default=-1, choices=[-1, 0, 64, 128],
                    help="batch rows per cluster of the LSTM table kernel in the timed step (0 = the library's choice: 64 when every cluster "
                         "still gets its own SMs; -1 = 128 when the scan is capped for pipelining -- the encoder then fits the SMs the cap "
                         "leaves free -- else 0)")
    ap.add_argument("--search-late", type=int, default=-1, help="with a scan grid cap: extra LATE scan CTAs that start on the SMs the concurrent encoder frees mid-scan "
                                                                   "(-1 = one per SM the cap leaves to the encoder: measured 1.53 -> 1.60 M q/s at the headline shape)")
    ap.add_argument("--search-late-share", type=int, default=40, help="tile share of a late scan CTA, percent of a regular one")
    ap.add_argument("--train-steps", type=int, default=5, help="timed train steps for the secondary train-step/s figure (0 = skip)")
    ap.add_argument("--train-rows", type=int, default=0, help="pair rows per GPU per train step (0 = the config's, default 1024 = 512 pos + 512 neg)")
    ap.add_argument("--no-replicas", action="store_true", help="scan one copy of a small (L2-resident) shard every step instead of rotating replicas")
    ap.add_argument("--no-real-regime", action="store_true", help="skip the REAL-regime (short queries, pad-prefix start) measurement")
    ap.add_argument("--emulate-world", type=int, default=0, help="development aid: run ONE rank's share of a G-GPU step on one GPU "
                    "(collectives replaced by local copies); the line is marked emulated")
    ap.add_argument("--cpu-sample-targets", type=int, default=1_000_000)
    ap.add_argument("--cpu-sample-queries", type=int, default=64)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed paths computed in their last step to DIR/<name>.npy (float32/float64): the top-k scores "
                         "and ids of the headline step and, if train steps ran, a fixed row sample of the parameters they updated")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    a.cfg = dict(CONFIGS[a.config])
    if a.targets:
        a.cfg["targets"] = a.targets
    if a.queries:
        a.cfg["queries"] = a.queries
    return a


def load_peaks():
    try:
        with open(os.path.join(REPO, "MEASURED_PEAKS.json")) as f:
            pk = json.load(f)
        return pk.get("hbm_gbs", 6650.0), pk.get("bf16_tflops", 1590.0), "measured"
    except Exception:
        return 6650.0, 1590.0, "fallback"


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed regions: NVML polled every ~2 ms from a thread (started
    before the first timed region, stopped after the last); falls back to `nvidia-smi -lms` if NVML is unavailable."""

    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, index=0, uuid=None):
        self.index, self.uuid = index, uuid
        self.sm, self.mx, self.reasons = [], 0, set()
        self.stop_flag = False
        self.thread = None
        self.proc = None
        self.source = None

    def _nvml_loop(self, nv, handle):
        while not self.stop_flag:
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(handle, nv.NVML_CLOCK_SM)))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(handle) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(handle)
                for name, bit in self.REASONS:
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            handle = None
            if self.uuid:
                for cand in ("GPU-" + str(self.uuid), str(self.uuid)):
                    try:
                        handle = nv.nvmlDeviceGetHandleByUUID(cand.encode() if isinstance(cand, str) else cand)
                        break
                    except Exception:
                        handle = None
            if handle is None:
                handle = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.mx = float(nv.nvmlDeviceGetMaxClockInfo(handle, nv.NVML_CLOCK_SM))
            self.source = "nvml"
            self.thread = threading.Thread(target=self._nvml_loop, args=(nv, handle), daemon=True)
            self.thread.start()
            return
        except Exception:
            self.source = None
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.source = "nvidia-smi"
            self.thread = threading.Thread(target=self._smi_loop, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _smi_loop(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 6:
                continue
            try:
                self.sm.append(float(f[0])); self.mx = max(self.mx, float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[2:6]):
                if v.lower().startswith("active"):
                    self.reasons.add(name)

    def stop(self):
        self.stop_flag = True
        if self.proc:
            self.proc.terminate()
        if self.thread:
            self.thread.join(timeout=1.0)
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.mx or None,
                "reasons": sorted(self.reasons), "samples": len(self.sm), "source": self.source}


# ------------------------------------------------------------------------------------------ synthetic inputs (SURVEY 8d)
def synth_tokens(rng, B, cfg, regime="full", mean_len=3.0):
    """FULL rows: [PAD] + (T-2 ids ~ Zipf-like over [2,V)) + [EOS]; REAL rows: L ~ clip(Poisson(mean_len), 1, T-2) real
    tokens, left-padded (data_utils.py:149-155)."""
    V, T = cfg["V"], cfg["T"]
    u = rng.random((B, T - 2))
    ids = np.minimum(2 + np.floor((V - 2) * u ** 3), V - 1).astype(np.int32)
    out = np.zeros((B, T), np.int32)
    out[:, T - 1] = 1
    if regime == "full":
        out[:, 1:T - 1] = ids
        return out
    L = np.clip(rng.poisson(mean_len, size=B), 1, T - 2)
    col = np.arange(T - 2)[None, :]
    keep = col >= (T - 2 - L)[:, None]                       # the last L of the T-2 token slots
    out[:, 1:T - 1] = np.where(keep, ids, 0)
    return out


def init_weights(cfg, seed=1234):
    """Reference initialisers (sse_model.py:160,188-189,227; BasicLSTMCell Glorot kernel / zero bias) -- the oracle's."""
    sys.path.insert(0, os.path.join(REPO, "oracle"))
    import sse_oracle as O
    kw = {}
    if cfg["mode"] in ("dual-cnn", "source_only_cnn"):
        kw = dict(cnn_filter_sizes=cfg.get("cnn_k", ()), cnn_num_filters=cfg.get("cnn_f", ()))
    if cfg["mode"] in ("source-encoder-only", "source_only_cnn"):
        kw["target_space_size"] = cfg["targets"]
    return O.init_params(cfg["mode"], cfg["V"], cfg["We"], cfg["E"], cfg["H"], cfg["H"], seed=seed, **kw)


def encoder_flops(cfg):
    """flops per encoded sequence (SURVEY 8d): LSTM 2 T (We+H) 4H + 2 H E; CNN sum_k 2 (T-k+1) k We F_k + 2 (sum F) E."""
    T, We, H, E = cfg["T"], cfg["We"], cfg["H"], cfg["E"]
    if cfg["mode"] in ("dual-cnn", "source_only_cnn"):
        ks, fs = cfg["cnn_k"], cfg["cnn_f"]
        return sum(2 * (T - k + 1) * k * We * f for k, f in zip(ks, fs)) + 2 * sum(fs) * E
    return 2 * T * (We + H) * 4 * H + 2 * H * E


def make_handle(cfg, device, sse_ffi, k=K_TOP):
    return sse_ffi.Handle(cfg["mode"], cfg["V"], cfg["We"], cfg["E"], cfg["H"], cfg["H"], cfg["T"], predict_nbest=k, device=device,
                          precision=sse_ffi.PRECISION_TC, target_space_size=cfg["targets"] if "only" in cfg["mode"] else 0,
                          cnn_filter_sizes=cfg.get("cnn_k", ()), cnn_num_filters=cfg.get("cnn_f", ()))


# ------------------------------------------------------------------------------------------
def run_b200(args):
    import torch
    import torch.distributed as dist
    import sse_dist
    import sse_ffi

    cfg = args.cfg
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries exactly ONE JSON line: anything libraries print (e.g. NCCL's version banner) goes to stderr
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the B200 arm has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    emu = args.emulate_world if world == 1 and args.emulate_world > 1 else 0
    G = emu or world                             # ranks whose queries this rank scans for
    V, WE, H, E, T = cfg["V"], cfg["We"], cfg["H"], cfg["E"], cfg["T"]
    Ql, k = cfg["queries"], K_TOP                # query rows this rank encodes per step
    Q = Ql * G                                   # query rows this rank scans for per step
    # rows per shard: the config's total over the GPU count it names (c5: 5M over 8), else over this job's ranks
    shard_div = cfg.get("targets_at_gpus", 0) or G
    n_local = cfg["targets"] // shard_div
    n_total = n_local * G
    table_mode = "only" in cfg["mode"]           # target side is a variable [targetSpaceSize, E], not an encoder
    F_ENC = encoder_flops(cfg)

    h = make_handle(cfg, local, sse_ffi)
    params = init_weights(cfg)
    h.set_params(params)
    h.set_option("search", args.search)

    # ---- index shard, resident in HBM
    rng_t = np.random.default_rng(7 + rank)
    index_kind = args.index
    t_build = None
    if table_mode:
        tab = params["target_embedding/tgt_seq_embedding"][rank * n_local:(rank + 1) * n_local]
        tab = tab / np.sqrt(np.maximum((tab * tab).sum(-1, keepdims=True), 1e-12))      # norm_tgt_seq_embedding of the table (sse_model.py:233,283)
        h.index_set(tab.astype(np.float32), n_local, global_offset=rank * n_local)
        index_kind = "target table (variable target_embedding/tgt_seq_embedding, l2-normalised)"
    elif index_kind == "encoded":
        ttok = synth_tokens(rng_t, n_local, cfg, "real", 8.0)                           # titles: ~8 subtokens (SURVEY appendix C)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        h.index_build(torch.from_numpy(ttok).cuda(), global_offset=rank * n_local, batch=16384)
        torch.cuda.synchronize()
        t_build = time.perf_counter() - t0
        del ttok
    else:
        g = torch.Generator(device="cuda").manual_seed(7 + rank)
        idx = torch.randn(n_local, E, device="cuda", generator=g)
        idx = idx / idx.norm(dim=1, keepdim=True)
        h.index_set(idx, n_local, global_offset=rank * n_local)
        del idx
    # Timing rule "inputs larger than L2": a shard whose fp16 copy is smaller than ~2x the 126 MB L2 would be served from
    # cache after the first step.  Such shards are held in several identical replicas (separate handles = separate HBM
    # buffers) scanned in rotation, so every step streams bytes last touched more than an L2-full of index traffic ago.
    scan_handles = [h]
    shard_fp16 = n_local * E * 2
    if shard_fp16 < 2 * L2_BYTES and not args.no_replicas:
        try:
            n_rep = int(2 * L2_BYTES // shard_fp16) + 2
            host_idx = torch.from_numpy(h.index_get(0, n_local)).cuda()
            for _ in range(n_rep - 1):
                hr = make_handle(cfg, local, sse_ffi)
                hr.set_option("search", args.search)
                hr.index_set(host_idx, n_local, global_offset=rank * n_local)
                scan_handles.append(hr)
            del host_idx
        except Exception as ex:                  # never lose the run over the cache-hygiene measure: fall back and say so
            print("bench.py: index replicas not created (%r); scanning a single L2-resident shard" % (ex,), file=sys.stderr)
            scan_handles = [h]
    n_rep = len(scan_handles)
    scan_state = {"i": 0}

    def scan_handle():
        hs = scan_handles[scan_state["i"] % n_rep]
        scan_state["i"] += 1
        return hs

    def total_launches():
        return sum(x.launch_count() for x in scan_handles)

    # ---- query batches: the step's G x Ql queries; rank r encodes rows [Ql r, Ql r + Ql)
    n_batches = 4
    tokens = {}
    for regime, mean in (("full", 0.0), ("real", 3.0)):
        rng = np.random.default_rng(42 if regime == "full" else 43)
        host = [torch.from_numpy(synth_tokens(rng, Q, cfg, regime, mean)[rank * Ql:(rank + 1) * Ql].copy()).pin_memory() for _ in range(n_batches)]
        tokens[regime] = (host, [t.cuda() for t in host])
    cur = {"host": tokens["full"][0], "dev": tokens["full"][1]}

    enc_local = [torch.empty(Ql, E, device="cuda") for _ in range(2)]
    enc2 = [torch.empty(Q, E, device="cuda") for _ in range(2)]
    sc = torch.empty(Q, k, device="cuda")
    ix = torch.empty(Q, k, device="cuda", dtype=torch.int32)
    packed = torch.empty(Q, 2 * k, device="cuda")
    recv = torch.empty(G * Ql, 2 * k, device="cuda") if G > 1 else None
    fs = torch.empty(Ql, k, device="cuda")
    fi = torch.empty(Ql, k, device="cuda", dtype=torch.int32)
    n_out = Ql if G > 1 else Q
    out_s_host2 = [torch.empty(n_out, k).pin_memory() for _ in range(2)]
    out_i_host2 = [torch.empty(n_out, k, dtype=torch.int32).pin_memory() for _ in range(2)]
    e2e_done = [torch.cuda.Event(), torch.cuda.Event()]
    e2e_state = {"n": 0}
    stream = torch.cuda.current_stream()

    pipeline = not args.no_pipeline
    enc_stream = torch.cuda.Stream() if pipeline else stream
    enc_ready = [torch.cuda.Event(), torch.cuda.Event()]
    enc_free = [torch.cuda.Event(), torch.cuda.Event()]
    state = {"primed": False, "n": 0}
    if args.search_ctas < 0:
        args.search_ctas = 108 if G <= 4 else 0
    if args.search_late < 0:        # one late scan CTA per SM the cap reserves for the encoder (measured: 0 -> 1.53, 32 -> 1.57, 40 -> 1.60 M q/s)
        n_sm = torch.cuda.get_device_properties(local).multi_processor_count
        args.search_late = max(0, n_sm - args.search_ctas) if (pipeline and args.search_ctas > 0) else 0
    if args.cluster_rows < 0:
        args.cluster_rows = 128 if (pipeline and args.search_ctas > 0) else 0
    h.set_option("cluster_rows", args.cluster_rows)
    if pipeline:
        for hs in scan_handles:
            hs.set_option("search_ctas", args.search_ctas)
            hs.set_option("search_late_ctas", args.search_late if args.search_ctas else 0)
            hs.set_option("search_late_share", args.search_late_share)

    def encode_all(b, out, scratch, st):
        """this rank's Ql queries through the source encoder; N > 1: all-gather of the [Ql, E] encodings so that every rank
        holds the step's G x Ql query vectors for its index shard"""
        if G == 1:
            h.encode(sse_ffi.SIDE_SRC, cur["dev"][b], Ql, out, True, st)
        else:
            h.encode(sse_ffi.SIDE_SRC, cur["dev"][b], Ql, scratch, True, st)
            if emu:
                out.view(G, Ql, E).copy_(scratch.unsqueeze(0).expand(G, Ql, E))
            else:
                sse_dist.allgather_rows(scratch, out)

    def issue_encode(b, slot):
        with torch.cuda.stream(enc_stream):
            enc_stream.wait_event(enc_free[slot])          # the scan that last read this slot has finished
            encode_all(b, enc2[slot], enc_local[slot], enc_stream)
            enc_ready[slot].record(enc_stream)

    def scan_and_merge(q_all):
        if G == 1:
            scan_handle().search(q_all, Q, k, sc, ix, stream)
            return
        # one packed [Q, 2k] block straight from the scan's finalize kernel; rows [Ql r, Ql r + Ql) belong to rank r:
        # the all-to-all hands every rank the G per-shard blocks of its OWN Ql queries, merged by one kernel
        scan_handle().search_packed(q_all, Q, k, packed, stream)
        if emu:
            recv.view(G, Ql, 2 * k).copy_(packed[:Ql].unsqueeze(0).expand(G, Ql, 2 * k))
        else:
            dist.all_to_all_single(recv, packed)
        h.merge_packed(recv, G, Ql, k, fs, fi, stream)

    def step_device(b):
        if pipeline:
            # software pipeline over steps: this step's scan runs while the NEXT step's batch is encoded on the
            # other stream (every step still encodes one batch and scans the index once for one batch)
            n = state["n"]
            if not state["primed"]:
                for sl in range(2):
                    enc_free[sl].record(stream)
                enc_stream.wait_stream(stream)
                issue_encode(b, n & 1)
                state["primed"] = True
            stream.wait_event(enc_ready[n & 1])
            issue_encode((b + 1) % n_batches, (n + 1) & 1)
            scan_and_merge(enc2[n & 1])
            enc_free[n & 1].record(stream)
            state["n"] = n + 1
        else:
            encode_all(b, enc2[0], enc_local[0], stream)
            scan_and_merge(enc2[0])

    def step_e2e(b):
        if pipeline:
            with torch.cuda.stream(enc_stream):                          # H2D of the NEXT step's inputs, ahead of its encode
                cur["dev"][(b + 1) % n_batches].copy_(cur["host"][(b + 1) % n_batches], non_blocking=True)
        else:
            cur["dev"][b].copy_(cur["host"][b], non_blocking=True)       # H2D of the step's inputs
        step_device(b)
        src_s, src_i = (fs, fi) if G > 1 else (sc, ix)
        n = e2e_state["n"]
        out_s_host2[n & 1].copy_(src_s, non_blocking=True)             # D2H of the step's result
        out_i_host2[n & 1].copy_(src_i, non_blocking=True)
        if pipeline:
            # the host consumes step s-1's result while step s runs (every step's result is still read on the host:
            # double-buffered pinned outputs; the last one is awaited by the closing barrier)
            e2e_done[n & 1].record(stream)
            if n > 0:
                e2e_done[(n - 1) & 1].synchronize()
        else:
            stream.synchronize()
        e2e_state["n"] = n + 1

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        state["primed"] = False
        state["n"] = 0
        e2e_state["n"] = 0

    def timed(fn, steps, warmup, repeats):
        """`repeats` x [W warm-up steps, then EXACTLY `steps` steps bracketed by barrier + synchronize, CUDA events, max over
        ranks]; returns (median ms of the K-step region, all samples)"""
        samples = []
        for _ in range(max(1, repeats)):
            for w in range(warmup):
                fn(w % n_batches)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for s in range(steps):
                fn(s % n_batches)
            e1.record()
            barrier()
            ms = e0.elapsed_time(e1)
            if world > 1:
                t = torch.tensor([ms], device="cuda")
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms = float(t.item())
            samples.append(ms)
            warmup = min(warmup, 1)              # later repeats are already warm: one step re-primes the pipeline
        return float(np.median(samples)), samples

    try:
        dev_uuid = torch.cuda.get_device_properties(local).uuid
    except Exception:
        dev_uuid = None
    sampler = ClockSampler(local, dev_uuid)
    if rank == 0:
        sampler.start()
    W = max(args.warmup, 3)
    h.set_option("pad_skip", 0)                  # FULL regime: all T steps are executed, as the reference does
    l0 = total_launches()
    ms_dev, dev_samples = timed(step_device, args.steps, W, args.repeats)
    dump = {}
    if args.dump_outputs and rank == 0:          # the last timed step's result, before later regions reuse the buffers
        src_s, src_i = (fs, fi) if G > 1 else (sc, ix)
        dump["top_scores"] = src_s.cpu().numpy().astype(np.float32)
        dump["top_ids"] = src_i.cpu().numpy().astype(np.float64)
    n_steps_run = sum([args.steps + (W if i == 0 else min(W, 1)) for i in range(max(1, args.repeats))])
    launches_per_step = (total_launches() - l0) / float(n_steps_run)
    ms_e2e, e2e_samples = timed(step_e2e, args.steps, W, args.repeats)

    # ---- REAL regime (queries ~3 tokens of T, per-tile pad-prefix start on): same step, same index
    real = None
    if not args.no_real_regime and not table_mode and "cnn" not in cfg["mode"]:
        cur["host"], cur["dev"] = tokens["real"]
        h.set_option("pad_skip", 1)
        # a REAL-regime encode is a few steps long: no point reserving SMs for it (measured 1.29 M q/s with the 108-CTA cap, 1.75 M without)
        h.set_option("cluster_rows", 0)
        if pipeline:
            for hs in scan_handles:
                hs.set_option("search_ctas", 0)
                hs.set_option("search_late_ctas", 0)
        ms_r, _ = timed(step_device, args.steps, W, args.repeats)
        ms_re, _ = timed(step_e2e, args.steps, W, args.repeats)
        real = {"value": Ql * world * args.steps / (ms_r * 1e-3), "unit": "queries/s", "ms_per_step": ms_r / args.steps,
                "e2e": {"value": Ql * world * args.steps / (ms_re * 1e-3), "ms_per_step": ms_re / args.steps},
                "queries": "L ~ clip(Poisson(3), 1, T-2) real tokens per row, left-padded", "pad_prefix_start": True,
                "pipeline": "same 2-stage pipeline, scan grid uncapped (the short encode shares the SMs)"}
        cur["host"], cur["dev"] = tokens["full"]
        h.set_option("pad_skip", 0)
        h.set_option("cluster_rows", args.cluster_rows)
        if pipeline:
            for hs in scan_handles:
                hs.set_option("search_ctas", args.search_ctas)
                hs.set_option("search_late_ctas", args.search_late if args.search_ctas else 0)

    # ---- dominant kernel (the index scan) timed alone, CUDA events on the launching stream, for the roofline
    for hs in scan_handles:
        hs.set_option("search_ctas", 0)
        hs.set_option("search_late_ctas", 0)
    torch.cuda.synchronize()
    # The GPU runs these kernels under its power cap, and the cap's controller remembers the load before: right after the timed
    # regions above the same search measures 8-15 % slower than after a pause (0.337 vs 0.369 ms on one box).  The roofline
    # denominator is the BURST figure of MEASURED_PEAKS.json (a kernel timed alone after idle), so the kernel is timed the same way.
    time.sleep(2.0)
    encode_all(0, enc2[0], enc_local[0], stream)
    for _ in range(3):
        scan_handle().search(enc2[0], Q, k, sc, ix, stream)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = max(5, args.steps)
    e0.record()
    for _ in range(reps):
        scan_handle().search(enc2[0], Q, k, sc, ix, stream)
    e1.record()
    torch.cuda.synchronize()
    ms_search = e0.elapsed_time(e1) / reps
    enc_alone = {}
    time.sleep(1.0)
    for rows_opt in (0, 128):             # the encoder alone on all SMs: the library's own choice (64-row clusters for a query batch) and 128-row clusters
        h.set_option("cluster_rows", rows_opt)
        for _ in range(2):
            h.encode(sse_ffi.SIDE_SRC, cur["dev"][0], Ql, enc_local[0], True, stream)
        e0.record()
        for _ in range(reps):
            h.encode(sse_ffi.SIDE_SRC, cur["dev"][0], Ql, enc_local[0], True, stream)
        e1.record()
        torch.cuda.synchronize()
        enc_alone[rows_opt] = e0.elapsed_time(e1) / reps
    h.set_option("cluster_rows", args.cluster_rows)
    ms_enc = enc_alone[0]
    clocks = sampler.stop() if rank == 0 else None

    # ---- verification (outside every timed region): the last scan's rows against the exact fp32 SIMT scan of the same shard,
    # and the filter's bookkeeping (candidates that passed the sampled threshold, rows that fell back to brute force)
    verify = None
    try:
        stats = scan_handles[(scan_state["i"] - 1) % n_rep].search_stats() if args.search != 1 else None
        nv = min(Q, 64)
        rows = np.linspace(0, Q - 1, nv).astype(np.int64)
        qv = enc2[0][torch.from_numpy(rows).cuda()].contiguous()
        vs, vi = torch.empty(nv, k, device="cuda"), torch.empty(nv, k, device="cuda", dtype=torch.int32)
        h.set_option("search", 1)
        h.search(qv, nv, k, vs, vi, stream)
        h.set_option("search", args.search)
        torch.cuda.synchronize()
        got_i, got_s = ix[torch.from_numpy(rows).cuda()].cpu().numpy(), sc[torch.from_numpy(rows).cuda()].cpu().numpy()
        verify = {"rows_checked": int(nv), "against": "exact fp32 SIMT scan of the same shard (search_simt.cu)",
                  "index_agreement": float((got_i == vi.cpu().numpy()).mean()),
                  "max_score_diff": float(np.abs(got_s - vs.cpu().numpy()).max())}
        if stats:
            verify.update({"candidates_per_row": stats["candidates"] / max(1, stats["rows"]), "fallback_rows": stats["fallback_rows"],
                           "scan_work_items": stats["scan_items"]})
    except Exception as ex:
        verify = {"error": repr(ex)}

    # ---- secondary metric: train-step/s (pair-loss step: fwd both towers, BPTT, clip, Adagrad)
    train = None
    trainable = cfg["mode"] in ("dual-encoder", "shared-encoder")
    if args.train_steps > 0 and trainable:
        Bt = args.train_rows or cfg.get("train_rows", 1024)
        rng_tr = np.random.default_rng(100 + rank)
        n_pos = Bt // 3 if Bt % 3 == 0 and cfg.get("train_rows") else Bt // 2        # c4: 512 positives + 1024 negatives
        reps_neg = Bt // n_pos
        src_t = torch.from_numpy(np.repeat(synth_tokens(rng_tr, n_pos, cfg), reps_neg, axis=0)).cuda()
        tgt_t = torch.from_numpy(synth_tokens(rng_tr, Bt, cfg)).cuda()
        lab_t = torch.tensor(([1.0] + [0.0] * (reps_neg - 1)) * n_pos, device="cuda")

        def tstep():
            if world > 1:
                sse_dist.allreduce_train_step(h, src_t, tgt_t, lab_t, Bt * world)
            else:
                h.train_step(src_t, tgt_t, lab_t, stream=stream, want_scalars=False)
        for _ in range(2):
            tstep()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.train_steps):
            tstep()
        e1.record()
        barrier()
        ms_t = e0.elapsed_time(e1)
        if world > 1:
            tt = torch.tensor([ms_t], device="cuda")
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            ms_t = float(tt.item())
        fl = 3.0 * Bt * world * 2 * F_ENC
        train = {"metric": "train-step/s", "value": args.train_steps / (ms_t * 1e-3), "ms_per_step": ms_t / args.train_steps,
                 "pair_rows_per_gpu": Bt, "pair_rows_global": Bt * world, "positives_per_gpu": n_pos, "dtype": "bf16 operands / f32 accumulate, state, stash and optimizer (tcgen05 GEMMs)" if Bt % 8 == 0 and WE % 8 == 0 and H % 8 == 0 else "f32",
                 "flops_per_step": fl, "achieved_tflops": fl / (ms_t / args.train_steps * 1e-3) / 1e12,
                 "parallelism": "data-parallel x%d, all-reduce of the gradient arena" % world if world > 1 else "single GPU"}
        if args.dump_outputs and rank == 0:      # the parameters the last train step wrote; large tables as a fixed row sample
            rng_d = np.random.default_rng(0)
            for name, _ in h.param_names():
                v = h.get_param(name)
                if v.ndim and v.shape[0] > 4096:
                    v = v[np.sort(rng_d.choice(v.shape[0], 4096, replace=False))]
                dump["param." + name.replace("/", ".")] = v.astype(np.float32)

    if dump:
        total = sum(v.nbytes for v in dump.values())
        if total > 64 << 20:
            raise SystemExit("bench.py: --dump-outputs: %d bytes exceed 64 MB" % total)
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, v in dump.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), v)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    hbm_gbs, bf16_tf, src = load_peaks()
    use_tc = args.search != 1
    flops = 2.0 * Q * n_local * E
    bytes_alg = n_local * E * (2 if use_tc else 4) + Q * E * 4 + Q * k * 8
    t_s = ms_search * 1e-3
    tensor_bound_s = flops / (bf16_tf * 1e12)
    hbm_bound_s = bytes_alg / (hbm_gbs * 1e9)
    if use_tc and tensor_bound_s >= hbm_bound_s:
        roof = {"bound": "tensor", "achieved": flops / t_s / 1e12, "peak": bf16_tf, "unit": "TFLOP/s"}
    else:
        roof = {"bound": "hbm", "achieved": bytes_alg / t_s / 1e9, "peak": hbm_gbs, "unit": "GB/s"}
    roof["frac"] = roof["achieved"] / roof["peak"]
    roof["traffic"] = None
    try:        # dram__bytes_read.sum + dram__bytes_write.sum of the scan kernel from the committed ncu --set full capture
        with open(os.path.join(REPO, "profiles", "traffic.json")) as f:
            tj = json.load(f)
        if tj.get("targets_per_gpu") == n_local and tj.get("queries") == Q and tj.get("E", 256) == E:
            roof["traffic"] = tj["scan_filter_dram_bytes"]
            roof["traffic_source"] = tj.get("source")
    except Exception:
        pass
    roof["peak_source"] = src
    roof["kernel"] = "search (prep+sample scan+select_tau+filter scan+finalize)" if use_tc else "search_simt_kernel+merge"
    roof["ms_per_launch"] = ms_search
    roof["timing"] = "CUDA events around %d back-to-back searches on the launching stream, after 3 warm-up searches and a 2 s idle (burst conditions, like the peak it is divided by)" % reps
    roof["algorithmic"] = {"flops": flops, "bytes": bytes_alg}
    roof["encoder"] = {"ms": ms_enc, "rows": Ql, "flops": Ql * F_ENC, "achieved_tflops": Ql * F_ENC / (ms_enc * 1e-3) / 1e12,
                       "achieved_frac_of_bf16_peak": Ql * F_ENC / (ms_enc * 1e-3) / 1e12 / bf16_tf,
                       "ms_128_row_clusters": enc_alone[128], "cluster_rows_in_timed_step": args.cluster_rows,
                       "kernel": "source tower of the step, timed alone on all SMs with the library's own cluster size (token check + tower + "
                                 "projection/l2-norm); flops = the full encoder (x and h parts, all T steps)"}

    total_q = Ql * world * args.steps
    out = {
        **({"emulated": "one rank's share of a %d-GPU step on one GPU; collectives replaced by local copies -- NOT a multi-GPU result" % emu} if emu else {}),
        "metric": "queries/sec encode+cosine-top-k", "value": total_q / (ms_dev * 1e-3), "unit": "queries/s",
        "n_gpus": world, "steps": args.steps, "warmup": W, "ms_per_step": ms_dev / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f16 operands / f32 accumulate (tcgen05 scan + encoder), exact f32 re-rank of the top-k" if use_tc else "f32",
        "data": "synthetic",
        "config": {"workload": "%s; Q=%d queries/step (FULL-length rows), cosine top-%d over N=%d targets (%d per GPU shard)"
                               % (cfg["name"], Ql * world, k, n_local * world, n_local),
                   "name": args.config, "mode": cfg["mode"], "index": index_kind,
                   "index_build_s": t_build, "targets_per_gpu": n_local, "targets_total": n_local * world, "queries_per_step": Ql * world,
                   "queries_per_step_per_gpu": Ql, "k": k, "regime": "FULL (pad-prefix start off: all T steps run)",
                   "parallelism": ("index row-shard x%d, %d queries/step: each rank encodes its %d, NCCL all-gather of the [%d,E] encodings, every rank "
                                   "scans its shard for all %d and emits one packed [Q,2k] block, NCCL all-to-all of the per-owner row blocks, "
                                   "merge of G*k candidates for the rank's own %d rows" % (world, Q, Ql, Ql, Q, Ql)) if world > 1 else "single GPU",
                   "pipeline": ("2-stage over steps: encoder of batch s+1 (its own stream, %d SMs left free by the scan grid cap %d%s) overlaps the scan of batch s"
                                % (148 - (args.search_ctas or 148), args.search_ctas or 148,
                                   (" + %d late scan CTAs at %d%% share for those SMs once the encoder leaves" % (args.search_late, args.search_late_share))
                                   if args.search_late and args.search_ctas else "")) if pipeline else "none (encode then scan on one stream)",
                   "timing": "median of %d repeats of the %d-step region (CUDA events, barrier + synchronize on both sides, max over ranks)" % (max(1, args.repeats), args.steps),
                   "l2": (("no flush: the fp16 index shard (%.0f MB) is re-streamed every step and exceeds L2 (126 MB); query batches rotate"
                           % (shard_fp16 / 1e6)) if n_rep == 1 and shard_fp16 > L2_BYTES else
                          ("no flush: the fp16 index shard is %.0f MB, so %d identical replicas in separate HBM buffers are scanned in "
                           "rotation (%.0f MB of index between two scans of the same bytes > L2 126 MB); query batches rotate"
                           % (shard_fp16 / 1e6, n_rep, (n_rep - 1) * shard_fp16 / 1e6)) if n_rep > 1 else
                          ("no flush: the fp16 index shard (%.0f MB) FITS in L2 (126 MB) and is scanned every step: after the first "
                           "step the scan is served from L2; query batches rotate" % (shard_fp16 / 1e6)))},
        "repeats_ms": dev_samples,
        "e2e": {"value": total_q / (ms_e2e * 1e-3), "unit": "queries/s", "h2d_bytes_per_step": Ql * T * 4,
                "d2h_bytes_per_step": n_out * k * 8, "ms_per_step": ms_e2e / args.steps, "repeats_ms": e2e_samples},
        "gpu_launches": int(round(launches_per_step * args.steps)),
        "clocks": clocks,
        "roofline": roof,
        "verify": verify,
        "regimes": {"real": real} if real else None,
        "train": train,
    }
    if args.config == "c4" and train:           # the config's own metric leads the line; the retrieval figures stay under "retrieval"
        out = {"metric": "train-step/s", "value": train["value"], "unit": "steps/s", "n_gpus": world, "steps": args.train_steps, "warmup": 2,
               "ms_per_step": train["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": train["dtype"],
               "data": "synthetic", "config": {"workload": cfg["name"], "name": "c4", **{kk: train[kk] for kk in ("pair_rows_per_gpu", "pair_rows_global", "positives_per_gpu", "parallelism")}},
               "roofline": {"bound": "tensor", "achieved": train["achieved_tflops"], "peak": bf16_tf, "unit": "TFLOP/s", "frac": train["achieved_tflops"] / bf16_tf,
                            "traffic": None, "peak_source": src, "kernel": "train step (forward with stash, BPTT, clip, Adagrad)", "algorithmic": {"flops": train["flops_per_step"]}},
               "clocks": clocks, "gpu_launches": None, "retrieval": {kk: out[kk] for kk in ("value", "ms_per_step", "e2e")}}
    if not args.no_cpu_baseline and world == 1:
        out["cpu_baseline"] = cpu_reference(cfg, args.cpu_sample_queries, min(n_local, args.cpu_sample_targets))["line"]
    os.write(json_fd, (json.dumps(out) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------
class CpuReference(object):
    """The reference's CPU path on a bounded sample: numpy restatement of the TF1 encoder (oracle, BLAS threads = all
    cores) + the reference's float64 np.dot and full argsort (sse_evaluator.py:110-111, data_utils.py:263-267).
    Inputs (weights, tokens, the float64 index the Evaluator holds) are built ONCE; step() times only
    encode + np.dot + getSortedResults."""

    def __init__(self, cfg, Qs, Ns):
        sys.path.insert(0, os.path.join(REPO, "oracle"))
        import sse_oracle as O
        self.O, self.cfg, self.Qs, self.Ns = O, cfg, Qs, Ns
        self.p = init_weights(cfg)
        self.tok = synth_tokens(np.random.default_rng(42), Qs, cfg)
        r2 = np.random.default_rng(7)
        tgt = r2.standard_normal((Ns, cfg["E"]), dtype=np.float32)
        tgt /= np.linalg.norm(tgt, axis=1, keepdims=True)
        self.tgt64 = tgt.astype(np.float64)              # Evaluator.__init__ parses the index into float64 (sse_evaluator.py:80-92)
        self.cores = os.cpu_count() or 1

    def step(self):
        t0 = time.perf_counter()
        enc = self.O.encode(self.p, self.cfg["mode"], "src", self.tok, True)
        t1 = time.perf_counter()
        d = np.dot(enc, self.tgt64.T)
        t2 = time.perf_counter()
        self.O.get_sorted_results(d)
        t3 = time.perf_counter()
        return (t3 - t0, t1 - t0, t2 - t1, t3 - t2)

    def line(self, best):
        return {"value": self.Qs / best[0], "unit": "queries/s", "cores": self.cores, "kind": "port",
                "sample": "Q=%d queries x N=%d targets (same model shape; encode %.2fs + np.dot f64 %.2fs + full argsort %.2fs = %.2fs per step; "
                          "gaussian unit-vector index: building 1M encodings with the numpy encoder would take hours and the dot / sort cost does "
                          "not depend on the values)" % (self.Qs, self.Ns, best[1], best[2], best[3], best[0])}


def cpu_reference(cfg, Qs, Ns, steps=1, warm=0):
    ref = CpuReference(cfg, Qs, Ns)
    for _ in range(warm):
        ref.step()
    runs = [ref.step() for _ in range(max(1, steps))]
    best = min(runs, key=lambda r: r[0])
    return {"runs": runs, "line": ref.line(best), "ref": ref}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = args.cfg
    shard_div = cfg.get("targets_at_gpus", 0) or max(1, args.gpus)
    n_local = cfg["targets"] // shard_div
    Qs, Ns = min(cfg["queries"], args.cpu_sample_queries), min(n_local, args.cpu_sample_targets)
    # keep the whole run within a few minutes: one warm-up + at most 3 timed steps of the bounded sample
    steps = min(max(1, args.steps), 3)
    warm = min(max(0, args.warmup), 1)
    r = cpu_reference(cfg, Qs, Ns, steps=steps, warm=warm)
    total = sum(x[0] for x in r["runs"])
    val = Qs * steps / total
    mean = tuple(float(np.mean([x[i] for x in r["runs"]])) for i in range(4))
    out = {"impl": "reference", "metric": "queries/sec encode+cosine-top-k", "value": val, "unit": "queries/s",
           "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": total / steps * 1e3, "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "f32 encoder / f64 scoring", "data": "synthetic",
           "config": {"workload": "%s; CPU bounded sample Q=%d x N=%d (B200 arm: Q=%d x N=%d per GPU)" % (cfg["name"], Qs, Ns, cfg["queries"], n_local),
                      "name": args.config},
           "cpu_baseline": dict(r["ref"].line(mean), value=val),
           "e2e": {"value": val, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
