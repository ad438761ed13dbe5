#!/usr/bin/env python3
"""bench.py — requests/sec through tokenize + block-hash + prefix-match (+ cache-aware routing) at
4K-token prompts (BASELINE.json metric) on N B200s, next to the CPU oracle on the host cores.

  python bench.py --gpus N --steps K --warmup W          # this repo's CUDA path
  python bench.py --impl reference --gpus N ...          # the reference's CPU path (oracle port)
  torchrun --nproc-per-node N bench.py --gpus N ...      # N > 1: one rank per GPU, weak scaling

A step = one pass of the hot path over one batch of synthetic prompts (default 65 536 prompts x
4 096 tokens per GPU, BASELINE config 2, matched against a 1 048 576-key prefix index over 64
instances with the 80 %-shared-prefix Zipf-0.9 workload of config 3).

  value      : device-resident throughput — prompts already in HBM, the four kernels back to back
  e2e        : the same work through the C-ABI call xllm_ingest_batch with page-locked HOST
               buffers; host->device and device->host copies are inside the timed region
  roofline   : the dominant kernel's algorithmic bytes / its CUDA-event time vs MEASURED_PEAKS.json
  cpu_baseline: the CPU oracle (port of the reference path) on a bounded sample, all host cores
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
MODEL_DIR = os.path.join(ROOT, "tests", "golden", "sp_bpe_8k")
METRIC = "requests/sec tokenize+hash+match @4K-token prompts"
N_INST = 64
BLOCK = 128
SEED = 1024


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--requests", type=int, default=65536, help="prompts per GPU per step")
    ap.add_argument("--tokens", type=int, default=4096)
    ap.add_argument("--index-keys", type=int, default=1 << 20)
    ap.add_argument("--cpu-sample", type=int, default=0, help="prompts in the CPU-baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--chunk-requests", type=int, default=0)
    ap.add_argument("--no-c5", action="store_true", help="skip the config-5 (EPD mix) side measurement at N = 1")
    ap.add_argument("--c5-requests", type=int, default=8192)
    ap.add_argument("--no-honest-text", action="store_true", help="skip the natural-text / memo-off / large-vocabulary "
                                                                   "tokenizer side measurements")
    ap.add_argument("--no-latency", action="store_true", help="skip the service-shaped latency side measurement")
    ap.add_argument("--index", default="auto", choices=["auto", "replicated", "sharded"],
                    help="prefix index placement at N > 1: sharded = BASELINE config 4 (hash-range shards, index N x "
                         "--index-keys, one NCCL all-to-all each way per batch); auto = sharded when N > 1")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed (rank 0's requests, "
                                                          "a fixed sample of rows) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the CUDA path's results (--impl b200)")
    return args


def host_threads():
    """Threads the CPU arm may really use: the smaller of the scheduler affinity mask and the cgroup CPU quota
    (os.cpu_count() reports the machine, not the container's share).  Returns (threads, detail dict)."""
    ncpu = os.cpu_count() or 1
    try:
        aff = len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        aff = ncpu
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            with open(path) as f:
                txt = f.read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    quota = float(txt[0]) / float(txt[1])
            else:
                q = float(txt[0])
                if q > 0:
                    with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f2:
                        quota = q / float(f2.read().split()[0])
            break
        except (OSError, ValueError, IndexError):
            continue
    use = aff if quota is None else max(1, min(aff, int(quota + 0.5)))
    return use, {"os_cpu_count": ncpu, "sched_affinity": aff, "cgroup_quota_cpus": quota}


# ----------------------------------------------------------------------------------------------
# workload: prompts + the index content they are matched against
def word_token_counts_gpu(h, vocab):
    from xllm_service_b200 import workload
    wb = workload.pack_prompts(vocab)
    _, n, st = h.encode_batch(wb.text, wb.offsets, 32)
    assert (st == 0).all()
    return n


def word_token_counts_cpu(sp, vocab, threads):
    from xllm_service_b200 import workload
    wb = workload.pack_prompts(vocab)
    _, n = sp.encode_batch(wb.text, wb.offsets, 32, n_threads=threads)
    return n


def make_batch(n_req, n_tok, wcnt, seed, device):
    from xllm_service_b200 import workload
    return workload.make_prompts_exact_tokens(
        n_req, n_tok, wcnt, seed=seed, device=device,
        shared_prefix=dict(n_prefixes=1024, frac=0.8, min_blocks=8, max_blocks=24, block_tokens=BLOCK))


def index_events(prefix_keys, n_total, rng):
    """The KvCacheEvent stream that populates the index (SURVEY §8d config 3): every shared-prefix block
    is held in HBM by 1-3 instances over a leading part of the prefix, filler keys by one instance;
    then 10 % of the entries are offloaded to DRAM and 10 % on to SSD.  Returns a list of
    ("prefix" | "fill", instance_id, stored, offload, removed) uint8 [k,16] events, in order, with publish markers
    (None).  Prefix and filler keys are disjoint, so a consumer that only ever looks up prefix keys (the CPU oracle of
    the sharded gate) may skip the "fill" events."""
    stored = [[] for _ in range(N_INST)]
    used = 0
    for keys in prefix_keys:                      # keys: [L,16] of one shared prefix
        L = keys.shape[0]
        for _ in range(int(rng.integers(1, 4))):
            i = int(rng.integers(0, N_INST))
            stored[i].append(keys[:int(rng.integers(max(1, L // 2), L + 1))])
        used += L
    n_fill = max(0, n_total - used)
    fill = rng.integers(0, 256, size=(n_fill, 16), dtype=np.uint8)
    owner = rng.integers(0, N_INST, size=n_fill)
    ev = []
    for i in range(N_INST):
        ev.append(("prefix", i, np.concatenate(stored[i]) if stored[i] else np.zeros((0, 16), np.uint8), None, None))
        ev.append(("fill", i, fill[owner == i], None, None))
    first = list(ev)
    ev.append(None)
    off1, off2 = [], []
    for tag, i, k, _, _ in first:
        sel = rng.random(k.shape[0]) < 0.2
        off1.append((tag, i, None, k[sel], None))                      # HBM -> DRAM
        sel2 = sel & (rng.random(k.shape[0]) < 0.5)
        off2.append((tag, i, None, k[sel2], None))                     # DRAM -> SSD
    return ev + off1 + [None] + off2 + [None]


def instance_view(rng):
    """(type, schedulable, waiting, usage) per instance: half prefill-side, half decode."""
    out = []
    for i in range(N_INST):
        t = 2 if i % 2 else int(rng.choice([0, 1, 3]))
        out.append((t, True, int(rng.integers(0, 32)), float(np.float32(rng.random() * 0.9))))
    return out


# ----------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu):
        self.gpu, self.rows, self.proc = gpu, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


DUMP_ROWS = 1024
DUMP_BYTES = 56 << 20


def dump_outputs(out_dir, d_ids, d_nids, d_st, d_keys, d_match, d_route):
    """Writes the results of the device-resident step — what xllm_ingest_batch would hand a caller: token ids, their
    count and status, block keys, match and routing — as float32 / float64 arrays (exact for every value stored) to
    out_dir/<name>.npy.  A fixed seeded sample of rows (rows.npy) keeps the files under 64 MB, so two builds run
    with the same arguments can be compared output for output."""
    import torch
    from xllm_service_b200 import _lib
    n, T = d_ids.shape
    nb = d_keys.shape[1]
    row_bytes = 8 * T + 4 * 16 * nb + 4 * 4 * 64 + 8 * 10
    rows = np.sort(np.random.default_rng(0).choice(n, size=min(n, DUMP_ROWS, DUMP_BYTES // row_bytes), replace=False))
    idx = torch.from_numpy(rows).to(d_ids.device)
    take = lambda t: t.index_select(0, idx).cpu().numpy()  # noqa: E731
    match = take(d_match).view(_lib.MATCH_DTYPE)[:, 0]
    route = take(d_route).view(_lib.ROUTING_DTYPE)[:, 0]
    inst = match["instances"][:, None] >> np.arange(64, dtype=np.uint64) & np.uint64(1)
    out = {"rows": rows.astype(np.float64), "ids": take(d_ids).astype(np.float64),
           "n_ids": take(d_nids).astype(np.float64), "status": take(d_st).astype(np.float64),
           "keys": take(d_keys).astype(np.float32),
           "match_max_block_num": match["max_block_num"].astype(np.float64),
           "match_max_matched_block_num": match["max_matched_block_num"].astype(np.float64),
           "match_instances": inst.astype(np.float32)}
    for f in ("hbm", "dram", "ssd"):
        out["match_" + f] = match[f].astype(np.float32)
    for f in ("prefill_id", "decode_id", "ok", "prefill_score", "decode_score"):
        out["routing_" + f] = route[f].astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def traffic_from_profiles(kernel):
    """dram bytes per launch of `kernel` from the committed ncu capture of this command, or None."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f).get(kernel)
    return None


# ----------------------------------------------------------------------------------------------
def run_c5(h, wcnt, n_req, steps, rank_seed=0):
    """BASELINE config 5 (EPD multimodal mix; synthetic, no reference semantics — SURVEY.md §8d C5): requests of
    log-uniform 64-8192 tokens, 30 % with 1-4 spans of 256-1024 ready-made image-placeholder ids between their text
    pieces (the spans bypass BPE but are hashed and matched), 70:30 online / offline.  Measured end to end through
    xllm_ingest_batch_segments with page-locked host buffers: the online requests go first, the offline ones are
    batch-deferred behind them.  Returns the dict that becomes the bench line's "c5" key."""
    from oracle import oracle as o
    from xllm_service_b200 import HostBuffer, workload
    T, nbk = 8192, 8192 // BLOCK
    b = workload.make_c5_batch(n_req, wcnt, seed=555 + rank_seed,
                               shared_prefix=dict(n_prefixes=256, frac=0.5, min_blocks=1, max_blocks=8,
                                                  block_tokens=BLOCK))
    parts = {"online": b.select(np.nonzero(~b.offline)[0]), "offline": b.select(np.nonzero(b.offline)[0])}

    def pin(arr):
        hb = HostBuffer(arr.shape, arr.dtype)
        hb.array[...] = arr
        return hb

    bufs = {}
    for name, sb in parts.items():
        n = sb.n
        bufs[name] = dict(text=pin(sb.text), off=pin(sb.offsets), rss=pin(sb.req_seg_start), sl=pin(sb.seg_len),
                          span=pin(sb.span_ids if sb.span_ids.size else np.zeros(1, np.int32)),
                          ids=HostBuffer((n, T), np.int32), nids=HostBuffer((n,), np.int32),
                          st=HostBuffer((n,), np.int32), keys=HostBuffer((n, nbk, 16), np.uint8),
                          match=HostBuffer((n, 400), np.uint8), route=HostBuffer((n, 20), np.uint8))

    def call(name, with_match=True):
        sb, B = parts[name], bufs[name]
        h.ingest_batch_segments_ptrs(sb.n, B["text"].ptr, B["off"].ptr, B["ids"].ptr, T, B["nids"].ptr, B["st"].ptr,
                                     sb.seg_len.size, B["rss"].ptr, B["sl"].ptr, B["span"].ptr if sb.span_ids.size else 0,
                                     sb.span_ids.size, B["keys"].ptr, nbk, B["match"].ptr if with_match else 0,
                                     B["route"].ptr if with_match else 0)

    # first pass: ids + keys; every request must come out at exactly the length the generator promised
    for name in parts:
        call(name, with_match=False)
        assert (bufs[name]["st"].array == 0).all() and (bufs[name]["nids"].array == parts[name].n_tokens).all()
    # the shared prefixes of this workload enter the index (instance = prefix id mod 64), then one publish
    on = parts["online"]
    seen = {}
    pid = b.prefix_id[np.nonzero(~b.offline)[0]]
    ptk = b.prefix_tokens[np.nonzero(~b.offline)[0]]
    for r in range(on.n):
        j = int(pid[r])
        if j >= 0 and j not in seen:
            seen[j] = bufs["online"]["keys"].array[r, :ptk[r] // BLOCK].copy()
            h.index_apply(j % N_INST, seen[j])
    h.index_publish()
    # parity gate on a sample: ids = per-piece oracle encodes + spans appended; keys = the oracle's hash chain
    sp = o.SentencePieceOracle(MODEL_DIR)
    piece_of_seg = np.cumsum(on.seg_len < 0) - (on.seg_len < 0)
    span_of_seg = np.cumsum(np.maximum(on.seg_len, 0)) - np.maximum(on.seg_len, 0)
    n_chk = min(24, on.n)
    for r in range(n_chk):
        want = []
        for sg in range(on.req_seg_start[r], on.req_seg_start[r + 1]):
            ln = int(on.seg_len[sg])
            if ln < 0:
                p = piece_of_seg[sg]
                want.extend(sp.encode(on.text[on.offsets[p]:on.offsets[p + 1]].tobytes()).tolist())
            else:
                want.extend(on.span_ids[span_of_seg[sg]:span_of_seg[sg] + ln].tolist())
        want = np.asarray(want, np.int32)
        assert (bufs["online"]["ids"].array[r, :want.size] == want).all(), "c5: token ids differ from the oracle"
        wk = o.block_hash_chain(want, BLOCK, SEED)
        assert (bufs["online"]["keys"].array[r, :wk.shape[0]] == wk).all(), "c5: block keys differ from the oracle"
    # timed: online batch, then the deferred offline batch
    import torch
    for name in parts:
        call(name)
    torch.cuda.synchronize()
    t_on = t_all = 0.0
    for _ in range(steps):
        w0 = time.perf_counter()
        call("online")
        w1 = time.perf_counter()
        call("offline")
        w2 = time.perf_counter()
        t_on += w1 - w0
        t_all += w2 - w0
    from xllm_service_b200 import _lib
    mt = bufs["online"]["match"].array.view(_lib.MATCH_DTYPE)[:, 0]
    # the persistent grid's tail: per-warp busy time of the tokenizer over this batch's text pieces
    _, st, warp_ns = h.encode_batch_profile(b.text, b.offsets, 0)
    warp_ms = warp_ns.astype(np.float64) / 1e6
    tokens = int(b.n_tokens.sum())
    return {
        "workload": "c5: %d requests, log-uniform %d-%d tokens (mean %.0f), %.0f%% with 1-4 spans of 256-1024 "
                    "placeholder ids (%d text pieces + %d id spans, %.0f%% of all tokens pre-tokenised), "
                    "%d online + %d offline (offline batch-deferred behind online)"
                    % (b.n, int(b.n_tokens.min()), int(b.n_tokens.max()), b.n_tokens.mean(),
                       100.0 * np.mean([(b.seg_len[b.req_seg_start[r]:b.req_seg_start[r + 1]] >= 0).any()
                                        for r in range(b.n)]),
                       int((b.seg_len < 0).sum()), int((b.seg_len >= 0).sum()), 100.0 * b.span_ids.size / tokens,
                       parts["online"].n, parts["offline"].n),
        "api": "xllm_ingest_batch_segments (C-ABI, page-locked host buffers, ids rows of 8192)",
        "e2e_req_per_s": b.n * steps / t_all, "e2e_tokens_per_s": tokens * steps / t_all,
        "ms_per_step": t_all / steps * 1e3, "online_batch_ms": t_on / steps * 1e3,
        "offline_batch_ms": (t_all - t_on) / steps * 1e3,
        "text_bytes": int(b.text.size),
        "parity_gate": {"checked": n_chk, "ids": "bit-exact", "keys": "bit-exact",
                        "lengths": "all %d requests encode to exactly the generated length" % b.n},
        "mean_matched_blocks_online": float(mt["max_matched_block_num"].mean()),
        "persistent_grid_tail": {"warps": int(warp_ms.size), "max_ms": float(warp_ms.max()),
                                 "mean_ms": float(warp_ms.mean()), "max_over_mean": float(warp_ms.max() / warp_ms.mean()),
                                 "note": "busy time per warp slot of the tokenizer kernels (sp_express_kernel + what it hands to sp_encode_kernel) over all text pieces of the batch "
                                         "(one warp takes one piece at a time from a shared counter)"},
    }


def service_latency(batch, n_prompts=256, seconds=2.5):
    """p50 / p99 of one request through the micro-batcher at the reference's concurrency (32 worker threads and 128
    concurrent requests, global_gflags.cpp:32-36): tests/cpp/latency_main.cc, compiled here with g++ against the
    C-ABI, one 4 K-token prompt per submit, token ids + routing back.  Returns a list of result dicts (or an error)."""
    import struct
    import tempfile
    import xllm_service_b200 as x
    tmp = tempfile.mkdtemp(prefix="xllm_lat_")
    exe = os.path.join(tmp, "latency_main")
    pf = os.path.join(tmp, "prompts.bin")
    libdir = os.path.dirname(x.lib_path())
    try:
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-pthread", "-I", os.path.join(ROOT, "include"), "-I",
                               os.path.join(ROOT, "xllm_service_b200", "host"),
                               os.path.join(ROOT, "tests", "cpp", "latency_main.cc"), "-o", exe, "-L", libdir,
                               "-lxllm_ingest", "-Wl,-rpath," + libdir, "-Wl,--allow-shlib-undefined"],
                              stderr=subprocess.DEVNULL)
        with open(pf, "wb") as f:
            for i in range(min(n_prompts, batch.n)):
                t = batch.prompt(i)
                f.write(struct.pack("<I", len(t)) + t)
        out = []
        for threads, max_batch, wait_us in ((1, 1, 0), (32, 32, 50), (128, 128, 50)):
            p = subprocess.run([exe, MODEL_DIR, pf, str(threads), str(seconds), str(max_batch), str(wait_us)],
                               capture_output=True, text=True, timeout=120)
            if p.returncode != 0:
                return {"error": "latency_main rc %d: %s" % (p.returncode, p.stderr[-300:])}
            out.append(json.loads(p.stdout.strip().split("\n")[-1]))
        return out
    except (OSError, subprocess.SubprocessError, ValueError) as e:
        return {"error": repr(e)[:300]}


def honest_text(local, headline_batch, iters=3, corpus_bytes=256 << 20):
    """The tokenizer kernel away from the headline's comfort zone (VERDICT r1 weak #6), device-resident, CUDA events:
      natural_sp32k   real text (this image's site-packages sources and docs, workload.natural_corpus) cut into 16 KB
                      prompts, SentencePiece BPE 32 000 trained on that kind of text, word memo on
      natural_hf128k  the same prompts through an HF byte-level BPE with 128 471 entries: ids beyond 16 bits, i.e. the
                      non-SMALL kernel variants (12-byte pair state, 4-id memo payload)
      headline_memo_off  the headline workload with the word memo disabled (XLLM_SP_MEMO_SLOTS=0)
    Each with a bit-exact gate of 24 prompts against the CPU oracle."""
    import torch
    import xllm_service_b200 as x
    from oracle import oracle as o
    from xllm_service_b200 import workload
    dev = torch.device("cuda", local)
    t0 = time.time()
    corpus = workload.natural_corpus(corpus_bytes)
    pb = workload.cut_prompts(corpus, 16384)
    words = corpus[: 32 << 20].split()
    out = {"corpus": {"bytes": len(corpus), "prompts": pb.n, "read_s": round(time.time() - t0, 1),
                      "what": "*.py/*.md/*.rst/*.txt/*.h/*.hpp of site-packages in path order, UTF-8 files only "
                              "(all there is in the image: no repetition, so less than 1 GB)",
                      "distinct_whitespace_words_ratio_first_32MB": round(len(set(words)) / max(1, len(words)), 4)}}
    stream = torch.cuda.current_stream()

    def timed(h, text_np, off_np, stride, check_encode, n_check=24):
        n = off_np.size - 1
        d_text = torch.from_numpy(text_np).to(dev)
        d_off = torch.from_numpy(off_np).to(dev)
        d_ids = torch.empty((n, stride), dtype=torch.int32, device=dev)
        d_n = torch.empty((n,), dtype=torch.int32, device=dev)
        d_st = torch.empty((n,), dtype=torch.int32, device=dev)
        run = lambda: h.encode_batch_device(n, d_text.data_ptr(), d_off.data_ptr(), d_ids.data_ptr(), stride,  # noqa: E731
                                            d_n.data_ptr(), d_st.data_ptr(), stream.cuda_stream or None)
        run()
        torch.cuda.synchronize()
        st = d_st.cpu().numpy()
        nid = d_n.cpu().numpy()
        assert (st == 0).all(), np.unique(st)
        ids = d_ids[:n_check].cpu().numpy()
        for r in range(min(n_check, n)):
            want = check_encode(text_np[off_np[r]:off_np[r + 1]].tobytes())
            assert ids[r, :nid[r]].tolist() == want, "honest_text: ids differ from the oracle"
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(iters):
            run()
        e1.record(stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / iters
        tokens = int(nid.sum())
        return {"prompts": int(n), "text_bytes": int(text_np.size), "tokens": tokens, "ms": round(ms, 3),
                "prompts_per_s": round(n / ms * 1e3), "MB_per_s": round(text_np.size / ms / 1e3),
                "tokens_per_s": round(tokens / ms * 1e3), "bytes_per_token": round(text_np.size / max(1, tokens), 2),
                "algo_GBps": round((text_np.size + 4 * tokens) / ms / 1e6, 1), "oracle_gate": "bit-exact on 24 prompts"}

    d_sp = os.path.join(ROOT, "tests", "golden", "sp_natural_32k")
    d_hf = os.path.join(ROOT, "tests", "golden", "hf_natural_128k")
    h1 = x.Ingest(tokenizer_path=d_sp, device=local)
    S = o.SentencePieceOracle(d_sp)
    out["natural_sp32k"] = timed(h1, pb.text, pb.offsets, 16384, lambda t: S.encode(t).tolist())
    out["natural_sp32k"]["tokenizer"] = "SentencePiece BPE 32000 (byte fallback, nmt_nfkc), memo on"
    h1.close()
    os.environ["XLLM_SP_WARM"] = "1"
    try:
        h1w = x.Ingest(tokenizer_path=d_sp, device=local)
        h2w = x.Ingest(tokenizer_path=d_hf, device=local)
    finally:
        del os.environ["XLLM_SP_WARM"]
    H = o.HfBpeOracle(d_hf)
    out["natural_sp32k_warm"] = timed(h1w, pb.text, pb.offsets, 16384, lambda t: S.encode(t).tolist())
    out["natural_sp32k_warm"]["tokenizer"] = ("the same, through the opt-in warm-up kernels (XLLM_SP_WARM=1: memo misses "
                                              "merged ahead in full rounds, long words resolved ahead of the rounds)")
    h1w.close()
    out["natural_hf128k_warm"] = timed(h2w, pb.text, pb.offsets, 16384,
                                       lambda t: H.prefix_ids + H.encode(t).tolist() + H.suffix_ids)
    out["natural_hf128k_warm"]["tokenizer"] = "HF byte-level BPE 128471 entries through the warm-up kernels"
    h2w.close()
    h2 = x.Ingest(tokenizer_path=d_hf, device=local)
    out["natural_hf128k"] = timed(h2, pb.text, pb.offsets, 16384,
                                  lambda t: H.prefix_ids + H.encode(t).tolist() + H.suffix_ids)
    out["natural_hf128k"]["tokenizer"] = ("HF byte-level BPE, GPT-2 regex, 128471 entries (non-SMALL kernels: ids "
                                          "beyond 16 bits), memo on")
    h2.close()
    os.environ["XLLM_SP_MEMO_SLOTS"] = "0"
    try:
        h3 = x.Ingest(tokenizer_path=MODEL_DIR, device=local)
    finally:
        del os.environ["XLLM_SP_MEMO_SLOTS"]
    S8 = o.SentencePieceOracle(MODEL_DIR)
    n3 = min(headline_batch.n, 16384)
    off3 = headline_batch.offsets[: n3 + 1]
    out["headline_memo_off"] = timed(h3, headline_batch.text[: off3[-1]], off3, 4096 + 64,
                                     lambda t: S8.encode(t).tolist())
    out["headline_memo_off"]["tokenizer"] = "the headline's SentencePiece BPE 8000 and prompts, word memo disabled"
    h3.close()
    # the two backends rows a2 / a3 count on parity only: SentencePiece Unigram (Viterbi per word from a running
    # score, no memo) and tiktoken as the service runs it (no regex: the whole prompt is one piece -> long-word path)
    d_uni = os.path.join(ROOT, "tests", "golden", "sp_unigram_4k_bf")
    h4 = x.Ingest(tokenizer_path=d_uni, device=local)
    SU = o.SentencePieceOracle(d_uni)
    n4 = min(headline_batch.n, 4096)
    off4 = headline_batch.offsets[: n4 + 1]
    out["unigram_4k_headline_text"] = timed(h4, headline_batch.text[: off4[-1]], off4, 8192,
                                            lambda t: SU.encode(t).tolist(), n_check=8)
    out["unigram_4k_headline_text"]["tokenizer"] = "SentencePiece Unigram 4000 (byte fallback) on the headline prompts"
    h4.close()
    d_tik = os.path.join(ROOT, "tests", "golden", "tiktoken_1k")
    h5 = x.Ingest(tokenizer_path=d_tik, device=local)
    TK = o.TiktokenOracle(d_tik)
    n5 = min(headline_batch.n, 256)
    off5 = headline_batch.offsets[: n5 + 1]
    out["tiktoken_1k_regexless"] = timed(h5, headline_batch.text[: off5[-1]], off5, 20480,
                                         lambda t: TK.encode(t).tolist(), n_check=2)
    out["tiktoken_1k_regexless"]["tokenizer"] = ("tiktoken 1453 ranks, regex-less as the service configures it: every "
                                                 "16 KB prompt is ONE piece (tiktoken_tokenizer.cpp:238-241)")
    h5.close()
    return out


def cpu_reference_pass(sp, P, batch, n_sample, threads):
    """One bounded pass of the reference's per-request path (encode + select_instances_pair) on the host."""
    from oracle import oracle as o
    off = batch.offsets[:n_sample + 1]
    t0 = time.perf_counter()
    res = o.ingest_batch(sp, P, batch.text, off, 4096 + 64, n_threads=threads, want_ids=False)
    dt = time.perf_counter() - t0
    return n_sample / dt, dt, res


def build_cpu_side(names, events, view, with_fill=True):
    from oracle import oracle as o
    sp = o.SentencePieceOracle(MODEL_DIR)
    P = o.PrefixOracle(names, BLOCK, SEED)
    for i, (t, s, w, u) in enumerate(view):
        P.set_instance(names[i], t, s)
        P.set_load(names[i], w, u)
    for e in events:
        if e is None:
            P.upload()
        elif with_fill or e[0] == "prefix":
            _, i, st, of, rm = e
            P.record(names[i], st if st is not None else (), of if of is not None else (),
                     rm if rm is not None else ())
    return sp, P


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path (the oracle port; the
    reference cannot be compiled here — all its third-party submodules are absent, DESIGN.md) on the
    host cores, same metric / config, bounded sample per step.  Rank 0 only."""
    if rank != 0:
        return
    from oracle import oracle as o
    from xllm_service_b200 import workload
    o.build()
    threads, thread_detail = host_threads()
    rng = np.random.default_rng(2026)
    names = ["instance-%02d" % i for i in range(N_INST)]
    vocab = workload.make_vocabulary()
    sp0 = o.SentencePieceOracle(MODEL_DIR)
    wcnt = word_token_counts_cpu(sp0, vocab, threads)
    n_sample = args.cpu_sample or max(256, min(args.requests, threads * 24))
    batch, meta = make_batch(n_sample, args.tokens, wcnt, seed=1000, device="cpu")
    # index content from the prompts' own prefixes (CPU hash chain) + filler keys
    ids, _ = sp0.encode_batch(batch.text, batch.offsets, args.tokens, n_threads=threads)
    pref = {}
    for r in range(n_sample):
        j = int(meta["prefix_id"][r])
        if j >= 0 and j not in pref:
            pref[j] = o.block_hash_chain(ids[r, :meta["prefix_blocks"][r] * BLOCK], BLOCK, SEED)
    events = index_events(list(pref.values()), args.index_keys, rng)
    view = instance_view(rng)
    sp, P = build_cpu_side(names, events, view)
    for _ in range(max(1, min(args.warmup, 1))):
        cpu_reference_pass(sp, P, batch, min(n_sample, threads * 2), threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_reference_pass(sp, P, batch, n_sample, threads)
    dt = time.perf_counter() - t0
    v = n_sample * args.steps / dt
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "req/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": {"workload": "c2+c3: %d-token prompts, SentencePiece-BPE 8k, 1Mi-key prefix index, 64 instances"
                                   % args.tokens, "sample_prompts_per_step": n_sample},
            "cpu_baseline": {"value": v, "unit": "req/s", "cores": threads, "kind": "port", "host": thread_detail,
                             "sample": "%d prompts x %d tokens per step, %d threads, one request per thread at a time"
                                       % (n_sample, args.tokens, threads),
                             "note": "tokenizer = the CPU port (libsentencepiece is not in the image); the port's "
                                     "hash / match / routing are pinned to the reference's own code compiled "
                                     "unmodified (oracle/_ref, tests/test_ref_parity.py)"},
            "e2e": {"value": v, "unit": "req/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------
def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import xllm_service_b200 as x
    from xllm_service_b200 import HostBuffer, _lib, workload

    if not os.path.exists(x.lib_path()):
        import __graft_entry__ as ge
        ge.build()
    torch.cuda.set_device(local)
    if world > 1:
        # keep stdout to the one JSON line: at NCCL_DEBUG=VERSION (set on the GPU boxes) NCCL prints its version
        # banner on stdout, NCCL_DEBUG_FILE does not move it; VERSION has no other effect, so drop it
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            del os.environ["NCCL_DEBUG"]
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)

    n, T = args.requests, args.tokens
    nb = T // BLOCK
    # BASELINE config 4: at N > 1 the index is N x the single-GPU one and hash-range-sharded over the N GPUs (one NCCL
    # all-to-all of (hash, request, block) tuples per batch and one of tier masks back, csrc/shard_exchange.cu); a
    # replicated twin of the whole index on every GPU serves the "sharded == replicated == oracle" gate only.
    sharded_mode = world > 1 and args.index != "replicated"
    total_keys = args.index_keys * (world if sharded_mode else 1)
    h_full = None
    if sharded_mode:
        from xllm_service_b200 import sharded
        h = sharded.create_sharded(tokenizer_path=MODEL_DIR, block_size=BLOCK, xxh3_seed=SEED, device=local,
                                   index_capacity=total_keys // world * 5 // 4 + (1 << 16), max_batch=n, max_tokens=T)
        h_full = x.Ingest(block_size=BLOCK, xxh3_seed=SEED, device=local, index_capacity=total_keys + (1 << 16))
    else:
        h = x.Ingest(tokenizer_path=MODEL_DIR, block_size=BLOCK, xxh3_seed=SEED, device=local,
                     index_capacity=args.index_keys + (1 << 16))
    if args.chunk_requests:
        h.set_pipeline(args.chunk_requests, 1 << 40)
    vocab = workload.make_vocabulary()
    wcnt = word_token_counts_gpu(h, vocab)
    t_gen = time.time()
    batch, meta = make_batch(n, T, wcnt, seed=1000 + rank, device=str(dev))
    t_gen = time.time() - t_gen
    text_bytes = int(batch.text.size)

    # ---- page-locked host buffers (the e2e call's inputs / outputs)
    # xllm_host_alloc: page-locked AND on the GPU's NUMA node (the box has two sockets)
    class Pinned:
        def __init__(self, shape, dtype):
            self.buf = HostBuffer(shape, torch.empty(0, dtype=dtype).numpy().dtype)

        def numpy(self):
            return self.buf.array

        def data_ptr(self):
            return self.buf.ptr

    def pinned(shape, dtype):
        return Pinned(shape, dtype)

    h_text = pinned((text_bytes,), torch.uint8)
    h_text.numpy()[:] = batch.text
    h_off = pinned((n + 1,), torch.int64)
    h_off.numpy()[:] = batch.offsets
    h_ids = pinned((n, T), torch.int32)
    h_nids = pinned((n,), torch.int32)
    h_st = pinned((n,), torch.int32)
    h_keys = pinned((n, nb, 16), torch.uint8)
    h_match = pinned((n, 400), torch.uint8)
    h_route = pinned((n, 20), torch.uint8)

    def e2e_step(with_match=True):
        h.ingest_batch_ptrs(n, h_text.data_ptr(), h_off.data_ptr(), h_ids.data_ptr(), T, h_nids.data_ptr(),
                            h_st.data_ptr(), h_keys.data_ptr(), nb, h_match.data_ptr() if with_match else 0,
                            h_route.data_ptr() if with_match else 0)

    # ---- first pass without match: token ids + block keys, used to build the index content
    rng = np.random.default_rng(2026)
    names = ["instance-%02d" % i for i in range(N_INST)]
    e2e_step(with_match=False)
    assert (h_st.numpy() == 0).all() and (h_nids.numpy() == T).all(), "workload must encode to exactly T tokens"
    keys_np = h_keys.numpy()
    pref = {}
    pid = meta["prefix_id"]
    first = np.unique(pid[pid >= 0], return_index=True)
    rows_with = np.nonzero(pid >= 0)[0]
    for j, idx in zip(*first):
        r = rows_with[idx]
        pref[int(j)] = keys_np[r, :meta["prefix_blocks"][r]].copy()
    prefix_list = [pref[j] for j in sorted(pref)]
    if sharded_mode:   # one global event stream: every rank's shared prefixes, in rank order (identical on all ranks)
        box = [None] * world
        dist.all_gather_object(box, prefix_list)
        prefix_list = [p for part in box for p in part]
    events = index_events(prefix_list, total_keys, rng)
    view = instance_view(rng)
    handles = [h] + ([h_full] if h_full is not None else [])
    for hh in handles:
        for i, (t, s, w, u) in enumerate(view):
            hh.set_instance(i, t, s)
            hh.set_load_metrics(i, w, u)
        for e in events:          # every rank is given every event; a sharded handle keeps the keys it owns
            if e is None:
                hh.index_publish()
            else:
                hh.index_apply(e[1], e[2], e[3], e[4])
    index_size = h.index_size()
    if sharded_mode:
        t_sz = torch.tensor([index_size], dtype=torch.int64, device=dev)
        dist.all_reduce(t_sz)
        assert int(t_sz.item()) == h_full.index_size(), "the shards do not add up to the replicated index"
        index_size = int(t_sz.item())

    # ---- parity gate, part 1 (every rank, whole batch): the sharded index answers exactly like a replicated one
    shard_gate = None
    if sharded_mode:
        e2e_step(with_match=True)                                   # collective
        d_k = torch.from_numpy(h_keys.numpy().reshape(-1, 16)).to(dev)
        d_ks0 = torch.arange(n, device=dev, dtype=torch.int64) * nb
        d_nb0 = torch.full((n,), nb, dtype=torch.int32, device=dev)
        d_m0 = torch.empty((n, 400), dtype=torch.uint8, device=dev)
        d_r0 = torch.empty((n, 20), dtype=torch.uint8, device=dev)
        h_full.match_route_device(n, d_k.data_ptr(), n * nb, d_ks0.data_ptr(), d_nb0.data_ptr(), d_m0.data_ptr(),
                                  d_r0.data_ptr(), None)
        torch.cuda.synchronize()
        same = (torch.equal(d_m0.cpu(), torch.from_numpy(h_match.numpy())) and
                torch.equal(d_r0.cpu(), torch.from_numpy(h_route.numpy())))
        t_ok = torch.tensor([1 if same else 0], dtype=torch.int64, device=dev)
        dist.all_reduce(t_ok, op=dist.ReduceOp.MIN)
        assert int(t_ok.item()) == 1, "sharded match / routing differs from the replicated index"
        shard_gate = "sharded == replicated on all %d requests of every rank (match + routing, bit for bit)" % n
        del d_k, d_m0, d_r0
        h_full.close()
        h_full = None
        torch.cuda.empty_cache()
    # ---- parity gate, part 2 (rank 0): a sample of the batch against the CPU oracle, bit for bit
    gate = {"checked": 0}
    if rank == 0:
        from oracle import oracle as o
        o.build()
        threads, thread_detail = host_threads()
        # the oracle of the sharded run holds the prefix entries only (filler keys are disjoint and never looked up):
        # N x 1 Mi string-set entries would take minutes and gigabytes on the host
        sp, P = build_cpu_side(names, events, view, with_fill=not sharded_mode)
        if not sharded_mode:
            e2e_step(with_match=True)
        n_chk = min(n, 64)
        res = o.ingest_batch(sp, P, batch.text, batch.offsets[:n_chk + 1], T, n_threads=threads)
        assert (res["ids"] == h_ids.numpy()[:n_chk]).all(), "token ids differ from the CPU oracle"
        want_keys, _ = o.block_hash_chain_batch(res["ids"].reshape(-1), np.arange(n_chk + 1, dtype=np.int64) * T,
                                                BLOCK, SEED)
        assert (want_keys.reshape(n_chk, nb, 16) == keys_np[:n_chk]).all(), "block keys differ from the CPU oracle"
        routing = h_route.numpy().view(_lib.ROUTING_DTYPE)[:, 0]
        match = h_match.numpy().view(_lib.MATCH_DTYPE)[:, 0]
        for r in range(n_chk):
            m = P.match(res["ids"][r])
            assert match["max_matched_block_num"][r] == m["max_matched_block_num"]
            assert (match["hbm"][r] == m["hbm"]).all()
            ro = P.route(res["ids"][r])
            assert bool(routing["ok"][r]) == ro["ok"] and routing["prefill_score"][r] == np.float32(ro["prefill_score"])
            assert (ro["prefill_argmax"] >> int(routing["prefill_id"][r])) & 1
        gate = {"checked": n_chk, "ids": "bit-exact", "keys": "bit-exact", "routing": "score-exact, choice in argmax set",
                "mean_matched_blocks": float(match["max_matched_block_num"].mean())}
        if shard_gate:
            gate["sharded"] = shard_gate

    # ---- device-resident buffers
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    d_text = torch.from_numpy(h_text.numpy()).to(dev)
    d_off = torch.from_numpy(h_off.numpy()).to(dev)
    d_ids = torch.empty((n, T), dtype=torch.int32, device=dev)
    d_nids = torch.empty((n,), dtype=torch.int32, device=dev)
    d_st = torch.empty((n,), dtype=torch.int32, device=dev)
    d_tok_start = torch.arange(n, device=dev, dtype=torch.int64) * T
    d_key_start = torch.arange(n, device=dev, dtype=torch.int64) * nb
    d_nblk = torch.full((n,), nb, dtype=torch.int32, device=dev)
    d_keys = torch.empty((n, nb, 16), dtype=torch.uint8, device=dev)
    d_match = torch.empty((n, 400), dtype=torch.uint8, device=dev)
    d_route = torch.empty((n, 20), dtype=torch.uint8, device=dev)
    sp_ = stream.cuda_stream
    torch.cuda.synchronize()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(args.steps)]

    def dev_step(e=None):
        if e:
            e[0].record(stream)
        h.encode_batch_device(n, d_text.data_ptr(), d_off.data_ptr(), d_ids.data_ptr(), T, d_nids.data_ptr(),
                              d_st.data_ptr(), sp_)
        if e:
            e[1].record(stream)
        h.hash_blocks_device(n, d_ids.data_ptr(), d_tok_start.data_ptr(), d_nids.data_ptr(), d_keys.data_ptr(),
                             d_key_start.data_ptr(), sp_)
        if e:
            e[2].record(stream)
        h.match_route_device(n, d_keys.data_ptr(), n * nb, d_key_start.data_ptr(), d_nblk.data_ptr(),
                             d_match.data_ptr(), d_route.data_ptr(), sp_)
        if e:
            e[3].record(stream)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for _ in range(args.warmup):
        dev_step()
    barrier()
    clocks = ClockSampler(local)
    clocks.start()
    t0 = torch.cuda.Event(enable_timing=True)
    t1 = torch.cuda.Event(enable_timing=True)
    t0.record(stream)
    for k in range(args.steps):
        dev_step(ev[k])
    t1.record(stream)
    barrier()
    dev_ms = max_over_ranks(t0.elapsed_time(t1))
    k_ms = np.array([[e[i].elapsed_time(e[i + 1]) for i in range(3)] for e in ev]).mean(axis=0)
    assert (torch.equal(d_ids.cpu(), torch.from_numpy(h_ids.numpy())) and
            torch.equal(d_keys.cpu(), torch.from_numpy(h_keys.numpy()))), "device-resident != e2e results"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, d_ids, d_nids, d_st, d_keys, d_match, d_route)

    shard_stats = h.shard_last_stats() if sharded_mode else None   # the last device-resident step's round

    # ---- the box's copy floor for this step's bytes: the same page-locked buffers, H2D and D2H at once on two
    # streams, every rank at the same time, nothing else running — what the e2e step cannot beat
    h2d_bytes = text_bytes + 8 * (n + 1)
    d2h_bytes = 4 * n * T + 8 * n + 16 * n * nb + 420 * n
    cp_in, cp_out = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    d_sink = torch.empty(text_bytes, dtype=torch.uint8, device=dev)
    import ctypes

    def bare_copies():
        rt = ctypes.CDLL("libcudart.so.12")     # the runtime libxllm_ingest.so already brought into the process
        rt.cudaMemcpyAsync.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p]
        cp = lambda dst, src, nbytes, kind, st: rt.cudaMemcpyAsync(dst, src, nbytes, kind, st.cuda_stream)  # noqa: E731
        rc = cp(d_sink.data_ptr(), h_text.data_ptr(), text_bytes, 1, cp_in)
        rc |= cp(h_ids.data_ptr(), d_ids.data_ptr(), 4 * n * T, 2, cp_out)
        rc |= cp(h_keys.data_ptr(), d_keys.data_ptr(), 16 * n * nb, 2, cp_out)
        rc |= cp(h_match.data_ptr(), d_match.data_ptr(), 400 * n, 2, cp_out)
        if rc:
            raise RuntimeError("cudaMemcpyAsync failed")

    floor_ms = None
    try:
        bare_copies()
        barrier()
        w0 = time.perf_counter()
        for _ in range(3):
            bare_copies()
        torch.cuda.synchronize()
        floor_ms = max_over_ranks(time.perf_counter() - w0) / 3 * 1e3
    except Exception:   # noqa: BLE001  (cudart binding differences: the floor is informative only)
        floor_ms = None
    del d_sink
    barrier()

    # ---- end to end through the C-ABI with host buffers
    for _ in range(max(1, min(args.warmup, 2))):
        e2e_step()
    barrier()
    w0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - w0)
    barrier()
    # the same end-to-end step with the opt-in narrow id download (xllm_ingest_io::ids_u16: uint16 ids for this
    # 8 000-piece vocabulary, what host/ingest_batcher.h takes and widens while it hands results out)
    h_ids16 = pinned((n, T), torch.int16)

    def e2e_step_u16():
        h.ingest_batch_ptrs(n, h_text.data_ptr(), h_off.data_ptr(), 0, T, h_nids.data_ptr(), h_st.data_ptr(),
                            h_keys.data_ptr(), nb, h_match.data_ptr(), h_route.data_ptr(), ids_u16=h_ids16.data_ptr())

    e2e_step_u16()
    assert (h_ids16.numpy().view(np.uint16) == h_ids.numpy()).all(), "uint16 ids differ from the int32 ids"
    barrier()
    w0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step_u16()
    torch.cuda.synchronize()
    e2e16_s = max_over_ranks(time.perf_counter() - w0)
    barrier()
    clk = clocks.stop()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = peaks()
    enc_bytes = text_bytes + 4 * n * T
    hash_bytes = n * nb * 528
    match_bytes = n * nb * 82
    kernels = {
        "sp_encode": {"ms": float(k_ms[0]), "algo_bytes": enc_bytes, "GBps": enc_bytes / k_ms[0] / 1e6},
        "xxh3_chain128": {"ms": float(k_ms[1]), "algo_bytes": hash_bytes, "GBps": hash_bytes / k_ms[1] / 1e6},
        ("shard_round(bucket+a2a+probe+a2a+scan)" if sharded_mode else "match_route(probe+scan+route)"):
            {"ms": float(k_ms[2]), "algo_bytes": match_bytes, "GBps": match_bytes / k_ms[2] / 1e6},
    }
    for k in kernels.values():
        k["frac"] = k["GBps"] / peak
    dom = max(kernels, key=lambda k: kernels[k]["ms"])
    roofline = {"kernel": dom, "bound": "hbm", "achieved": kernels[dom]["GBps"], "peak": peak, "unit": "GB/s",
                "frac": kernels[dom]["frac"], "traffic": traffic_from_profiles(dom), "peak_source": peak_src,
                "share_of_step": float(k_ms[list(kernels).index(dom)] / k_ms.sum()),
                "note": "achieved = (text bytes + 4 B/token) / CUDA-event time of the encode launches (memo clear + "
                        "sp_express_kernel + the buffer-path and long-word kernels, empty grids on this workload); the "
                        "tokenizer is bound by instruction issue and L2 latency, not HBM (DESIGN.md 4.2)"}
    line = {
        "metric": METRIC, "value": world * n * args.steps / (dev_ms / 1e3), "unit": "req/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": "c2+c3: %d prompts x %d tokens per GPU, SentencePiece-BPE 8k (byte fallback), "
                               "block 128 seed 1024, %d-key prefix index over %d instances, 80%% shared-prefix "
                               "Zipf-0.9" % (n, T, index_size, N_INST),
                   "text_bytes_per_step": text_bytes,
                   "parallelism": ("dp%d requests + prefix index hash-range-sharded over %d GPUs (%d keys each): one "
                                   "NCCL all-to-all of 24-B (hash128, req, blk) tuples per batch and one of tier "
                                   "masks back" % (world, world, index_size // world)) if sharded_mode else
                                  ("dp%d (requests sharded, index replicated, no collective)" % world),
                   "l2": "inputs larger than L2 (%.2f GB text + %.2f GB ids per step): no flush" %
                         (text_bytes / 1e9, 4 * n * T / 1e9),
                   "parity_gate": gate, "generation_s": round(t_gen, 1)},
        "clocks": clk,
        "e2e": {"value": world * n * args.steps / e2e_s, "unit": "req/s", "ms_per_step": e2e_s / args.steps * 1e3,
                "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                "copy_floor_ms": floor_ms,
                "frac_of_copy_floor": (floor_ms / (e2e_s / args.steps * 1e3)) if floor_ms else None,
                "api": "xllm_ingest_batch (C-ABI, page-locked host buffers)"},
        "e2e_ids_u16": {"value": world * n * args.steps / e2e16_s, "unit": "req/s",
                        "ms_per_step": e2e16_s / args.steps * 1e3, "h2d_bytes_per_step": h2d_bytes,
                        "d2h_bytes_per_step": d2h_bytes - 2 * n * T,
                        "note": "same call with xllm_ingest_io::ids_u16 (opt-in; vocabulary < 65536): token ids come "
                                "back as uint16, checked equal to the int32 ids"},
        # value region: encode (express kernel + buffer-path kernel + long-word pass) + hash + match/route (sharded:
        # bucket, headers, owner probe, header gather, scan) per step; e2e region: the library's own count for one batch
        "gpu_launches": args.steps * ((10 if sharded_mode else 5) + h.last_batch_stats()[1]),
        "roofline": roofline,
        "kernels": kernels,
    }
    if shard_stats:
        line["shard_round_us"] = {k[:-3]: round(v * 1e3, 1) for k, v in shard_stats.items() if k.endswith("_ms")}
        line["shard_round_us"]["bucket_capacity"] = shard_stats["bucket_capacity"]
        line["shard_round_us"]["overflow_rounds"] = shard_stats["overflow_rounds"]
    if world == 1 and not args.no_honest_text:
        line["honest_text"] = honest_text(local, batch)
    if world == 1 and not args.no_latency:
        line["service_latency"] = {
            "what": "per-request submit latency through host/ingest_batcher.h (one 4K-token prompt per call, ids + "
                    "routing back) at the reference's concurrency; 1 thread = an idle service's single request",
            "runs": service_latency(batch)}
    if world == 1 and not args.no_c5:
        line["c5"] = run_c5(h, wcnt, args.c5_requests, max(2, min(args.steps, 5)))
    if world == 1 and not args.no_cpu_baseline:
        from oracle import oracle as o
        threads, thread_detail = host_threads()
        n_sample = args.cpu_sample or max(256, min(n, threads * 24))
        v, dt, res = cpu_reference_pass(sp, P, batch, n_sample, threads)
        rr = h_route.numpy().view(_lib.ROUTING_DTYPE)[:, 0]
        assert (res["n_ids"] == T).all() and (res["ok"] == rr["ok"][:n_sample]).all()
        line["cpu_baseline"] = {"value": v, "unit": "req/s", "cores": threads, "kind": "port", "host": thread_detail,
                                "sample": "%d of this step's prompts, %d threads, one request per thread at a time "
                                          "(encode + select_instances_pair), %.1f s" % (n_sample, threads, dt)}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
