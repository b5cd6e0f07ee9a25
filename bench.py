#!/usr/bin/env python3
"""bench.py -- the driver's measurement contract for the batched subword-encode path.

A "step" = one pass of the hot path (normalize -> unigram Viterbi / BPE merge -> ids) over one batch of
synthetic sentences.  The headline workload (N=1) is BASELINE.json configs[1]: 32k-vocab unigram model,
1,000,000 synthetic ~128-byte English sentences per GPU.

  value : whole-job sentences/s with inputs already resident in HBM (device-pointer C ABI), timed with CUDA
          events over exactly K steps, max over ranks.  With N > 1 the NCCL gather of the packed id buffers
          (ids + per-sentence counts) to rank 0 -- the path's only exchange -- is INSIDE the timed region: output
          buffers are double-buffered, the gather of step k overlaps the encode of step k+1, and the last gathers are
          waited for before the closing event.
  e2e   : the same metric through the host-buffer C ABI (spm_encode_ids): pinned host input, H2D + kernels +
          D2H of ids/offsets inside the timed region; `e2e_variants` adds pageable input and the C++ class
          (Encode(vector<string_view>, vector<vector<int>>*)).
  parity: the e2e output of the timed path, all sentences of rank 0's shard, compared with the unmodified
          reference's ids (oracle/_ref) -- "bit-exact" or the run fails; `ids_md5` is printed by both arms.
  roofline : algorithmic bytes / encode-kernel time vs the measured HBM peak.
  cpu_baseline : the reference's own Encode (oracle/_ref, all host threads) on rank 0's shard.

One JSON line is printed (rank 0).  By default it is the headline workload with the other BASELINE.json
configurations nested under "workloads" (configs[2] bpe32k_en, configs[3] bytefallback_mixed, configs[4]
sample_nbest64_en, and Decode(ids)) and, for N > 1, the strong-scaling run of the same 1M-sentence corpus under
"strong_scaling".  `--workload NAME` measures one workload alone; `--scaling strong` makes the strong-scaling
run the top-level line.  `--impl reference` times the unmodified reference on the host cores instead.
`--dump-outputs DIR` writes what the timed path of each measured workload returned in its last timed step (rank 0's
shard; a fixed, seeded sample of its sentences) as DIR/<workload>_<name>.npy, so that two builds can be compared
output for output on identical inputs.
"""
import argparse
import ctypes
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

WORKLOADS = {
    # name: (model, corpus kind, description)
    "unigram32k_en": ("uni32k", "en", "32k-vocab unigram Viterbi encode, synthetic ~128-byte English sentences"),
    "bpe32k_en": ("bpe32k", "en", "32k-vocab BPE merge encode, synthetic ~128-byte English sentences"),
    "bytefallback_mixed": ("mix_bf8k", "mixed", "byte-fallback unigram + NFKC on mixed CJK/emoji synthetic corpus"),
    "decode_unigram32k_en": ("uni32k", "en", "Decode(ids) -> text of the ids of the unigram32k_en workload (the step after the path)"),
    "sample_nbest64_en": ("uni32k", "en", "unigram SampleEncode nbest=64 alpha=0.5 (subword regularization lattice), "
                          "256k synthetic English sentences"),
}
HEADLINE = "unigram32k_en"
NESTED = ["bpe32k_en", "bytefallback_mixed", "sample_nbest64_en", "decode_unigram32k_en"]
ENCODE_WORKLOADS = ("unigram32k_en", "bpe32k_en", "bytefallback_mixed")
CORPUS_SEED = 20260922
# --dump-outputs: sentences kept per workload (a fixed, seeded sample; a 1M-sentence step returns ~120 MB of ids)
DUMP_SENTENCES = 16384
DUMP_SEED = 20261017
DUMP_LIMIT = 64 << 20
_dumped = [0]
DTYPE = "u8 text / int32 ids / f32+f64 scores"


def model_bytes(name):
    with open(os.path.join(ROOT, "tests", "golden", "models", name + ".model"), "rb") as f:
        return f.read()


def model_path(name):
    return os.path.join(ROOT, "tests", "golden", "models", name + ".model")


def make_config(workload, n_per_gpu, mean_bytes, ids_per_sentence):
    """The `config` object: identical in both arms (ours and --impl reference) for the same workload."""
    model, _, desc = WORKLOADS[workload]
    return {"workload": workload, "description": desc, "model": model + ".model",
            "sentences_per_gpu_per_step": int(n_per_gpu), "mean_bytes_per_sentence": round(float(mean_bytes), 4),
            "ids_per_sentence": round(float(ids_per_sentence), 4)}


def ids_md5(ids, ido):
    h = hashlib.md5()
    h.update(np.ascontiguousarray(ids, dtype=np.int32).tobytes())
    h.update(np.ascontiguousarray(ido, dtype=np.uint64).tobytes())
    return h.hexdigest()


def dump_lists(args, workload, name, values, offsets):
    """--dump-outputs: the lists values[offsets[i]:offsets[i+1]] of a fixed, seeded sample of the sentences, written as
    <workload>_<name>.npy (float32: ids and bytes are exact in it), their lengths as <workload>_<name>_lengths.npy and
    the sampled sentence indices as <workload>_sentences.npy (float64)."""
    offsets = np.asarray(offsets, dtype=np.int64)
    n = len(offsets) - 1
    pick = np.sort(np.random.default_rng(DUMP_SEED).choice(n, size=min(n, DUMP_SENTENCES), replace=False))
    lo, hi = offsets[pick], offsets[pick + 1]
    out = {f"{workload}_sentences": pick.astype(np.float64),
           f"{workload}_{name}_lengths": (hi - lo).astype(np.float32),
           f"{workload}_{name}": np.concatenate([np.zeros(0)] + [values[a:b] for a, b in zip(lo, hi)]).astype(np.float32)}
    _dumped[0] += sum(v.nbytes for v in out.values())
    if _dumped[0] > DUMP_LIMIT:
        raise SystemExit(f"bench.py: --dump-outputs would exceed {DUMP_LIMIT >> 20} MB")
    os.makedirs(args.dump_outputs, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(args.dump_outputs, k + ".npy"), v)


def load_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def load_traffic(workload, n):
    """dram bytes of the dominant kernel per launch from the newest committed ncu capture of this batch size."""
    best = None
    pdir = os.path.join(ROOT, "profiles")
    for name in sorted(os.listdir(pdir)) if os.path.isdir(pdir) else []:
        if name.endswith("_traffic.json"):
            try:
                t = json.load(open(os.path.join(pdir, name))).get(workload)
            except Exception:
                t = None
            if t and t.get("sentences") == n:
                best = dict(t, source="profiles/" + name)
    return best


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cgroup_cpu_limit():
    """CPU quota of this container in cores (cgroup v2 cpu.max / v1 cfs quota), or None when unlimited/unknown."""
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        return None if q == "max" else float(q) / float(p)
    except Exception:
        pass
    try:
        q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        p = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        return None if q <= 0 else q / p
    except Exception:
        return None


def reference_encode(mb, buf, offs, threads, repeats=2):
    """Unmodified reference (oracle/_ref) on the whole batch with `threads` std::threads: (ids, id_offsets, best s)."""
    from oracle import oracle_py
    rm = oracle_py.RefModel(mb)
    n = len(offs) - 1
    rm.encode_count(buf, offs[: min(n, 2000) + 1], threads)  # warm caches / thread creation
    best, out = None, None
    for _ in range(repeats):
        t0 = time.perf_counter()
        out = rm.encode_batch(buf, offs, threads)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return out[0], out[1], best


def cpu_baseline_encode(mb, buf, offs, n):
    """cpu_baseline for the encode workloads: the reference on all of rank 0's shard with every host thread, its
    single-thread rate on a sample, and the cores that throughput is worth."""
    from oracle import oracle_py
    threads = host_threads()
    if not oracle_py.ref_available():
        om = oracle_py.OracleModel(mb)
        sample = min(n, 100000)
        t0 = time.perf_counter()
        ids, ido = om.encode_batch(buf, offs[: sample + 1])
        dt = time.perf_counter() - t0
        return {"value": sample / dt, "unit": "sentences/s", "cores": 1, "kind": "port",
                "sample": f"first {sample} sentences, scalar C oracle (oracle/_ref missing on this box)"}, (ids, ido, sample)
    ids, ido, secs = reference_encode(mb, buf, offs, threads)
    rate = n / secs
    s1 = min(n, 40000)
    rm = oracle_py.RefModel(mb)
    t0 = time.perf_counter()
    rm.encode_count(buf, offs[: s1 + 1], 1)
    rate1 = s1 / (time.perf_counter() - t0)
    return {"value": rate, "unit": "sentences/s", "cores": threads, "kind": "reference",
            "single_thread_value": rate1, "effective_cores": round(rate / rate1, 2), "cgroup_cpu_limit": cgroup_cpu_limit(),
            "sample": f"all {n} sentences of rank 0's shard per pass, best of 2 passes; unmodified reference Encode via "
                      f"oracle/_ref with {threads} std::threads (effective_cores = this rate / the single-thread rate)"}, \
        (ids, ido, n)


# ------------------------------------------------------------------------------------------ reference arm ----

def run_reference_arm(args, rank, world):
    """The reference's own CPU implementation on this box's host cores (rank 0 only)."""
    if rank != 0:
        return
    import corpus
    from oracle import oracle_py
    workload = HEADLINE if args.workload == "all" else args.workload
    model, kind, desc = WORKLOADS[workload]
    mb = model_bytes(model)
    if not oracle_py.ref_available():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref is not built on this box"}))
        return
    threads = host_threads()
    g = corpus.CorpusGen()
    rm = oracle_py.RefModel(mb)
    if workload == "sample_nbest64_en":
        n = min(args.sentences, 262144)
        sample = min(n, 4000 * max(1, min(threads, 8)))
        buf, offs = g.fill(kind, CORPUS_SEED, sample)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            rm.sample_encode_batch(buf, offs, 64, 0.5, 1)
        dt = time.perf_counter() - t0
        rate, ids_ps, md5, used = sample * args.steps / dt, None, None, 1
        sample_txt = (f"first {sample} sentences per step, ONE thread over SentencePieceProcessor::SampleEncode (its "
                      "thread_local generator makes a multi-thread run non-reproducible)")
    elif workload == "decode_unigram32k_en":
        n = args.sentences
        buf, offs = g.fill(kind, CORPUS_SEED, n)
        ids, ido = rm.encode_batch(buf, offs, threads)
        for _ in range(args.warmup):
            rm.decode_batch(ids, ido, threads=threads)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            rm.decode_batch(ids, ido, threads=threads)
        dt = time.perf_counter() - t0
        rate, ids_ps, md5, used, sample = n * args.steps / dt, float(ido[-1]) / n, None, threads, n
        sample_txt = f"all {n} id lists per step, {threads} std::threads over SentencePieceProcessor::Decode (oracle/_ref)"
    else:
        n = args.sentences
        sample = n
        buf, offs = g.fill(kind, CORPUS_SEED, n)
        for _ in range(max(1, args.warmup)):
            rm.encode_count(buf, offs, threads)
        t0 = time.perf_counter()
        total_ids = 0
        for _ in range(args.steps):
            total_ids = rm.encode_count(buf, offs, threads)
        dt = time.perf_counter() - t0
        ids, ido = rm.encode_batch(buf, offs, threads)  # untimed: the hash both arms print
        md5 = ids_md5(ids, ido)
        rate, ids_ps, used = n * args.steps / dt, total_ids / n, threads
        sample_txt = (f"all {n} sentences of one GPU's shard per step, {threads} std::threads over "
                      "SentencePieceProcessor::Encode (oracle/_ref)")
    in_bytes = int(offs[-1])
    cfg = make_config(workload, args.sentences if workload != "sample_nbest64_en" else min(args.sentences, 262144),
                      in_bytes / sample, ids_ps if ids_ps is not None else 0.0)
    print(json.dumps({
        "impl": "reference", "metric": "sentences_per_sec", "value": rate, "unit": "sentences/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": DTYPE,
        "data": "synthetic", "input_MBps": in_bytes * args.steps / dt / 1e6, "config": cfg, "ids_md5": md5,
        "cpu_baseline": {"value": rate, "unit": "sentences/s", "cores": used, "kind": "reference", "sample": sample_txt,
                         "cgroup_cpu_limit": cgroup_cpu_limit()},
        "e2e": {"value": rate, "unit": "sentences/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# ---------------------------------------------------------------------------------------- encode workloads ----

def run_encode_workload(args, workload, rank, world, local_rank, scaling, light=False, dump=False):
    """One encode workload (unigram / BPE / byte-fallback).  Returns the result dict on rank 0, None elsewhere.
    scaling = "weak": every rank encodes its own `--sentences` sentences; "strong": the `--sentences` corpus of rank 0
    is cut into byte-balanced contiguous ranges (sharding.shard_ranges), one per rank.
    light = True (nested workloads): fewer repeats of the host-side variants.
    dump = True: the ids of the last timed step go to --dump-outputs."""
    import torch
    import torch.distributed as dist
    import corpus
    from sentencepiece_b200 import Engine, _capi
    from sentencepiece_b200.sharding import shard_ranges

    model, kind, desc = WORKLOADS[workload]
    mb = model_bytes(model)
    dev = torch.device("cuda", local_rank)
    eng = Engine(mb, device=local_rank)
    if args.lanes or args.cap or args.threads:
        eng.set_tuning(args.lanes, args.cap, args.threads)
    lib = _capi.load()
    g = corpus.CorpusGen()
    # BPE: the engine remembers the ids of words it has merged (word cache).  A bench that encodes the SAME batch K
    # times would find every word of the batch in it from the second step on, which no stream of fresh text does: the
    # cache is emptied before every step, inside the timed region, so each step only profits from repeats inside its
    # own 1M sentences.  The warm figure (cache kept across steps) is reported beside it as a variant.
    cold_cache = model.startswith("bpe") and not args.warm_cache

    # ---- this rank's shard, generated straight into pinned host memory ----
    if scaling == "strong" and world > 1:
        n_all = args.sentences
        cap_all = (320 if kind == "en" else 512) * (n_all + 1)
        tmp = np.empty(cap_all, dtype=np.uint8)
        b_all, o_all = g.fill(kind, CORPUS_SEED, n_all, first=0, out=tmp)
        ranges = shard_ranges(o_all, world)
        lo, hi = ranges[rank]
        n = hi - lo
        sizes = [r[1] - r[0] for r in ranges]
        o = (o_all[lo:hi + 1] - o_all[lo]).astype(np.uint64)
        total_bytes = int(o[-1])
        pin_bytes = lib.spm_host_alloc(total_bytes + 64)
        pin_offs = lib.spm_host_alloc(8 * (n + 1))
        hbuf = np.ctypeslib.as_array(ctypes.cast(pin_bytes, ctypes.POINTER(ctypes.c_uint8)), (total_bytes + 64,))
        hbuf[:total_bytes] = b_all[int(o_all[lo]):int(o_all[hi])]
        del tmp, b_all
        n_job = n_all
    else:
        n = args.sentences
        sizes = [n] * world
        cap_bytes = (320 if kind == "en" else 512) * (n + 1)
        pin_bytes = lib.spm_host_alloc(cap_bytes)
        pin_offs = lib.spm_host_alloc(8 * (n + 1))
        hbuf = np.ctypeslib.as_array(ctypes.cast(pin_bytes, ctypes.POINTER(ctypes.c_uint8)), (cap_bytes,))
        b, o = g.fill(kind, CORPUS_SEED, n, first=rank * n, out=hbuf)
        total_bytes = int(o[-1])
        n_job = n * world
    if not pin_bytes or not pin_offs:
        raise SystemExit("pinned allocation failed")
    hoffs = np.ctypeslib.as_array(ctypes.cast(pin_offs, ctypes.POINTER(ctypes.c_uint64)), (n + 1,))
    hoffs[:] = o

    # ---- device-resident copies (the "value" leg starts with inputs in HBM) ----
    d_bytes = torch.empty(total_bytes + 64, dtype=torch.uint8, device=dev)
    d_bytes[:total_bytes].copy_(torch.from_numpy(hbuf[:total_bytes]))
    d_offs = torch.from_numpy(o.astype(np.int64)).to(dev)
    stream = torch.cuda.current_stream().cuda_stream

    # Output buffers are double-buffered per step: the NCCL gather of step k's ids (async, NCCL stream) overlaps the
    # encode of step k+1; every gather is waited for before the timed region ends.  `--chunks C` (C > 1) additionally
    # cuts a shard into C pieces per step (more, smaller launches).
    C = max(1, args.chunks) if world > 1 else 1
    cuts = [(n * c) // C for c in range(C + 1)]
    max_piece = [max((sizes[r] * (c + 1)) // C - (sizes[r] * c) // C for r in range(world)) for c in range(C)]

    def make_pieces():
        out = []
        for c in range(C):
            lo_c, hi_c = cuts[c], cuts[c + 1]
            nb = int(o[hi_c] - o[lo_c])
            cap_ids = nb + 4 * (hi_c - lo_c) + 1024
            out.append({"lo": lo_c, "n": hi_c - lo_c, "bytes": nb, "cap": cap_ids,
                        "ids": torch.empty(cap_ids, dtype=torch.int32, device=dev),
                        "ido": torch.zeros(max_piece[c] + 1, dtype=torch.int64, device=dev),
                        "recv_ids": None, "recv_ido": None})
        return out
    slots = [make_pieces(), make_pieces()] if world > 1 else [make_pieces()]
    inflight = [[], []]   # NCCL work handles of the gathers reading slot 0 / 1

    def encode_piece(p):
        return eng.encode_device(d_bytes.data_ptr(), d_offs.data_ptr() + 8 * p["lo"], p["n"], p["bytes"],
                                 p["ids"].data_ptr(), p["cap"], p["ido"].data_ptr(), stream)

    gathered = {"bytes": 0}
    step_no = [0]

    def step():
        """one pass over the shard; returns (ids, launches, main kernel ms, all kernels ms)"""
        k = step_no[0] % len(slots)
        step_no[0] += 1
        if cold_cache:
            eng.cache_reset()
        for w in inflight[k]:   # the gather that read this slot two steps ago
            w.wait()
        inflight[k] = []
        tot, launches, main, allk, moved = 0, 0, 0.0, 0.0, 0
        for p in slots[k]:
            t = encode_piece(p)
            info = eng.info()
            tot += t
            launches += info.last_kernel_launches
            main += info.last_main_kernel_ms
            allk += info.last_kernel_ms
            if world > 1 and not args.no_gather:
                cnt = torch.tensor([t], dtype=torch.int64, device=dev)
                cnts = torch.empty(world, dtype=torch.int64, device=dev)
                dist.all_gather_into_tensor(cnts, cnt)
                cl = cnts.tolist()
                mx = int(max(cl))
                if rank == 0 and (p["recv_ids"] is None or p["recv_ids"][0].numel() < mx):
                    p["recv_ids"] = [torch.empty(int(mx * 1.02) + 64, dtype=torch.int32, device=dev) for _ in range(world)]
                    p["recv_ido"] = [torch.empty_like(p["ido"]) for _ in range(world)]
                recv = [x[:mx] for x in p["recv_ids"]] if rank == 0 else None
                inflight[k].append(dist.gather(p["ids"][:mx], recv, dst=0, async_op=True))
                inflight[k].append(dist.gather(p["ido"], p["recv_ido"] if rank == 0 else None, dst=0, async_op=True))
                moved += 4 * int(sum(cl[1:])) + 8 * p["ido"].numel() * (world - 1)
        gathered["bytes"] = moved
        return tot, launches, main, allk

    def finish_gathers():
        for k in range(len(inflight)):
            for w in inflight[k]:
                w.wait()
            inflight[k] = []

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    total_ids = 0
    for _ in range(args.warmup):
        total_ids = step()[0]
    finish_gathers()

    # ---- timed: exactly K steps, CUDA events, barrier + synchronize on both sides ----
    sampler = ClockSampler(local_rank)
    sync_all()
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    main_ms, all_ms, launches = [], [], 0
    ev0.record()
    for _ in range(args.steps):
        total_ids, ln, mm, am = step()
        launches += ln
        main_ms.append(mm)
        all_ms.append(am)
    finish_gathers()   # every step's gather completes inside the timed region
    ev1.record()
    sync_all()
    clocks = sampler.stop()
    if dump and args.dump_outputs and rank == 0:
        ids_l, offs_l = [], [np.zeros(1, np.int64)]
        for p in slots[(step_no[0] - 1) % len(slots)]:   # the output slot of the last timed step
            po = p["ido"][: p["n"] + 1].cpu().numpy()
            ids_l.append(p["ids"][: int(po[-1])].cpu().numpy())
            offs_l.append(po[1:] + offs_l[-1][-1])
        dump_lists(args, workload, "ids", np.concatenate(ids_l), np.concatenate(offs_l))
    ms = ev0.elapsed_time(ev1)
    enc_ms = statistics.mean(all_ms)
    job_ids = total_ids
    if world > 1:
        t = torch.tensor([ms, enc_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, enc_ms = float(t[0].item()), float(t[1].item())
        t = torch.tensor([total_ids, total_bytes], dtype=torch.int64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        job_ids, job_bytes = int(t[0].item()), int(t[1].item())
    else:
        job_bytes = total_bytes
    value = n_job * args.steps / (ms / 1e3)

    # ---- e2e through the host-buffer C ABI (pinned host input; H2D and D2H inside), each rank its shard ----
    e2e, e2e_out = None, None
    if not args.no_e2e:
        for _ in range(2):
            eng.encode_packed_ptr(pin_bytes, pin_offs, n)
        sync_all()
        t0 = time.perf_counter()
        h2d = d2h = 0
        for _ in range(args.steps):
            if cold_cache:
                eng.cache_reset()
            tot, ids_p, ido_p = eng.encode_packed_ptr(pin_bytes, pin_offs, n)
            info = eng.info()
            h2d, d2h = info.last_h2d_bytes, info.last_d2h_bytes
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
            t = torch.tensor([h2d, d2h], dtype=torch.int64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            h2d, d2h = int(t[0].item()), int(t[1].item())
        e2e = {"value": n_job * args.steps / dt, "unit": "sentences/s", "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(d2h), "ms_per_step": dt / args.steps * 1e3,
               "api": "spm_encode_ids (host buffers, pinned input); every rank's ids land in its own pinned host buffer",
               "timer": "host wall clock around K synchronous calls, max over ranks"}
        # the output of the LAST timed call: what the parity check looks at
        e2e_out = (np.ctypeslib.as_array(ctypes.cast(ids_p, ctypes.POINTER(ctypes.c_int32)), (max(tot, 1),))[:tot].copy(),
                   np.ctypeslib.as_array(ctypes.cast(ido_p, ctypes.POINTER(ctypes.c_uint64)), (n + 1,)).copy())

    result = None
    if rank == 0:
        # ---- other ways into the same path (rank 0, one GPU): what a caller without pinned buffers pays ----
        variants = None
        if e2e is not None and not args.no_variants:
            reps = 2 if light else 4
            pg_b = np.array(hbuf[:total_bytes], copy=True)      # pageable copies of the inputs
            pg_o = np.array(hoffs, copy=True)
            eng.encode_packed(pg_b, pg_o, copy=False)
            best = None
            for _ in range(reps):
                t0 = time.perf_counter()
                eng.encode_packed(pg_b, pg_o, copy=False)
                d1 = time.perf_counter() - t0
                best = d1 if best is None else min(best, d1)
            variants = {"pageable_input_spm_encode_ids": {"value": n / best, "unit": "sentences/s", "ms_per_step": best * 1e3,
                                                          "note": "best of %d calls, one GPU (rank 0's shard)" % reps}}
            if cold_cache:  # the same batch again with the word cache kept (device-resident and host-buffer calls)
                bw, bh = None, None
                for _ in range(reps + 1):
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    encode_piece(slots[0][0])
                    torch.cuda.synchronize()
                    d1 = time.perf_counter() - t0
                    bw = d1 if bw is None else min(bw, d1)
                    t0 = time.perf_counter()
                    eng.encode_packed_ptr(pin_bytes, pin_offs, n)
                    d1 = time.perf_counter() - t0
                    bh = d1 if bh is None else min(bh, d1)
                variants["warm_word_cache"] = {
                    "value_device_resident": slots[0][0]["n"] / bw, "value_host_buffers": n / bh, "unit": "sentences/s",
                    "note": "word cache NOT emptied between calls: every word of the batch is found (an upper bound; fresh "
                            "text lies between this and the headline); host wall clock, best of %d, rank 0's shard" % (reps + 1)}
            hb = os.path.join(ROOT, "sentencepiece_b200", "lib", "libspm_b200_hostbench.so")
            if os.path.exists(hb):
                H = ctypes.CDLL(hb)
                H.spm_hostclass_encode_bench.argtypes = [ctypes.c_char_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p,
                                                         ctypes.c_size_t, ctypes.c_int] + [ctypes.c_void_p] * 3
                bm, mm, ti = ctypes.c_double(), ctypes.c_double(), ctypes.c_uint64()
                rc = H.spm_hostclass_encode_bench(model_path(model).encode(), local_rank, pg_b.ctypes.data, pg_o.ctypes.data,
                                                  n, reps, ctypes.byref(bm), ctypes.byref(mm), ctypes.byref(ti))
                if rc == 0:
                    variants["cpp_class_Encode_vector_string_view"] = {
                        "value": n / (bm.value / 1e3), "unit": "sentences/s", "ms_per_step": bm.value,
                        "ids": int(ti.value), "note": "sentencepiece::SentencePieceProcessor::Encode(const std::vector<"
                        "std::string_view>&, std::vector<std::vector<int>>*) of csrc/host: packs the views, one engine "
                        "call, one std::vector<int> per sentence; best of %d calls" % reps}
        # ---- CPU baseline + parity of the timed path against the unmodified reference ----
        cpu, parity = None, {"result": "unchecked", "reason": "--no-cpu or --no-e2e"}
        if not args.no_cpu:
            cpu, (r_ids, r_ido, r_n) = cpu_baseline_encode(mb, hbuf, o, n)
            if e2e_out is not None:
                o_ids, o_ido = e2e_out
                k = int(r_ido[r_n])
                ok = (np.array_equal(o_ido[: r_n + 1], r_ido[: r_n + 1]) and np.array_equal(o_ids[:k], r_ids[:k]))
                parity = {"result": "bit-exact" if ok else "MISMATCH", "sentences_compared": int(r_n), "ids_compared": k,
                          "against": "oracle/_ref (unmodified reference)" if cpu["kind"] == "reference" else "oracle port",
                          "what": "ids + id_offsets returned by the last timed spm_encode_ids call (rank 0's shard)"}
        md5 = ids_md5(*e2e_out) if e2e_out is not None else None
        # ---- roofline of the dominant kernel (the encode kernel) ----
        peak, peak_src = load_peak()
        alg_bytes = total_bytes + 8 * n + 4 * total_ids  # SURVEY 8d: input + 4 + 4*ids + 4 per sentence (this rank's launches)
        kernel_ms = statistics.mean(main_ms)
        achieved = alg_bytes / (kernel_ms / 1e3) / 1e9
        tr = load_traffic(workload, n)
        kname = ("encode_bpe_lane2_kernel" if "bpe" in model else
                 "encode_unigram_lane_plain_kernel" if kind == "mixed" else "encode_unigram_lane_kernel")
        roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": tr["traffic_bytes"] if tr else None, "traffic_source": tr["source"] if tr else None,
                    "kernel": kname, "kernel_ms": kernel_ms, "launches_per_step": C,
                    "all_kernels_ms": statistics.mean(all_ms), "algorithmic_bytes_per_step": alg_bytes, "peak_source": peak_src,
                    "note": "dependent-lookup / instruction-issue bound integer path (hundreds of dependent trie lookups "
                            "per sentence against ~256 B of compulsory HBM traffic); see DESIGN.md 5"}
        cfg = make_config(workload, args.sentences, job_bytes / n_job, job_ids / n_job)
        result = {
            "metric": "sentences_per_sec", "value": value, "unit": "sentences/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": scaling, "vs_baseline": None, "dtype": DTYPE, "data": "synthetic",
            "input_MBps": job_bytes * args.steps / (ms / 1e3) / 1e6, "config": cfg,
            "run": {"sentences_per_step_whole_job": n_job, "parallelism": f"sentence-sharded x{world}",
                    "shard_sentences": sizes,
                    "l2": "inputs+outputs per step (%.0f MB per GPU) exceed the 126 MB L2" % ((total_bytes + 4 * total_ids) / 1e6),
                    "tuning": {"lanes": args.lanes, "cap": args.cap, "threads": args.threads},
                    "bpe_word_cache": ("emptied before every step, inside the timed region (value and e2e)" if cold_cache
                                       else ("kept across steps" if model.startswith("bpe") else "n/a"))},
            "clocks": clocks, "e2e": e2e, "e2e_variants": variants, "gpu_launches": int(launches), "roofline": roofline,
            "cpu_baseline": cpu, "parity": parity, "ids_md5": md5,
        }
        if world > 1:
            result["gather"] = {
                "inside_timed_region": not args.no_gather, "chunks": C, "bytes_to_rank0_per_step": gathered["bytes"],
                "encode_only_ms_per_step": enc_ms,
                "how": "per step: all_gather of the id counts, then async torch.distributed.gather (NCCL over NVLink) of the "
                       "padded int32 ids and the per-sentence offsets to rank 0 from one of two output slots; the gather of step "
                       "k overlaps the encode of step k+1 and all gathers are waited for before the closing event"}
    lib.spm_host_free(pin_bytes)
    lib.spm_host_free(pin_offs)
    eng.close()
    del d_bytes, d_offs, slots
    torch.cuda.empty_cache()
    return result


# ------------------------------------------------------------------------------------- the step after the path ----

def run_decode_workload(args, rank, world, local_rank):
    """SURVEY 8f item 2: Decode(ids) -> text for the id lists of the headline workload, through spm_decode_ids with
    host buffers.  `value` = device time of the engine's kernels, `e2e` = wall clock of the synchronous call incl. both copies."""
    import torch
    import torch.distributed as dist
    import corpus
    from sentencepiece_b200 import Engine
    model, kind, desc = WORKLOADS["decode_unigram32k_en"]
    mb = model_bytes(model)
    eng = Engine(mb, device=local_rank)
    n = args.sentences
    g = corpus.CorpusGen()
    buf, offs = g.fill("en", CORPUS_SEED, n, first=rank * n)
    ids0, ido0 = eng.encode_packed(buf, offs)          # the ids to decode ...
    total_ids = int(ido0[-1])
    lib = eng._lib
    # ... in pinned host memory (like the encode workloads' inputs); the pageable variant is measured separately
    p_ids = lib.spm_host_alloc(4 * total_ids + 64)
    p_ido = lib.spm_host_alloc(8 * (n + 1))
    ids = np.ctypeslib.as_array(ctypes.cast(p_ids, ctypes.POINTER(ctypes.c_int32)), (max(total_ids, 1),))[:total_ids]
    ido = np.ctypeslib.as_array(ctypes.cast(p_ido, ctypes.POINTER(ctypes.c_uint64)), (n + 1,))
    ids[:] = ids0
    ido[:] = ido0
    text_p, to_p = ctypes.c_void_p(), ctypes.c_void_p()

    def step(src=None):
        a = ids if src is None else src
        rc = lib.spm_decode_ids(eng._h, a.ctypes.data, ido.ctypes.data, n, ctypes.byref(text_p), ctypes.byref(to_p))
        if rc:
            raise RuntimeError(lib.spm_last_error(eng._h).decode())
    for _ in range(max(3, args.warmup)):
        step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    sampler.start()
    kernel_ms, main_ms, launches = 0.0, 0.0, 0
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
        info = eng.info()
        kernel_ms += info.last_kernel_ms
        main_ms += info.last_main_kernel_ms
        launches += info.last_kernel_launches
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    clocks = sampler.stop()
    to = np.ctypeslib.as_array(ctypes.cast(to_p, ctypes.POINTER(ctypes.c_uint64)), (n + 1,))
    text_bytes = int(to[n])
    text = np.ctypeslib.as_array(ctypes.cast(text_p, ctypes.POINTER(ctypes.c_uint8)), (max(text_bytes, 1),))[:text_bytes].copy()
    to = to.copy()
    if args.dump_outputs and rank == 0:
        dump_lists(args, "decode_unigram32k_en", "text", text, to)
    h2d, d2h = int(eng.info().last_h2d_bytes), int(eng.info().last_d2h_bytes)
    if world > 1:
        t = torch.tensor([dt, kernel_ms, main_ms], device=torch.device("cuda", local_rank))
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt, kernel_ms, main_ms = (float(x) for x in t.tolist())
    variants = None
    if rank == 0 and not args.no_variants:
        best = None
        for _ in range(3):
            t1 = time.perf_counter()
            step(ids0)
            d1 = time.perf_counter() - t1
            best = d1 if best is None else min(best, d1)
        variants = {"pageable_input_spm_decode_ids": {"value": n / best, "unit": "sentences/s", "ms_per_step": best * 1e3,
                                                      "note": "ids in ordinary (pageable) host memory: the engine stages them "
                                                              "through pinned buffers; bounded by the host's memcpy bandwidth"}}
    ids = ids0
    ido = ido0
    lib.spm_host_free(p_ids)
    lib.spm_host_free(p_ido)
    eng.close()
    if rank != 0:
        return None
    cpu, parity = None, {"result": "unchecked"}
    if not args.no_cpu:
        from oracle import oracle_py
        if oracle_py.ref_available():
            threads = host_threads()
            rm = oracle_py.RefModel(mb)
            t1 = time.perf_counter()
            r_text, r_to = rm.decode_batch(ids, ido, threads=threads)
            d1 = time.perf_counter() - t1
            cpu = {"value": n / d1, "unit": "sentences/s", "cores": threads, "kind": "reference", "cgroup_cpu_limit": cgroup_cpu_limit(),
                   "sample": f"all {n} id lists, {threads} std::threads over SentencePieceProcessor::Decode (oracle/_ref)"}
            ok = np.array_equal(r_to, to) and np.array_equal(r_text, text)
            parity = {"result": "bit-exact" if ok else "MISMATCH", "lists_compared": n, "text_bytes_compared": text_bytes,
                      "against": "oracle/_ref (unmodified reference)"}
    alg = 4 * total_ids + text_bytes + 16 * n   # ids + text + one offset each way
    peak, peak_src = load_peak()
    ach = alg / (main_ms / args.steps * 1e-3) / 1e9
    return {
        "metric": "sentences_per_sec", "value": world * n * args.steps / (kernel_ms / 1e3), "unit": "sentences/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": kernel_ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32 ids / u8 text", "data": "synthetic",
        "config": dict(make_config("decode_unigram32k_en", n, text_bytes / n, total_ids / n), text_bytes_per_list=text_bytes / n),
        "run": {"l2": "inputs+outputs per step exceed the 126 MB L2",
                "value_is": "device time of the engine's kernels (CUDA events) with host buffers",
                "e2e_is": "wall clock of spm_decode_ids incl. H2D of the ids and D2H of the text"},
        "clocks": clocks,
        "e2e": {"value": world * n * args.steps / dt, "unit": "sentences/s", "ms_per_step": dt / args.steps * 1e3,
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "api": "spm_decode_ids (host buffers, pinned input)"},
        "e2e_variants": variants, "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                     "traffic": (load_traffic("decode_unigram32k_en", n) or {}).get("traffic_bytes"), "kernel": "decode_warp_kernel",
                     "kernel_ms": main_ms / args.steps,
                     "algorithmic_bytes_per_step": alg, "peak_source": peak_src},
        "cpu_baseline": cpu, "parity": parity}


def run_sample_workload(args, rank, world, local_rank):
    """BASELINE.json configs[4]: SampleEncode(nbest_size=64, alpha=0.5) on 256k sentences.  The path goes through
    the host-buffer C ABI only (n-best on the GPU, the seeded draw on the host), so `value` is the device time of
    the engine's kernels and `e2e` the wall clock of the synchronous call."""
    import torch
    import torch.distributed as dist
    import corpus
    from sentencepiece_b200 import Engine
    model, kind, desc = WORKLOADS["sample_nbest64_en"]
    mb = model_bytes(model)
    eng = Engine(mb, device=local_rank)
    n = min(args.sentences, 262144)
    g = corpus.CorpusGen()
    buf, offs = g.fill("en", CORPUS_SEED, n, first=rank * n)
    seed = 12345 + rank
    eng.set_random_seed(seed)
    for _ in range(max(1, min(args.warmup, 2))):
        eng.sample_encode(buf, offs, 64, 0.5)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    sampler.start()
    kernel_ms, main_ms, launches = 0.0, 0.0, 0
    steps = args.steps
    t0 = time.perf_counter()
    for _ in range(steps):
        ids, ido = eng.sample_encode(buf, offs, 64, 0.5)
        info = eng.info()
        kernel_ms += info.last_kernel_ms
        main_ms += info.last_main_kernel_ms
        launches += info.last_kernel_launches
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_lists(args, "sample_nbest64_en", "ids", ids, ido)
    h2d, d2h = int(eng.info().last_h2d_bytes), int(eng.info().last_d2h_bytes)
    if world > 1:
        t = torch.tensor([dt, kernel_ms, main_ms], device=torch.device("cuda", local_rank))
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt, kernel_ms, main_ms = (float(x) for x in t.tolist())
    result = None
    if rank == 0:
        cpu, parity = None, {"result": "unchecked"}
        nb = None
        if not args.no_cpu:
            from oracle import oracle_py
            if oracle_py.ref_available():
                # parity of a seeded batch (fresh seed on both sides) + the single-thread reference rate
                sample = 12000
                rm = oracle_py.RefModel(mb)
                t1 = time.perf_counter()
                r_ids, r_ido = rm.sample_encode_batch(buf, offs[: sample + 1], 64, 0.5, 4242)
                d1 = time.perf_counter() - t1
                eng.set_random_seed(4242)
                o_ids, o_ido = eng.sample_encode(buf, offs[: sample + 1], 64, 0.5)
                ok = np.array_equal(r_ido, o_ido) and np.array_equal(r_ids, o_ids)
                parity = {"result": "bit-exact" if ok else "MISMATCH", "sentences_compared": sample,
                          "against": "oracle/_ref SampleEncode with SetRandomGeneratorSeed(4242), one thread",
                          "what": "sampled ids of a freshly seeded batch through spm_sample_encode_ids"}
                cpu = {"value": sample / d1, "unit": "sentences/s", "cores": 1, "kind": "reference",
                       "sample": f"first {sample} sentences, one thread over SentencePieceProcessor::SampleEncode (the "
                                 "reference's sampling path is per-call; its thread_local generator makes multi-thread "
                                 "runs non-reproducible)"}
        # algorithmic bytes: the input, the n-best lists the search has to produce (ids + one float score per
        # candidate) and the sampled ids; the agenda / hypothesis records are scratch, not compulsory traffic
        nbl = eng.nbest_encode(buf, offs[: 2001], 64)
        cand_ids_per_sentence = float(nbl["cand_offsets"][-1]) / 2000
        cands_per_sentence = float(nbl["n_cands"].sum()) / 2000
        total_bytes = int(offs[-1])
        alg = total_bytes + 16 * n + 4 * int(ido[-1]) + int(n * (4 * cand_ids_per_sentence + 4 * cands_per_sentence))
        peak, peak_src = load_peak()
        ach = alg / (main_ms / steps * 1e-3) / 1e9
        result = {
            "metric": "sentences_per_sec", "value": world * n * steps / (kernel_ms / 1e3), "unit": "sentences/s",
            "n_gpus": world, "steps": steps, "warmup": max(1, min(args.warmup, 2)), "ms_per_step": kernel_ms / steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8 text / int32 ids / f32 lattice scores / f64 sampling", "data": "synthetic",
            "config": dict(make_config("sample_nbest64_en", n, total_bytes / n, float(ido[-1]) / n), nbest_size=64, alpha=0.5),
            "run": {"value_is": "device time of the engine's kernels (CUDA events)", "e2e_is": "wall clock of "
                    "spm_sample_encode_ids incl. H2D, n-best kernel, D2H of scores, host draw, gather, D2H of ids",
                    "candidate_ids_per_sentence": cand_ids_per_sentence, "candidates_per_sentence": cands_per_sentence},
            "clocks": clocks,
            "e2e": {"value": world * n * steps / dt, "unit": "sentences/s", "ms_per_step": dt / steps * 1e3,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                         "traffic": (load_traffic("sample_nbest64_en", n) or {}).get("traffic_bytes"),
                         "kernel": "nbest_lane_kernel", "kernel_ms": main_ms / steps, "algorithmic_bytes_per_step": alg,
                         "peak_source": peak_src,
                         "note": "input + the 64-best lists (ids and scores) + sampled ids; the A* agenda / hypothesis pool "
                                 "(~0.3 MB of scratch per sentence in flight) is what the kernel actually waits on"},
            "cpu_baseline": cpu, "parity": parity}
    eng.close()
    return result


def run_workload(args, name, rank, world, local_rank, scaling="weak", light=False):
    if name == "sample_nbest64_en":
        return run_sample_workload(args, rank, world, local_rank)
    if name == "decode_unigram32k_en":
        return run_decode_workload(args, rank, world, local_rank)
    return run_encode_workload(args, name, rank, world, local_rank, scaling, light, dump=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="all", choices=sorted(WORKLOADS) + ["all"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--sentences", type=int, default=1_000_000, help="sentences per GPU per step (strong scaling: of the whole job)")
    ap.add_argument("--chunks", type=int, default=1, help="N > 1: launches per shard and step")
    ap.add_argument("--lanes", type=int, default=0)
    ap.add_argument("--cap", type=int, default=0)
    ap.add_argument("--threads", type=int, default=0)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-gather", action="store_true")
    ap.add_argument("--no-variants", action="store_true")
    ap.add_argument("--warm-cache", action="store_true", help="BPE: keep the engine's word cache across steps")
    ap.add_argument("--no-nested", action="store_true", help="with --workload all: the headline workload only")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of each workload's last timed step to DIR")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback exists for the engine)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    head = HEADLINE if args.workload == "all" else args.workload
    out = run_workload(args, head, rank, world, local_rank, scaling=args.scaling)
    failed = False
    if args.workload == "all" and not args.no_nested:
        nested = {}
        if world > 1 and args.scaling == "weak":
            r = run_encode_workload(args, HEADLINE, rank, world, local_rank, "strong", light=True)
            if rank == 0:
                out["strong_scaling"] = r
        for name in NESTED:
            r = run_workload(args, name, rank, world, local_rank, scaling=args.scaling, light=True)
            if rank == 0:
                nested[name] = r
            if world > 1 and name in ENCODE_WORKLOADS and args.scaling == "weak":
                r2 = run_encode_workload(args, name, rank, world, local_rank, "strong", light=True)
                if rank == 0:
                    nested[name]["strong_scaling"] = r2
        if rank == 0:
            out["workloads"] = nested
    if rank == 0:
        def bad(d):
            return isinstance(d, dict) and ((d.get("parity") or {}).get("result") == "MISMATCH" or
                                            any(bad(v) for v in d.values() if isinstance(v, dict)))
        failed = bad(out)
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()
    if failed:
        raise SystemExit("bench.py: the timed path's output differs from the reference (parity MISMATCH)")


if __name__ == "__main__":
    main()
