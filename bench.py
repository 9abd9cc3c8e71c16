#!/usr/bin/env python
"""bench.py — gateway hot-path throughput on B200 (BASELINE.json metric, config 2).

  python bench.py [--gpus N] [--steps K] [--warmup W]            # our arm (CUDA, through the C ABI)
  python bench.py --impl reference ...                            # the reference's CPU path, restated (oracle port)
  python bench.py ... --dump-outputs DIR                          # + the last timed step's decisions as DIR/*.npy

Step      one pass of the hot path over one wave: the request phase of 65 536 non-streaming chat requests
          (1 KiB bodies, 10 000 tenants, Qwen-style chat JSON) followed by the response phase of every admitted
          request (~600 B completion JSON with usage). Counters persist across steps; `now` advances one day per
          step so every step starts fresh rpm/tpm and rpd/tpd windows (stationary admission pattern); quota accumulates.
value     whole-job requests/s with the waves already resident in HBM (kernels only, CUDA events on the library's
          stream). Three distinct waves rotate through staging slots, ~300 MB in total, so inputs exceed the 126 MB L2.
e2e       same metric through the public API (Gateway.handle_request_body / handle_response_body == the C-ABI submit
          calls) with pinned HOST buffers: H2D of bodies+tokens and D2H of the decision arrays inside the timed region.
roofline  dominant kernel (largest device-time share of the step): algorithmic bytes per launch / its mean duration (per-launch CUDA
          events recorded by the library on its stream), against MEASURED_PEAKS.json's HBM copy bandwidth.
N > 1     one process per GPU under torchrun; tenants are hash-partitioned, every rank owns 10 000 tenants and serves
          its own 65 536-request waves (weak scaling); no collective on the data path; time = max over ranks.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only; nothing is written into it

import numpy as np  # noqa: E402

WAVE = 65536
TENANTS = 10_000
BODY = 1024
RESP_BODY = 600
N_WAVES = 3
N_TEMPL = 0  # 0: every request / completion of a wave is generated on its own (no repeated bodies)
NOW0 = 1_700_000_000
STEP_S = 86_400  # `now` advances one day per step: fresh rpm/tpm and rpd/tpd windows each step (stationary admission pattern)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--wave", type=int, default=WAVE)
    ap.add_argument("--tenants", type=int, default=TENANTS)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-bpe", action="store_true", help="skip the BPE count section (builds a 151 k-merge stand-in vocabulary: ~30 s)")
    ap.add_argument("--shared-quota", type=int, default=0, metavar="K",
                    help="K quotas per GPU are replicas of quotas shared by all GPUs: every --fold-every steps the library folds "
                         "their increments with ncclAllReduce (arks_fold_quota_allreduce) INSIDE the timed region")
    ap.add_argument("--fold-every", type=int, default=8)
    ap.add_argument("--latency-requests", type=int, default=10_000_000,
                    help="requests per GPU in the 1.25 M/s open-loop latency run (SURVEY.md section 8d: >= 10 M; 8 s of arrivals)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the decisions of the last timed step (rank 0) as DIR/request_<field>.npy and DIR/response_<field>.npy "
                         "(float64); the inputs are seeded, so two builds run with the same arguments can be compared array by array")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    return a


def env_rank():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.p = index, [], None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                       "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=2)
        except Exception:
            self.p.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def build_waves(workload, n_waves, wave, rank):
    """n_waves distinct (request wave, matching response wave) pairs; responses answer the requests the ORACLE-FREE
    first pass admits, so they are produced after a dry request pass on the device (see run_b200)."""
    return [workload.request_batch(wave, NOW0, seed=1000 + 17 * rank + k, body_size=BODY, n_templates=N_TEMPL, varied=True)
            for k in range(n_waves)]


def bpe_section(g, w, reqs, resps, now, peak, ext, sample=2048):
    """Request waves with a vocabulary loaded: device time of the two BPE kernels per 65 536-body wave, their algorithmic
    bytes (body read once + decoded text written and read + one 8-byte work-list entry per piece written and read + the count),
    and SEPARATELY the merge-table slots they read (SURVEY.md section 8d: probes are not body bytes) - counted on the host build of
    the same code (tests/host_machine.cpp) over a sample and scaled by body bytes. Every sampled count is compared with HF
    `tokenizers` (the external oracle of this column). The Qwen2.5 vocabulary is not on disk: a seeded stand-in of the same
    size (151 k merges) trained with `tokenizers` on synthetic text, same pre-tokenizer and algorithm."""
    from arks_b200 import bpe
    t0 = time.perf_counter()
    tok, text = bpe.standin_tokenizer(151_643)
    tables = bpe.load_tokenizer(text)
    vocab_s = time.perf_counter() - t0
    import torch
    g.load_bpe(tables)
    try:
        for k in range(N_WAVES):
            g.select_slot(k)
            g.stage_request(reqs[k])
            g.stage_response(resps[k])
        g.set_profiling(True)
        ms, ms_resp = [], []
        for i in range(3 + 12):
            g.select_slot(i % N_WAVES)
            g.run_request(now)
            t = g.last_kernel_ms()
            g.run_response(now + 1)
            t2 = g.last_kernel_ms()
            now += STEP_S
            if i >= 3:
                ms.append(t[3])
                ms_resp.append(t2[2])
        g.set_profiling(False)
        # the whole step (request stage + admit + response stage) with both count columns on: BASELINE config 2 names the
        # vocabulary, the reference itself counts nothing (SURVEY.md section 0 F1), so the line's `value` is the step without the side
        # output and this is the same step with it
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(ext)
        for i in range(12):
            g.select_slot(i % N_WAVES)
            g.run_request(now)
            g.run_response(now + 1)
            now += STEP_S
        e1.record(ext)
        torch.cuda.synchronize()
        step_ms = e0.elapsed_time(e1) / 12
        g.select_slot(0)
        reqs[0].now_unix = now
        counts = g.handle_request_body(reqs[0]).bpe_count.copy()
    finally:
        g.set_profiling(False)
        g.load_bpe(None)
    # the sample: first `sample` rows of wave 0 against `tokenizers`, and through the host build for the table probes
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import hostmachine as hm
    with tempfile.TemporaryDirectory() as tmp:
        hm.OUT = os.path.join(tmp, os.path.basename(hm.OUT))  # compiled for this run, outside the tree
        hm.lib()
    hm.bpe_load(tables)
    hm.bpe_probes()
    rb = reqs[0]
    n = min(sample, rb.n)
    wrong = uncounted = 0
    sample_body_bytes = 0
    for i in range(n):
        body = bytes(rb.bodies[rb.body_off[i]:rb.body_off[i] + rb.body_len[i]])
        sample_body_bytes += len(body)
        hm.bpe_count(body)
        if counts[i] == bpe.UNCOUNTED:
            uncounted += 1
            continue
        wrong += int(counts[i]) != sum(len(tok.encode(x, add_special_tokens=False).ids) for x in bpe.content_strings(body))
    hot, full, pieces, text_bytes = hm.bpe_probes()
    body_bytes = float(np.mean([int(b.body_len.sum()) for b in reqs]))
    scale = body_bytes / sample_body_bytes
    alg = body_bytes + scale * (2 * text_bytes + 16 * pieces) + 4 * rb.n
    t_s = float(np.mean(ms)) / 1e3
    counted = counts[counts != bpe.UNCOUNTED]
    return {"kernels": "bpe_scan_kernel + bpe_merge_kernel", "ms_per_wave": t_s * 1e3, "bodies_per_wave": int(rb.n),
            "ms_per_response_wave": float(np.mean(ms_resp)), "response_bodies_per_wave": int(resps[0].n),
            "step_with_counts": {"ms_per_step": step_ms, "value": rb.n / (step_ms / 1e3), "unit": "req/s per GPU",
                                 "what": "request stage + limit_admit + response stage with the prompt and completion BPE counts on (12 steps, CUDA events, "
                                         "waves rotating through the staging slots as in the timed region of `value`)"},
            "tokens_per_wave_0": int(counted.sum()), "tokens_per_s": float(counted.sum()) / t_s, "uncounted_rows_wave_0": int((counts == bpe.UNCOUNTED).sum()),
            "roofline": {"bound": "hbm", "achieved": alg / t_s / 1e9, "peak": peak, "unit": "GB/s", "frac": alg / t_s / 1e9 / peak,
                         "algorithmic_bytes_per_launch": alg,
                         "what": "body bytes read once + decoded text written and read + 8 B work-list entry per pre-token written and read + 4 B count"},
            "table_probes": {"full_table_slots_per_wave": scale * full, "full_table_bytes_per_wave": scale * full * 16,
                             "hot_table_slots_per_wave": scale * hot, "pretokens_per_wave": scale * pieces,
                             "what": "16-byte merge-table slots read, NOT counted as body bytes: full table = open-addressing hash in HBM (8 MB, L2-resident), "
                                     "hot table = the 768 lowest-rank merges staged into shared memory by one bulk copy (TMA) per block; counted on the host "
                                     f"build of bpe.cuh over the first {n} bodies of wave 0 and scaled by body bytes"},
            "checked_against_tokenizers": {"rows": n, "uncounted": uncounted, "different": wrong},
            "vocabulary": f"stand-in byte-level BPE, {len(tables.left)} merges, Qwen2 pre-tokenizer, NFC flag {tables.flags} (the Qwen2.5 files are not on disk); built in {vocab_s:.1f} s"}


def bind_to_gpu_numa(local: int):
    """Run this rank's threads (and so, by first touch, its pinned staging buffers) on the NUMA node its GPU hangs off:
    round 1's 8-GPU end-to-end curve fell to 0.67 because GPUs 4-7 sit on node 1 while every rank's host buffers and
    batcher threads were wherever the scheduler put them. Returns what was done (for the report)."""
    try:
        bus = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(local)],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        dom, rest = bus.split(":", 1)
        node = int(open(f"/sys/bus/pci/devices/{dom[-4:]}:{rest}/numa_node").read())
        if node < 0:
            return {"numa_node": None, "note": "no NUMA information for this GPU"}
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return {"numa_node": node, "note": "node has no CPU this process may use"}
        os.sched_setaffinity(0, cpus)
        return {"numa_node": node, "cpus": len(cpus)}
    except Exception as e:  # no sysfs / nvidia-smi: run unpinned
        return {"numa_node": None, "note": f"not pinned: {e!r}"}


def pin_batch(b):
    """Re-home a batch's arrays in pinned host memory (what the Go batcher's ring buffers would be)."""
    import torch
    for name in ("bodies", "body_off", "body_len", "tokens", "token_off", "pick_rand", "qos", "flags"):
        a = getattr(b, name, None)
        if a is None:
            continue
        t = torch.from_numpy(a).pin_memory()
        setattr(b, name, t.numpy())
        b.__dict__.setdefault("_pins", []).append(t)
    return b


def write_outputs(out_dir, dump, cap=60 << 20):
    """The decision arrays a caller of the timed path receives, as float64 (every value is an integer below 2**53):
    request_<field>.npy and response_<field>.npy, one row per request / response (usage: 3 columns). <phase>_row.npy holds
    the row numbers: every row while the arrays fit in `cap` bytes, else the same seeded sample of rows on every run."""
    os.makedirs(out_dir, exist_ok=True)
    phases = {p: {"row": np.arange(len(dump[p].reason)), **dump[p].fields()} for p in ("request", "response")}
    total = sum(8 * a.size for f in phases.values() for a in f.values())
    for phase, f in phases.items():
        n = len(f["row"])
        keep = np.arange(n) if total <= cap else np.sort(np.random.default_rng(0).choice(n, n * cap // total, replace=False))
        for name, a in f.items():
            np.save(os.path.join(out_dir, f"{phase}_{name}.npy"), a[keep].astype(np.float64))


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def physical_cores():
    """[(socket, cpu)]: one logical CPU per physical core this process may run on, socket by socket (sysfs topology)"""
    allowed = sorted(os.sched_getaffinity(0))
    seen, out = set(), []
    for c in allowed:
        base = f"/sys/devices/system/cpu/cpu{c}/topology"
        try:
            sib = open(f"{base}/thread_siblings_list").read().strip()
            pkg = int(open(f"{base}/physical_package_id").read())
        except OSError:
            sib, pkg = str(c), 0
        if (pkg, sib) not in seen:
            seen.add((pkg, sib))
            out.append((pkg, c))
    return sorted(out)


def cpu_quota():
    """CPUs this container may use at once: the cgroup's CFS quota (cpu.max, v2; cpu.cfs_quota_us, v1) if there is one. A
    process that runs more busy threads than this is throttled — the kernel stops the WHOLE group for the rest of each
    100 ms period — which is what made the CPU arm swing 3.5x between boxes in round 1 (16-CPU quota on a 128-thread host)."""
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            return max(1, int(int(q) / int(per)))
    except (OSError, ValueError):
        pass
    try:
        q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        if q > 0:
            return max(1, q // per)
    except (OSError, ValueError):
        pass
    return None


def choose_threads(o, req, resp, now):
    """The threaded oracle is memory- and barrier-bound: more threads than physical cores of one socket rarely help and
    often hurt (round 1: 2.75 M vs 8.45 M req/s on two boxes of the same type because the count was picked from 4 noisy
    timings). Candidates are sets of PHYSICAL cores, the workers are pinned to them, every candidate gets a warm-up wave and
    5 timed waves, the median decides; all candidates' rates go into the report."""
    cores = physical_cores()
    sock0 = [c for p, c in cores if p == cores[0][0]]
    allc = [c for _, c in cores]
    quota = cpu_quota()
    # more busy threads than the quota get the group throttled; one CPU of it is left to everything that is not a worker
    cap = (lambda cpus: cpus[:max(1, quota - 1)]) if quota else (lambda cpus: cpus)
    cands = []
    for cpus in (sock0, sock0[:max(1, len(sock0) // 2)], sock0[:max(1, len(sock0) // 4)], allc, allc[:max(1, len(allc) // 2)],
                 sock0[:max(1, (quota or len(sock0)) // 2)]):
        cpus = cap(cpus)
        if cpus and cpus not in cands:
            cands.append(cpus)
    everything = set(os.sched_getaffinity(0))
    rates, best = [], None
    for cpus in cands:
        os.sched_setaffinity(0, cpus)  # the oracle's pool is re-created per thread count and inherits this mask
        ts = []
        for k in range(6):
            req.now_unix, resp.now_unix = now, now + 1
            t0 = time.perf_counter()
            o.request_batch(req, threads=len(cpus))
            o.response_batch(resp, threads=len(cpus))
            if k:
                ts.append(time.perf_counter() - t0)
            now += STEP_S
        med = float(np.median(ts))
        rates.append({"threads": len(cpus), "sockets": len({p for p, c in cores if c in cpus}), "req_per_s": round(req.n / med)})
        if best is None or med < best[0]:
            best = (med, cpus)
    os.sched_setaffinity(0, best[1])
    return best[1], rates, now, everything


def sharded_reference_workload(args, world):
    """What `world` tenant-sharded GPUs serve per step, for the CPU arm: world x tenants, world x wave requests. The bodies of
    the world shards are the same 64 Ki generated documents (generating world x 64 Ki distinct ones in Python would take
    minutes and changes nothing for a parser); every shard has its own tenants, tokens and counters."""
    from arks_b200 import abi, traffic
    from arks_b200.tables import Tables
    shards = [traffic.Workload(n_tenants=args.tenants, seed=0xA2C5 + r) for r in range(world)]
    if world == 1:
        w = shards[0]
        return w, w.request_batch(args.wave, NOW0, seed=1000, body_size=BODY, n_templates=N_TEMPL, varied=True)
    tokens, quotas, endpoints = [], [], []
    for r, sh in enumerate(shards):  # namespaces are per shard: prefix them so that the merged config keeps them apart
        for objs, out in ((sh.objects[0], tokens), (sh.objects[1], quotas), (sh.objects[2], endpoints)):
            for o in objs:
                o = json.loads(json.dumps(o))
                o["metadata"]["namespace"] = f"s{r}-" + o["metadata"]["namespace"]
                if "token" in o.get("spec", {}):
                    o["spec"]["token"] = f"s{r}-" + o["spec"]["token"]
                out.append(o)
    merged = traffic.Workload.__new__(traffic.Workload)
    merged.tables = Tables(tokens, quotas, endpoints)
    merged.n_tenants, merged.seed, merged.popularity = args.tenants * world, 0xA2C5, None
    merged.token_strings = [f"s{r}-".encode() + t for r, sh in enumerate(shards) for t in sh.token_strings]
    base = shards[0].request_batch(args.wave, NOW0, seed=1000, body_size=BODY, n_templates=N_TEMPL, varied=True)
    bodies = [bytes(base.bodies[base.body_off[i]:base.body_off[i] + base.body_len[i]]) for i in range(base.n)]
    toks = [bytes(base.tokens[base.token_off[i]:base.token_off[i + 1]]) for i in range(base.n)]
    req = abi.RequestBatch.from_lists(bodies * world, [f"s{r}-".encode() + t for r in range(world) for t in toks], NOW0,
                                      pick_rand=np.tile(base.pick_rand, world))
    return merged, req


def cpu_arm(args, world, seconds=None, steps=None, warmup=0):
    """The reference's CPU path as restated by the oracle (kind=port): the C restatement of the Go handlers with in-memory
    counters — it omits the ~9 Redis round trips per request the real gateway pays, i.e. a generous baseline (BASELINE.md §4).
    Tenant-sharded over pinned physical cores. Either a bounded sample (`seconds`) or exactly `steps` steps."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import orklib
    w, req = sharded_reference_workload(args, world)
    o = orklib.Oracle(w.tables)
    n_any = min(os.cpu_count() or 1, cpu_quota() or 1 << 30)
    a = o.request_batch(req, threads=n_any)
    resp = w.response_batch(a, NOW0 + 1, seed=2000, body_size=RESP_BODY, varied=True, n_templates=N_TEMPL or (0 if world == 1 else 4096))
    o.response_batch(resp, threads=n_any)
    cpus, rates, now, everything = choose_threads(o, req, resp, NOW0 + STEP_S)
    threads = len(cpus)
    for _ in range(warmup):
        req.now_unix, resp.now_unix = now, now + 1
        o.request_batch(req, threads=threads)
        o.response_batch(resp, threads=threads)
        now += STEP_S
    done, t_used, n_steps = 0, 0.0, 0
    while (steps is not None and n_steps < steps) or (steps is None and t_used < seconds and n_steps < 400):
        req.now_unix, resp.now_unix = now, now + 1
        t0 = time.perf_counter()
        o.request_batch(req, threads=threads)
        o.response_batch(resp, threads=threads)
        t_used += time.perf_counter() - t0
        done += req.n
        now += STEP_S
        n_steps += 1
    os.sched_setaffinity(0, everything)
    sample = (f"{n_steps} steps of {req.n} requests + {resp.n} responses ({world} tenant shard(s) of {args.tenants} tenants); "
              f"oracle/libarks_oracle.so = C restatement of the Go path, in-memory counters, no Redis; {threads} worker threads "
              f"pinned to physical cores {cpus[0]}..{cpus[-1]}; cgroup CPU quota {cpu_quota() or 'none'} (candidates are capped at it: more busy "
              f"threads get the whole group throttled); candidates (median of 5 waves each): {json.dumps(rates)}")
    return {"value": done / t_used, "unit": "req/s", "cores": threads, "kind": "port", "sample": sample}, t_used / max(n_steps, 1)


def run_reference(args):
    rank, local, world = env_rank()
    if rank != 0:
        return
    world = max(world, args.gpus)
    cb, s_per_step = cpu_arm(args, world, steps=args.steps, warmup=args.warmup)
    v = cb["value"]
    print(json.dumps({
        "impl": "reference", "metric": "gateway requests/s (request + response phase)", "value": v, "unit": "req/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * s_per_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/int64", "data": "synthetic",
        "config": workload_config(args, world),
        "cpu_baseline": cb,
        "e2e": {"value": v, "unit": "req/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def workload_config(args, world):
    return {"workload": f"BASELINE config 2: {args.wave} concurrent non-streaming /v1/chat/completions requests per wave, "
                        f"~{BODY} B prompts on average (OpenAI chat JSON, model qwen-7b; every body distinct: 256 client applications "
                        f"with their own parameters, key order, system prompt and JSON style, 1-6 turns of random lengths, escapes and "
                        f"UTF-8 in the text: 0.3-1.7 KiB), {args.tenants} tenants "
                        f"(ArksToken+ArksQuota+ArksEndpoint each, rpm/tpm/rpd/tpd + 3-item quota), ~{RESP_BODY} B completion JSON with "
                        f"usage in three server dialects; request phase + response phase per step",
            "token_counts": "the work the reference does per request: it counts no tokens itself (usage comes from the upstream's response, "
                            "pkg/gateway/check.go:124-126); the on-device BPE count is a side output, off in `value` / `e2e` and on in "
                            "`bpe.step_with_counts` (same step, both count columns, 151 k-merge vocabulary)",
            "tenants_per_gpu": args.tenants, "requests_per_wave_per_gpu": args.wave, "parallelism": f"tenant-sharded x{world}",
            "l2": f"inputs larger than L2: {N_WAVES} distinct waves rotate through staging slots (~{N_WAVES * (args.wave * (BODY + RESP_BODY)) >> 20} MiB)"}


def run_b200(args):
    # stdout carries exactly one JSON line: libraries that announce themselves there (NCCL prints its version on stdout when
    # NCCL_DEBUG asks for it, from torch's communicator as from the library's own) are sent to stderr for the whole run
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    import torch
    import __graft_entry__ as ge
    rank, local, world = env_rank()
    numa = bind_to_gpu_numa(local)  # before any pinned allocation and before the library starts its threads
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if rank == 0:
        ge.build()
    if world > 1:
        dist.barrier()
    from arks_b200 import abi, traffic
    from arks_b200.gateway import Gateway

    # every rank owns its own tenant shard (namespaces are the tenant boundary; no key is shared across GPUs)
    w = traffic.Workload(n_tenants=args.tenants, seed=0xA2C5 + rank)
    g = Gateway(local, max_batch=args.wave, max_batch_bytes=int(args.wave * (BODY + 64) * 1.05), share_quota=args.shared_quota > 0)
    g.load_tables(w.tables)
    if args.shared_quota:
        # the communicator id travels over torch.distributed once (plumbing); the fold itself is the library's
        box = [g.comm_unique_id() if rank == 0 else None]
        if world > 1:
            dist.broadcast_object_list(box, src=0)
        n_shared = min(args.shared_quota, w.tables.n_quotas)
        g.comm_init(rank, world, box[0], np.arange(n_shared, dtype=np.uint32))
        g.fold_quota_allreduce(wait=True)
    reqs = [pin_batch(b) for b in build_waves(w, N_WAVES, args.wave, rank)]
    # dry pass to learn which requests are admitted in a fresh window, then build the matching response waves
    resps = []
    for k, rb in enumerate(reqs):
        rb.now_unix = NOW0 + STEP_S * k
        a = g.handle_request_body(rb)
        resps.append(pin_batch(w.response_batch(a, NOW0 + STEP_S * k + 1, seed=3000 + k, body_size=RESP_BODY, varied=True,
                                                n_templates=N_TEMPL)))
    req_out = [abi.RequestResult.empty(b.n) for b in reqs]
    resp_out = [abi.ResponseResult.empty(b.n) for b in resps]
    now = NOW0 + STEP_S * N_WAVES
    ext = torch.cuda.ExternalStream(g.stream_handle, device=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- kernel-only arm: waves resident in HBM --------------------------------------------------
    for k in range(N_WAVES):
        g.select_slot(k)
        g.stage_request(reqs[k])
        g.stage_response(resps[k])
    torch.cuda.synchronize()

    fold_events, fold_host_us = [], []
    dump = {} if args.dump_outputs and rank == 0 else None

    def resident_step(i, now, fold=True, keep=None):
        k = i % N_WAVES
        g.select_slot(k)
        g.run_request(now)
        if keep is not None:
            # the response phase writes its decisions over the request phase's on the device: copy those out first, between
            # two events, so that the copy can be taken out of the timed region
            keep["events"] = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            keep["events"][0].record(ext)
            keep["request"] = g.fetch_request(reqs[k].n)
            keep["events"][1].record(ext)
        g.run_response(now + 1)
        if fold and args.shared_quota and i % args.fold_every == args.fold_every - 1:
            # stream-ordered behind this step's kernels; nobody waits on the host. Timed on both sides: the device time includes
            # waiting for the slowest peer to arrive, the host time is what the enqueue costs the launching thread.
            ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            ev[0].record(ext)
            t_h = time.perf_counter()
            g.fold_quota_allreduce(wait=False)
            fold_host_us.append(1e6 * (time.perf_counter() - t_h))
            ev[1].record(ext)
            fold_events.append(ev)

    for i in range(args.warmup):
        resident_step(i, now)
        now += STEP_S
    sampler = ClockSampler(local)
    sampler.start()
    # keep the GPU under this workload until nvidia-smi has produced its first samples. A wall-clock loop: its length differs
    # per rank (a collective inside would not pair up) and per run, so it runs request phases only. Those bill no quota, and
    # every step opens fresh rate windows, so the timed steps below start from the same counters however long this took.
    t_spin = time.perf_counter()
    i = 0
    while time.perf_counter() - t_spin < 0.6:
        g.select_slot(i % N_WAVES)
        g.run_request(now)
        now += STEP_S
        i += 1
    barrier()
    launches0 = g.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(ext)
    for i in range(args.steps):
        resident_step(args.warmup + i, now, keep=dump if i == args.steps - 1 else None)
        now += STEP_S
    e1.record(ext)
    barrier()
    launches = g.launch_count - launches0
    dev_ms = e0.elapsed_time(e1)
    if dump is not None:
        dev_ms -= dump["events"][0].elapsed_time(dump["events"][1])
        dump["response"] = g.fetch_response(resps[(args.warmup + args.steps - 1) % N_WAVES].n)
        write_outputs(args.dump_outputs, dump)
    shared_quota = None
    if args.shared_quota:
        # one fold epoch timed alone (gather + all-reduce + apply), every rank in step
        f0 = [torch.cuda.Event(enable_timing=True) for _ in range(20)]
        f1 = [torch.cuda.Event(enable_timing=True) for _ in range(20)]
        barrier()
        for a_, b_ in zip(f0, f1):
            a_.record(ext)
            g.fold_quota_allreduce(wait=False)
            b_.record(ext)
        barrier()
        us = sorted(1e3 * a_.elapsed_time(b_) for a_, b_ in zip(f0, f1))
        in_loop = sorted(1e3 * a_.elapsed_time(b_) for a_, b_ in fold_events[-(args.steps // args.fold_every):]) or [0.0]
        host_us = sorted(fold_host_us[-(args.steps // args.fold_every):]) or [0.0]
        shared_quota = {"rows": int(n_shared), "message_bytes": int(n_shared) * 24, "fold_every_steps": args.fold_every,
                        "folds_in_timed_region": args.steps // args.fold_every, "fold_us_p50": round(us[len(us) // 2], 1),
                        "fold_us_max": round(us[-1], 1),
                        "in_timed_region": {"device_us_p50": round(in_loop[len(in_loop) // 2], 1), "device_us_max": round(in_loop[-1], 1),
                                            "host_enqueue_us_p50": round(host_us[len(host_us) // 2], 1), "host_enqueue_us_max": round(host_us[-1], 1),
                                            "what": "device: CUDA events around the epoch inside the step loop (includes waiting for the "
                                                    "slowest rank to arrive); host: time the call holds the launching thread"}, "how": "arks_fold_quota_allreduce: ncclAllReduce(int64, sum) issued by the "
                        "library on its compute stream (libnccl dlopen()ed), CUDA events around one epoch"}
    # per-kernel timing for the roofline (separate pass so event records do not sit inside the timed region)
    g.set_profiling(True)
    scan_ms, admit_ms, resp_ms, fast_req_ms, fast_resp_ms = [], [], [], [], []
    for i in range(args.steps):
        k = i % N_WAVES
        g.select_slot(k)
        g.run_request(now)
        ms = g.last_kernel_ms()
        scan_ms.append(ms[0]); admit_ms.append(ms[1])
        if ms[2] > 0:
            fast_req_ms.append(ms[2])
        g.run_response(now + 1)
        ms = g.last_kernel_ms()
        resp_ms.append(ms[0])
        if ms[1] > 0:
            fast_resp_ms.append(ms[1])
        now += STEP_S
    g.set_profiling(False)

    # ---- end-to-end arm: host buffers through the public API --------------------------------------
    # Every step copies that step's bodies/tokens H2D from pinned host memory and reads the decision arrays back D2H.
    # Submits are asynchronous with two batches in flight (slot ping-pong): the host packs and queues step i+1 while
    # the PCIe copies and kernels of step i run; results of step i are consumed before step i+2 is queued.
    def e2e_steps(n_steps, now):
        inflight = None
        for i in range(n_steps):
            k, slot = i % N_WAVES, i % 2
            reqs[k].now_unix, resps[k].now_unix = now, now + 1
            g.select_slot(slot)
            g.submit_request_async(reqs[k])
            g.submit_response_async(resps[k])
            if inflight is not None:
                g.wait_request(inflight[0], req_out[inflight[1]])
                g.wait_response(inflight[0], resp_out[inflight[1]])
            inflight = (slot, k)
            now += STEP_S
        g.wait_request(inflight[0], req_out[inflight[1]])
        g.wait_response(inflight[0], resp_out[inflight[1]])
        return now

    now = e2e_steps(max(args.warmup, 2), now)
    barrier()
    t0 = time.perf_counter()
    now = e2e_steps(args.steps, now)
    torch.cuda.synchronize()
    own_e2e_s = time.perf_counter() - t0  # this rank's own finish (the job's time is taken after the barrier)
    barrier()
    e2e_s = time.perf_counter() - t0
    rank_e2e_s = [own_e2e_s]
    if world > 1:
        t = torch.tensor([own_e2e_s], device=f"cuda:{local}", dtype=torch.float64)
        got = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(got, t)
        rank_e2e_s = [float(x[0]) for x in got]
    clocks = sampler.stop()  # sampled across both timed regions (kernel-only and end-to-end)
    assert int((req_out[0].reason == 0).sum()) > 0  # the decisions really came back

    # ---- added latency of one synchronous micro-batch (submit -> decisions on the host), small batches -------------
    latency = {}
    if rank == 0:
        g.select_slot(0)
        for bs in (64, 256, 1024, 4096):
            small = pin_batch(w.request_batch(bs, now, seed=7000 + bs, body_size=BODY, n_templates=64, varied=True))
            out_small = abi.RequestResult.empty(bs)
            ts = []
            for it in range(220):
                small.now_unix = now
                t1 = time.perf_counter()
                g.handle_request_body(small, out_small)
                ts.append(time.perf_counter() - t1)
                now += STEP_S
            ts = np.sort(np.array(ts[20:])) * 1e6
            latency[str(bs)] = {"p50_us": float(ts[len(ts) // 2]), "p99_us": float(ts[int(len(ts) * 0.99)])}
    # ---- the compiled host (host/cpp Batcher) at BASELINE's operating point: requests ARRIVE at 1.25 M/s on EVERY GPU at the
    # same time (10 M req/s over 8 GPUs), open loop (exponential gaps, 8 producer threads per GPU, latency = decision handed
    # over - scheduled arrival: no coordinated omission), >= args.latency_requests requests per GPU drawn from 4096 distinct
    # bodies; p50 / p99 / p99.9 per rank, worst rank reported. Little's law puts ~150-250 requests in flight per GPU: the
    # 64 k concurrent streams of the metric are open connections, of which these are the ones with a message in the gateway.
    from arks_b200 import cpphost
    hb = cpphost.Batcher(cpphost.load(cpphost.build()), g._h, max_batch=8192, max_bytes=16 << 20)
    hb.set_fixed_clock(now)
    distinct = w.request_batch(4096, now, seed=7100 + rank, body_size=BODY, n_templates=0, varied=True)

    def arrivals(n, seed):
        """n requests drawn from the 4096 distinct ones: the same body bytes, row offsets repeated"""
        idx = np.random.default_rng(seed).integers(0, distinct.n, n)
        tl = np.diff(distinct.token_off)
        L = int(tl[0])  # every generated bearer token has the same length: gather them as a matrix
        assert np.all(tl == L)
        mat = distinct.tokens[:distinct.token_off[-1]].reshape(distinct.n, L)[idx]
        return abi.RequestBatch(distinct.bodies, distinct.body_off[idx].copy(), distinct.body_len[idx].copy(),
                                np.ascontiguousarray(mat).reshape(-1), (np.arange(n + 1, dtype=np.uint64) * L).astype(np.uint32), now,
                                distinct.pick_rand[idx].copy())

    # generator threads spin; together with every rank's dispatcher they must fit the container's CPU quota, or the kernel
    # throttles the whole group for milliseconds at a time and the tail measures that
    quota = cpu_quota()
    producers = 8 if not quota else max(2, min(8, quota // world - 2))
    hb.open_loop_requests(arrivals(8000, 1), rate_per_s=400_000, producers=producers)  # warm-up: first launches, page faults
    streams_lat, open_lat = {}, {}
    for streams in ((1, 64) if rank == 0 and args.latency_requests else ()):
        n_calls = {1: 2000, 64: 40000}[streams]
        now += STEP_S; hb.set_fixed_clock(now)
        before = hb.stats()
        _, lat_ns, wall = hb.run_requests(arrivals(n_calls, 7100 + streams), threads=streams)
        after = hb.stats()
        lat_us = np.sort(lat_ns[n_calls // 10:]) / 1e3
        nb = after["request_batches"] - before["request_batches"]
        streams_lat[str(streams)] = {"p50_us": float(lat_us[len(lat_us) // 2]), "p99_us": float(lat_us[int(len(lat_us) * 0.99)]),
                                     "req_per_s": n_calls / wall, "mean_batch": n_calls / max(nb, 1)}
    for rate in ((250_000, 1_250_000) if args.latency_requests else ()):
        n_calls = int(rate * 0.4) if rate < 1_000_000 else args.latency_requests
        now += STEP_S; hb.set_fixed_clock(now)
        load = arrivals(n_calls, 7200 + rate % 97 + rank)
        barrier()  # every GPU's batcher is under load at the same time
        hb.reset_tail()
        before = hb.stats()
        dec, lat_ns, wall = hb.open_loop_requests(load, rate_per_s=rate, producers=producers)
        after = hb.stats()
        lat_us = np.sort(lat_ns[n_calls // 20:]) / 1e3
        call_us = np.sort(hb.last_call_latency[n_calls // 20:]) / 1e3
        cyc = max(after["cycles"] - before["cycles"], 1)
        q = [float(lat_us[len(lat_us) // 2]), float(lat_us[int(len(lat_us) * 0.99)]), float(lat_us[int(len(lat_us) * 0.999)])]
        if world > 1:
            t = torch.tensor(q, device=f"cuda:{local}", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            q = [float(x) for x in t]
        open_lat[str(rate)] = {"p50_us": q[0], "p99_us": q[1], "p999_us": q[2], "requests_per_gpu": n_calls, "gpus_loaded_at_once": world,
                               "generator_threads_per_gpu": producers, "cpu_quota": quota,
                               "achieved_req_per_s_rank0": n_calls / wall, "mean_batch_rank0": n_calls / cyc,
                               "us_per_cycle_rank0": {k: round((after["ns_" + k] - before["ns_" + k]) / cyc / 1e3, 1) for k in ("submit", "device", "deliver")},
                               "admitted_rank0": int((dec["reason"] == 0).sum()),
                               # the same requests on the second clock (decision - the moment the generator made the call) and what
                               # the generator threads themselves were late by: a tail that is in `p999_us` but not here is the
                               # load generator being descheduled, not the batcher or the device
                               "from_call_rank0": {"p50_us": float(call_us[len(call_us) // 2]), "p99_us": float(call_us[int(len(call_us) * 0.99)]),
                                                   "p999_us": float(call_us[int(len(call_us) * 0.999)])},
                               "generator_rank0": hb.open_loop_lateness(),
                               "batcher_tail_rank0": {k: (round(v / 1e3, 1) if k.startswith("max") else v) for k, v in after.items()
                                                      if k.startswith(("max_ns", "slow_", "late_"))}}
    # what the compiled host itself can carry: the same generator with no pacing (every producer submits as fast as the
    # batcher takes rows: one compare-and-swap + the copy of the body into the pinned block per request), decisions delivered
    # by callback. This is the end-to-end rate of the path a gRPC server would use, per-request staging copies included.
    host_peak = None
    if rank == 0 and args.latency_requests:
        now += STEP_S; hb.set_fixed_clock(now)
        load = arrivals(1_000_000, 7300)
        dec, _, wall = hb.open_loop_requests(load, rate_per_s=1e9, producers=producers)
        st = hb.stats()
        host_peak = {"req_per_s": 1_000_000 / wall, "producer_threads": producers, "mean_batch": 1_000_000 / max(st["cycles"] - after["cycles"], 1),
                     "what": "host/cpp Batcher::SubmitRequest from unpaced producer threads, 1 M requests of ~1 KiB, one GPU"}
    hb.close()

    # ---- the same step on single-shape traffic (every request / completion the same template, exactly BODY / RESP_BODY
    # bytes): the lanes of a warp then move in lock step. Reported next to the headline because the scan kernels are
    # sensitive to how much the 32 bodies of a warp differ (DESIGN.md §5) ----------------------------------------
    uniform = None
    if rank == 0:
        ureq = pin_batch(w.request_batch(args.wave, now, seed=9001, body_size=BODY, n_templates=512))
        g.select_slot(0)
        ures = pin_batch(w.response_batch(g.handle_request_body(ureq), now + 1, seed=9002, body_size=RESP_BODY))
        g.stage_request(ureq)
        g.stage_response(ures)
        now += STEP_S
        torch.cuda.synchronize()
        for _ in range(3):
            g.run_request(now); g.run_response(now + 1); now += STEP_S
        u0, u1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        u0.record(ext)
        for _ in range(20):
            g.run_request(now); g.run_response(now + 1); now += STEP_S
        u1.record(ext)
        torch.cuda.synchronize()
        uniform = {"value": args.wave * 20 / (u0.elapsed_time(u1) / 1e3), "unit": "req/s per GPU",
                   "ms_per_step": u0.elapsed_time(u1) / 20,
                   "what": f"same step, every request {BODY} B of one shape and every completion {RESP_BODY} B of one shape (best case)"}

    if world > 1:
        t = torch.tensor([dev_ms, e2e_s * 1e3], device=f"cuda:{local}", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, e2e_s = float(t[0]), float(t[1]) / 1e3
    total_req = args.steps * args.wave * world
    value = total_req / (dev_ms / 1e3)
    e2e_value = total_req / e2e_s
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    # roofline of the DOMINANT kernel (largest share of the step's device time). Algorithmic bytes per launch
    # (DESIGN.md §5): every body byte once, plus per request 64 B token/offset record + 32 B token-table probe + 24 B of
    # intermediates (request scan), or per response 17 B offsets/qos/flag + 5 x 16 B counter atomics + 26 B result.
    req_bytes = float(np.mean([int(b.body_len.sum()) + b.n * (64 + 32 + 24) for b in reqs]))
    resp_bytes = float(np.mean([int(b.body_len.sum()) + b.n * (17 + 80 + 26) for b in resps]))
    kern = {"scan_request_stage": (float(np.mean(scan_ms)), req_bytes),
            "scan_response_stage": (float(np.mean(resp_ms)), resp_bytes)}
    # the fast-path kernel of each stage on its own (it decides every body it accepts, so it carries the same per-row
    # bytes as the stage: token record + table probe + intermediates / offsets + counter atomics + result row)
    if fast_req_ms:
        kern["fast_request_kernel"] = (float(np.mean(fast_req_ms)), req_bytes)
    if fast_resp_ms:
        kern["fast_response_kernel"] = (float(np.mean(fast_resp_ms)), resp_bytes)
    single = {k: v for k, v in kern.items() if not k.endswith("_stage")} or kern  # a kernel, not a stage of several
    dom = max(single, key=lambda k: single[k][0])
    dom_s, dom_bytes = kern[dom][0] / 1e3, kern[dom][1]
    peak, how = peaks()
    achieved = dom_bytes / dom_s / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tp):  # dram__bytes_read.sum + dram__bytes_write.sum of this kernel from the committed ncu --set full capture
        traffic = json.load(open(tp)).get(dom, {}).get("dram_bytes_per_launch")
    others = {k: {"achieved": v[1] / (v[0] / 1e3) / 1e9, "frac": v[1] / (v[0] / 1e3) / 1e9 / peak,
                  "algorithmic_bytes_per_launch": v[1]} for k, v in kern.items()}
    h2d = int(np.mean([b.bodies.nbytes + b.body_off.nbytes + b.body_len.nbytes + b.tokens.nbytes + b.token_off.nbytes +
                       b.pick_rand.nbytes for b in reqs]) +
              np.mean([b.bodies.nbytes + b.body_off.nbytes + b.body_len.nbytes + b.qos.nbytes + b.flags.nbytes for b in resps]))
    d2h = int(np.mean([b.n * (3 + 12 + 16 + 12) for b in reqs]) + np.mean([b.n * 26 for b in resps]))
    out = {
        "metric": "gateway requests/s (request + response phase)", "value": value, "unit": "req/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8/int64", "data": "synthetic",
        "config": workload_config(args, world),
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "req/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": 1e3 * e2e_s / args.steps,
                # what every GPU's uploads ran at while all of them were uploading (names the limiter when the curve bends:
                # ~55 GB/s is one PCIe Gen5 x16 link; less on every rank at once = the host side of the links)
                "h2d_GBps_per_rank": [round(h2d * args.steps / t_ / 1e9, 1) for t_ in rank_e2e_s],
                "note": "pinned host buffers; asynchronous submits, two batches in flight; PCIe-bound"},
        "latency_us": {"what": "one synchronous request micro-batch through the C ABI (H2D + 2 kernels + D2H), host wall clock",
                       "by_batch_size": latency,
                       "by_concurrent_streams": streams_lat,
                       "open_loop_by_arrival_rate": open_lat,
                       "open_loop_what": "requests ARRIVE at the given rate per GPU on every GPU at once (exponential gaps, 8 producer threads per GPU) through host/cpp Batcher::SubmitRequest; latency = decision callback - scheduled arrival; worst rank's percentiles; 1 250 000/s per GPU = BASELINE's 10 M req/s over 8 GPUs, target p99 < 200 us",
                       "host_batcher_peak": host_peak,
                       "numa": numa,
                       "streams_what": "N stream threads, one blocking HandleRequestBody at a time each, through host/cpp Batcher (C++); per-call latency"},
        "gpu_launches": int(launches),
        "single_shape_traffic": uniform,
        "kernels_ms": {"scan_request_stage": float(np.mean(scan_ms)), "limit_admit": float(np.mean(admit_ms)),
                       "scan_response_stage": float(np.mean(resp_ms)),
                       "fast_scan_request": float(np.mean(fast_req_ms)) if fast_req_ms else None,
                       "fast_scan_response": float(np.mean(fast_resp_ms)) if fast_resp_ms else None,
                       "what": "stage = length ordering + fast-path kernel (mask_scan.cuh) + exact-engine pass over the bodies it declined"},
        "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic, "peak_source": how,
                     "algorithmic_bytes_per_launch": dom_bytes, "per_kernel": others},
        "body_bytes_over_8TBps": (float(np.mean([int(b.body_len.sum()) for b in reqs])) +
                                  float(np.mean([int(b.body_len.sum()) for b in resps]))) * args.steps * world / (dev_ms / 1e3) / 8e12,
    }
    # ---- the BPE count kernels (north star side output; DESIGN.md section 9) on the same waves, timed by the library's own events
    # around bpe_scan_kernel + bpe_merge_kernel. Last GPU work of the run and self-contained: a failure here is reported
    # in the key and costs nothing else.
    if not args.no_bpe and world == 1:  # a one-GPU measurement: the scaling runs do not repeat it
        try:
            out["bpe"] = bpe_section(g, w, reqs, resps, now, peak, ext)
        except Exception as e:  # noqa: BLE001
            out["bpe"] = {"error": f"{type(e).__name__}: {e}"[:400]}
    if shared_quota:
        out["shared_quota"] = shared_quota
        out["config"]["parallelism"] += f" + {shared_quota['rows']} shared quotas folded every {args.fold_every} steps"
    if not args.no_cpu_baseline:
        out["cpu_baseline"], _ = cpu_arm(args, 1, seconds=12.0)
    print(json.dumps(out), file=real_stdout, flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
