#!/usr/bin/env python
"""bench.py -- utterances/sec of the CTC beam-search hot path on BASELINE.json's config 2
([256, T=1000, V=29] per GPU, beam 100, cutoff_top_n 40, cutoff_prob 1.0, no LM; synthetic CTC-like input).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config c2|c3|c4|c5]
                    [--dump-outputs DIR]

One process per GPU (torchrun sets RANK / LOCAL_RANK / WORLD_SIZE); utterances are independent, so each
rank decodes its own [256, T, V] shard and there is no data-path collective ("weak" scaling, N=8 is
BASELINE config 3: 2048 utterances over 8 GPUs).  Rank 0 prints ONE JSON line:

  value        whole-job utterances/s with inputs resident in HBM (device entry point of the C ABI), CUDA-event
               time of K steps, max over ranks; L2 is flushed between timed steps
  e2e          same metric through the host-buffer C-ABI call: pinned host probs -> H2D -> kernels -> D2H of the
               results into pinned host tensors, wall clock around the call, max over ranks (the call pipelines
               groups of utterances over streams: copies of one group overlap the kernels of the others)
  roofline     beam-search kernel: algorithmic bytes (B*T*V*4, SURVEY.md 8d) / its CUDA-event duration,
               against MEASURED_PEAKS.json's HBM copy bandwidth.  The kernel is T-serial per utterance
               (latency bound), so the fraction is tiny by construction; `scan` reports the HBM-bound
               prune/log pre-pass the same way.
  cpu_baseline the reference's own CPU path (oracle/_ref: unmodified reference sources, ThreadPool over all
               host cores; falls back to the single-threaded C port if that build is absent) on a bounded
               sample of the same batch

--impl reference times only that CPU path and prints the same line shape with "impl": "reference".
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    "c2": dict(B=256, T=1000, V=29, beam=100, cutoff_top_n=40, cutoff_prob=1.0,
               name="config2: [256 x T=1000 x V=29] per GPU, beam 100, cutoff_top_n 40, cutoff_prob 1.0, no LM"),
    # BASELINE config 3: a FIXED total of 2048 utterances, split over the ranks ("strong" scaling: 1 GPU runs ~7 waves
    # of CTAs, 8 GPUs one wave each -- SURVEY.md 8e)
    "c3": dict(B=2048, T=1000, V=29, beam=100, cutoff_top_n=40, cutoff_prob=1.0, strong=True,
               name="config3: [2048 x T=1000 x V=29] in total, split over the GPUs, beam 100, cutoff_top_n 40, cutoff_prob 1.0, no LM"),
    "c4": dict(B=256, T=2000, V=256, beam=200, cutoff_top_n=40, cutoff_prob=0.99,
               name="config4: [256 x T=2000 x V=256] per GPU, beam 200, cutoff_top_n 40, cutoff_prob 0.99, no LM"),
    # BASELINE config 5: KenLM scorer path with the reference's own test LM (its tests/test.arpa, kept as the fixture
    # tests/golden/test.arpa); the posteriors noisily spell sentences over that model's vocabulary.
    "c5": dict(B=64, T=1000, V=29, beam=100, cutoff_top_n=40, cutoff_prob=1.0, lm=True, alpha=2.0, beta=1.0,
               name="config5: [64 x T=1000 x V=29], beam 100, KenLM scorer hook (tests/test.arpa, alpha 2.0, beta 1.0)"),
}
L29 = ["_"] + [chr(ord("a") + i) for i in range(26)] + [" ", "'"]
TINY_LM = os.path.join(ROOT, "tests", "golden", "test.arpa")  # (name kept: tools/ import it) the reference's test LM
PROVIDER = os.path.join(ROOT, "providers", "_build", "libkenlm_provider.so")


def c5_inputs(B, T, seed):
    """Random sentences over the vocabulary of the reference's test.arpa, ~T/5 characters each."""
    import random
    from ctcdecode_b200.synth import text_probs
    rng = random.Random(seed)
    words = ["a", "also", "beyond", "call", "concerns", "consider", "for", "higher", "however", "i", "in", "is", "little",
             "loin", "look", "looking", "more", "on", "screening", "small", "the", "to", "watch", "what", "would"]
    texts = []
    for _ in range(B):
        s = ""
        while len(s) < T // 5:
            s += (" " if s else "") + rng.choice(words)
        texts.append(s[: T // 4])
    return text_probs(texts, L29, T, seed=seed)


METRIC = "utterances/sec at beam_width=100, T=1000, V=29; HBM GB/s vs roofline"


def traffic_of(config, kernel):
    """DRAM bytes per launch of `kernel` from the committed ncu capture of this config (profiles/traffic.json, written
    by tools/ncu_traffic.py from an `ncu --set full` report), or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            e = json.load(f)[config][kernel]
        return e["dram_read_bytes"] + e["dram_write_bytes"], e["source"]
    except Exception:  # noqa: BLE001
        return None, None


def pin_to_gpu_numa_node(index):
    """One process per GPU, N of them on one host: run this rank on the cores of the NUMA node its GPU hangs off, so
    that its pinned host buffers (first touch) and the threads that fill them are local to the GPU's PCIe root --
    what a production launcher does with numactl.  Best effort: any failure leaves the affinity as it was."""
    try:
        import torch
        bus = torch.cuda.get_device_properties(index).pci_bus_id
        dom = getattr(torch.cuda.get_device_properties(index), "pci_domain_id", 0)
        dev_id = torch.cuda.get_device_properties(index).pci_device_id
        path = "/sys/bus/pci/devices/%04x:%02x:%02x.0/numa_node" % (dom, bus, dev_id)
        node = int(open(path).read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        return node
    except Exception:  # noqa: BLE001
        return None


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:  # noqa: BLE001
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:  # noqa: BLE001
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


_REF_CACHE = {}


def reference_cpu(probs_np, cfg, n_utts, threads):
    """Times the reference's CPU path on the first n_utts utterances.  Returns (seconds, kind)."""
    from oracle import oracle as orc
    sample = probs_np[:n_utts]
    if cfg.get("lm"):
        if "lm" not in _REF_CACHE:
            _REF_CACHE["lm"] = orc.Reference(L29, model_path=TINY_LM, alpha=cfg["alpha"], beta=cfg["beta"])
        ref = _REF_CACHE["lm"]
        t0 = time.perf_counter()
        ref.decode(sample, beam=cfg["beam"], cutoff_prob=cfg["cutoff_prob"], cutoff_top_n=cfg["cutoff_top_n"],
                   num_processes=threads)
        return time.perf_counter() - t0, "reference"
    if orc.reference_available():
        ref = orc.Reference([str(i) for i in range(cfg["V"])])
        t0 = time.perf_counter()
        ref.decode(sample, beam=cfg["beam"], cutoff_prob=cfg["cutoff_prob"], cutoff_top_n=cfg["cutoff_top_n"],
                   num_processes=threads)
        return time.perf_counter() - t0, "reference"
    cp = orc.CPort()
    t0 = time.perf_counter()
    cp.decode(sample, beam=cfg["beam"], cutoff_prob=cfg["cutoff_prob"], cutoff_top_n=cfg["cutoff_top_n"])
    return time.perf_counter() - t0, "port"


def reference_outputs(probs_np, cfg, n_utts, threads):
    """The reference's results for the first n_utts utterances (no-LM configurations).  Returns (outputs, kind)."""
    from oracle import oracle as orc
    sample = probs_np[:n_utts]
    kw = dict(beam=cfg["beam"], cutoff_prob=cfg["cutoff_prob"], cutoff_top_n=cfg["cutoff_top_n"])
    if orc.reference_available():
        return orc.Reference([str(i) for i in range(cfg["V"])]).decode(sample, num_processes=threads, **kw), "reference"
    return orc.CPort().decode(sample, **kw), "port"


def bench_lm(args, cfg, config, rank, world, local_rank, dev, K, W, cores):
    """Config 5: the scorer path is a host-buffer API (the LM hook lives on the host), so value == e2e."""
    import torch
    import torch.distributed as dist
    from ctcdecode_b200 import CTCBeamDecoder
    B, T = cfg["B"], cfg["T"]
    probs = c5_inputs(B, T, rank)
    dec = CTCBeamDecoder(L29, model_path=TINY_LM, alpha=cfg["alpha"], beta=cfg["beta"], beam_width=cfg["beam"],
                         cutoff_top_n=cfg["cutoff_top_n"], cutoff_prob=cfg["cutoff_prob"], scorer_provider=PROVIDER,
                         device="cuda:%d" % local_rank)
    for _ in range(W):
        out = dec.decode(probs)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(K):
        out = dec.decode(probs)
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.destroy_process_group()
    if rank != 0:
        return
    val = B * world * K / float(t[0])
    top1 = "".join(L29[x] for x in out[0][0, 0, :out[3][0, 0]])
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, tokens=out[0].numpy(), timesteps=out[2].numpy(), scores=out[1].numpy(),
                     lens=out[3].numpy(), n_results=dec.last_n_results.numpy(), flags=dec.last_flags.numpy())
    line = {"metric": METRIC, "value": val, "unit": "utterances/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": 1e3 * float(t[0]) / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": config,
            "e2e": {"value": val, "unit": "utterances/s", "h2d_bytes_per_step": B * T * 29 * 4,
                    "d2h_bytes_per_step": int(2 * B * cfg["beam"] * int(out[3].max()) * 4 + 2 * B * cfg["beam"] * 4),
                    "note": "host-buffer API: the LM hook runs on the host, once per frame, inside one persistent "
                            "launch (per-frame handshake through mapped host memory); value == e2e"},
            "gpu_launches": K * (T + 2 if os.environ.get("CTCDEC_LM_PER_FRAME") else 3), "roofline": None,
            "sample_top1": top1}
    if world == 1 and not args.no_cpu_baseline:
        n = max(1, min(B, cores))
        dtr, kind = reference_cpu(probs.numpy(), cfg, n, cores)
        line["cpu_baseline"] = {"value": n / dtr, "unit": "utterances/s", "cores": cores, "kind": kind,
                                "sample": "the first %d utterances of the same batch, reference Scorer path" % n}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-strong", action="store_true", help="skip the fixed-2048 (BASELINE config 3) leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the results of the last timed step to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    cfg = CONFIGS[args.config]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    K, W = args.steps, max(args.warmup, 3 if args.impl == "ours" else 0)
    B, T, V = cfg["B"], cfg["T"], cfg["V"]
    scaling = "weak"
    if cfg.get("strong"):  # fixed global batch: every rank takes its contiguous share
        scaling = "strong"
        B = B // world
    cores = len(os.sched_getaffinity(0))
    config = {"workload": cfg["name"], "batch_per_gpu": B, "global_batch": B * world, "T": T, "V": V,
              "beam_width": cfg["beam"], "cutoff_top_n": cfg["cutoff_top_n"], "cutoff_prob": cfg["cutoff_prob"],
              "parallelism": "batch-sharded x%d (no data-path collective)" % world,
              "l2": "flushed between timed steps (256 MiB write)"}

    from ctcdecode_b200.synth import ctc_like_probs

    # ------------------------------------------------------------------------------------------------------
    if args.impl == "reference":
        if rank != 0:
            return
        probs = (c5_inputs(B, T, 0) if cfg.get("lm") else ctc_like_probs(B, T, V, seed=0)).numpy()
        n = max(1, min(B, cores))  # one utterance per host thread per step
        times, kind = [], "reference"
        for i in range(W + K):
            dt, kind = reference_cpu(probs, cfg, n, cores)
            if i >= W:
                times.append(dt)
        total = sum(times)
        val = n * K / total
        sample = "%d of the %d utterances of the same seeded batch per step (one per host thread)" % (n, B)
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": val, "unit": "utterances/s", "n_gpus": args.gpus,
            "steps": K, "warmup": W, "ms_per_step": 1e3 * total / K, "higher_is_better": True, "scaling": scaling,
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
            "cpu_baseline": {"value": val, "unit": "utterances/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": val, "unit": "utterances/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    # ------------------------------------------------------------------------------------------------------
    import torch
    import torch.distributed as dist
    from ctcdecode_b200 import _native

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        pin_to_gpu_numa_node(local_rank)  # before any pinned allocation: first touch puts the buffers next to the GPU
    if world > 1:
        # keep stdout for the one JSON line: NCCL prints its version line (NCCL_DEBUG=WARN / VERSION) to stdout when the
        # communicator comes up, so file descriptor 1 points at stderr until the first collective has run
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
    lib = _native.load()
    if cfg.get("lm"):
        return bench_lm(args, cfg, config, rank, world, local_rank, dev, K, W, cores)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()  # (before the warm-up: a 10-step timed region is only ~50 ms, a sample every 100 ms)
    m = measure(lib, dev, local_rank, cfg, B, rank, K, W, barrier)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, **{k: v.cpu().numpy() for k, v in m["device"].items()})
    # BASELINE config 3 beside it (SURVEY.md 8e): a FIXED total of 2048 utterances split over the ranks, so that the
    # driver's N = 1, 2, 4, 8 runs carry the strong-scaling curve next to the weak one
    strong = None
    if args.config == "c2" and not args.no_strong:
        c3 = CONFIGS["c3"]
        strong = measure(lib, dev, local_rank, c3, c3["B"] // world, 1000 + rank, K, 3, barrier)

    # ---- reduce over ranks (max time) ----------------------------------------------------------------------------
    vals = [m["total_ms"], m["e2e_ms"], float(m["n_err"]), float(m["n_tie"]), 0.0 if m["same"] else 1.0]
    if strong:
        vals += [strong["total_ms"], strong["e2e_ms"], float(strong["n_err"]), 0.0 if strong["same"] else 1.0]
    t = torch.tensor(vals, device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms_max, e2e_ms_max = float(t[0]), float(t[1])
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    kern_ms, total_ms = m["kern_ms"], m["total_ms"]
    Kb = cfg["beam"]
    value = B * world * K / (total_ms_max / 1e3)
    e2e_val = B * world * K / (e2e_ms_max / 1e3)
    peak, peak_src = peaks()
    beam_ms = statistics.mean(k[1] for k in kern_ms)
    scan_ms = statistics.mean(k[0] for k in kern_ms)
    fin_ms = statistics.mean(k[2] for k in kern_ms)
    alg_bytes = B * T * V * 4
    achieved = alg_bytes / (beam_ms * 1e-3) / 1e9
    # the scan reads the [B,T,V] input once and writes the pruned rows (NP floats, + NP uint16 when the
    # vocabulary is cut): its bytes per launch
    is_sorted = cfg["cutoff_prob"] < 1.0 or cfg["cutoff_top_n"] < V
    n_max = min(V, max(1, cfg["cutoff_top_n"])) if is_sorted else V
    NP = (n_max + 3 + 7) // 8 * 8
    scan_bytes = alg_bytes + B * T * NP * (6 if is_sorted else 4)
    beam_traffic, beam_traffic_src = traffic_of(args.config, "beam_kernel") if B == cfg["B"] else (None, None)
    scan_traffic, _ = traffic_of(args.config, "prune_kernel") if B == cfg["B"] else (None, None)
    line = {
        "metric": METRIC, "value": value, "unit": "utterances/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": total_ms_max / K, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": config,
        "e2e": {"value": e2e_val, "unit": "utterances/s", "h2d_bytes_per_step": m["h2d"], "d2h_bytes_per_step": m["d2h"],
                "ms_per_step": e2e_ms_max / K, "host_equals_device": bool(float(t[4]) == 0.0)},
        "gpu_launches": 3 * K,
        "kernels_ms": {"prune_log_scan": scan_ms, "beam_search": beam_ms, "finalize": fin_ms,
                       "beam_share_of_step": beam_ms * K / total_ms},
        "roofline": {"kernel": "beam_kernel", "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": beam_traffic, "traffic_source": beam_traffic_src,
                     "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": alg_bytes,
                     "ns_per_frame_per_cta": beam_ms * 1e6 / T,
                     "note": "T-serial per utterance: latency bound, far below the HBM roofline by construction",
                     "scan": {"kernel": "prune_kernel", "bound": "fp64 issue (exact glibc log per element), then hbm",
                              "bytes_per_launch": scan_bytes, "traffic": scan_traffic,
                              "achieved": scan_bytes / (scan_ms * 1e-3) / 1e9,
                              "unit": "GB/s", "frac": scan_bytes / (scan_ms * 1e-3) / 1e9 / peak}},
        "clocks": clocks,
        "parity": {"arena_errors": int(t[2]), "tie_flagged_utterances_max_per_rank": int(t[3])},
    }
    if strong:
        gb = CONFIGS["c3"]["B"] // world * world
        ks = K
        line["strong_c3"] = {
            "workload": CONFIGS["c3"]["name"], "global_batch": gb, "batch_per_gpu": gb // world, "steps": ks,
            "value": gb * ks / (float(t[5]) / 1e3), "unit": "utterances/s", "ms_per_step": float(t[5]) / ks,
            "e2e": {"value": gb * ks / (float(t[6]) / 1e3), "unit": "utterances/s", "ms_per_step": float(t[6]) / ks,
                    "h2d_bytes_per_step": strong["h2d"], "d2h_bytes_per_step": strong["d2h"],
                    "host_equals_device": bool(float(t[8]) == 0.0)},
            "arena_errors": int(t[7]),
            "kernels_ms": {"prune_log_scan": statistics.mean(k[0] for k in strong["kern_ms"]),
                           "beam_search": statistics.mean(k[1] for k in strong["kern_ms"]),
                           "finalize": statistics.mean(k[2] for k in strong["kern_ms"])},
            "note": "fixed total of 2048 utterances split over the ranks (strong scaling); time = max over ranks"}
    if world == 1 and not args.no_cpu_baseline:
        line.update(cpu_legs(m, cfg, cores))
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def measure(lib, dev, local_rank, cfg, B, seed, K, W, barrier):
    """W warm-up + K timed steps of one workload on this rank, device-resident (CUDA events, L2 flushed between steps)
    and end to end through the host entry point (pinned host buffers, wall clock).  Returns the raw times and the
    tensors of the last step."""
    import torch
    from ctcdecode_b200 import _native
    from ctcdecode_b200.synth import ctc_like_probs
    T, V, Kb = cfg["T"], cfg["V"], cfg["beam"]
    probs_cpu = ctc_like_probs(B, T, V, seed=seed)  # every rank its own shard of the global batch
    probs_dev = probs_cpu.to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    _native.check(lib.ctcdec_profile_enable(1))
    ms3 = (ctypes.c_float * 3)()

    # ---- value: inputs resident in HBM, the C ABI's device entry point on torch's current stream -----------------
    ccfg = _native.Config(V, Kb, 0, 0, cfg["cutoff_top_n"], float(cfg["cutoff_prob"]))
    ws_bytes = ctypes.c_size_t(0)
    _native.check(lib.ctcdec_workspace_bytes(ctypes.byref(ccfg), B, T, ctypes.byref(ws_bytes)))
    ws = torch.empty(ws_bytes.value, dtype=torch.uint8, device=dev)
    d_tok = torch.empty(B, Kb, T, dtype=torch.int32, device=dev)
    d_ts = torch.empty(B, Kb, T, dtype=torch.int32, device=dev)
    d_sc = torch.empty(B, Kb, dtype=torch.float32, device=dev)
    d_len = torch.zeros(B, Kb, dtype=torch.int32, device=dev)
    d_nres = torch.zeros(B, dtype=torch.int32, device=dev)
    d_flags = torch.zeros(B, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream

    def device_step():
        _native.check(lib.ctcdec_decode_batch_device(
            ctypes.byref(ccfg), probs_dev.data_ptr(), None, B, T, d_tok.data_ptr(), d_ts.data_ptr(), d_sc.data_ptr(),
            d_len.data_ptr(), d_nres.data_ptr(), d_flags.data_ptr(), ws.data_ptr(), ws.numel(), stream))

    for _ in range(W):
        device_step()
    torch.cuda.synchronize()
    barrier()
    step_ms, kern_ms = [], []
    for _ in range(K):
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        device_step()
        e1.record()
        e1.synchronize()
        step_ms.append(e0.elapsed_time(e1))
        _native.check(lib.ctcdec_profile_read(ms3))
        kern_ms.append(list(ms3))
    barrier()
    total_ms = sum(step_ms)
    n_err = int((d_flags & 256).sum())
    n_tie = int(((d_flags & 7) != 0).sum())

    # ---- e2e: host buffers through the C-ABI host entry point -------------------------------------------------
    h_probs = probs_cpu.pin_memory()
    h_tok = torch.empty(B, Kb, T, dtype=torch.int32).pin_memory()
    h_ts = torch.empty(B, Kb, T, dtype=torch.int32).pin_memory()
    h_sc = torch.empty(B, Kb, dtype=torch.float32).pin_memory()
    h_len = torch.zeros(B, Kb, dtype=torch.int32).pin_memory()
    h_nres = torch.zeros(B, dtype=torch.int32).pin_memory()
    h_flags = torch.zeros(B, dtype=torch.int32).pin_memory()

    def host_step():
        _native.check(lib.ctcdec_decode_batch_host(ctypes.byref(ccfg), h_probs.data_ptr(), None, B, T,
                                                   h_tok.data_ptr(), h_ts.data_ptr(), h_sc.data_ptr(),
                                                   h_len.data_ptr(), h_nres.data_ptr(), h_flags.data_ptr(),
                                                   local_rank))

    for _ in range(W):
        host_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        host_step()
    e2e_s = time.perf_counter() - t0
    barrier()
    max_len = int(h_len.max())
    h2d = B * T * V * 4
    d2h = 2 * B * Kb * max_len * 4 + 2 * B * Kb * 4 + 2 * B * 4
    # sanity: host path and device path agree
    same = bool(torch.equal(h_sc, d_sc.cpu()) and torch.equal(h_len, d_len.cpu()))
    return dict(total_ms=total_ms, e2e_ms=e2e_s * 1e3, kern_ms=kern_ms, n_err=n_err, n_tie=n_tie, same=same, h2d=h2d,
                d2h=d2h, probs_cpu=probs_cpu,
                device=dict(tokens=d_tok, timesteps=d_ts, scores=d_sc, lens=d_len, n_results=d_nres, flags=d_flags),
                host=dict(tokens=h_tok.numpy(), timesteps=h_ts.numpy(), scores=h_sc.numpy(), lens=h_len.numpy(),
                          n_results=h_nres.numpy(), ties=h_flags.numpy()))


def dump_outputs(directory, tokens, timesteps, scores, lens, n_results, flags):
    """Writes the results of the last timed step as float32 DIR/<name>.npy, so that two builds can be compared output
    for output (the inputs are seeded): scores, lens, n_results and flags of every utterance, and tokens / timesteps of
    a fixed, seeded sample of utterances (sample_utterances) that keeps the files under ~50 MB in all.  Rows past an
    utterance's n_results and steps past a beam's length hold no result: they are written as 0 and -1."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    B, beam, T = tokens.shape
    n_results = n_results.astype(np.int64)
    row = np.arange(beam)[None, :] < n_results[:, None]
    lens = np.where(row, lens, 0)
    k = max(1, min(B, (48 << 20) // (beam * T * 8)))
    idx = np.sort(np.random.default_rng(0).choice(B, k, replace=False))
    step = np.arange(T)[None, None, :] < lens[idx][:, :, None]
    out = {"scores": np.where(row, scores, 0.0), "lens": lens, "n_results": n_results, "flags": flags,
           "sample_utterances": idx, "tokens": np.where(step, tokens[idx], -1),
           "timesteps": np.where(step, timesteps[idx], -1)}
    for name, a in out.items():
        np.save(os.path.join(directory, name + ".npy"), np.asarray(a, np.float32))


def cpu_legs(m, cfg, cores):
    """cpu_baseline (the reference's CPU path on a bounded sample of the same batch, all host threads; plus one thread
    and a mid-size pool, so that the CPU's best is on record) and the parity block: the reference outputs of that
    sample against what the CUDA path returned for the same utterances (host entry point), through tests/parity."""
    from tests import parity
    probs = m["probs_cpu"].numpy()
    B = probs.shape[0]
    n = max(1, min(B, max(cores, 128)))  # at least 128 utterances go through the comparison
    t0 = time.perf_counter()
    ref, kind = reference_outputs(probs, cfg, n, cores)
    spent, reps = time.perf_counter() - t0, 1
    while spent < 10.0 and reps < 8:
        d2, _ = reference_cpu(probs, cfg, n, cores)
        spent += d2
        reps += 1
    out = {"cpu_baseline": {"value": n * reps / spent, "unit": "utterances/s", "cores": cores if kind == "reference" else 1,
                            "kind": kind, "threads": cores if kind == "reference" else 1,
                            "sample": "%d x the first %d utterances of the same batch, ThreadPool of %d" % (reps, n, cores)}}
    if kind == "reference":
        alt = []
        for th, nu in ((1, 2), (max(2, min(32, cores // 4)), max(2, min(32, cores // 4)))):
            d, _ = reference_cpu(probs, cfg, nu, th)
            alt.append({"threads": th, "utterances": nu, "value": nu / d})
        out["cpu_baseline"]["other_pool_sizes"] = alt
        best = max([out["cpu_baseline"]["value"]] + [a["value"] for a in alt])
        out["cpu_baseline"]["best_pool_value"] = best
    cnt = parity.count(ref, m["host"], None, n)
    cnt["against"] = "oracle/_ref (unmodified reference build)" if kind == "reference" else "oracle C port"
    cnt["utterances"] = n
    return {"cpu_baseline": out["cpu_baseline"], "parity_vs_reference": cnt}


if __name__ == "__main__":
    main()
