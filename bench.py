#!/usr/bin/env python
"""bench.py — input-assembly Mbp/s through compress -> unitig GFA (BASELINE.json's metric).

A "step" is one pass of the hot path over one batch of synthetic input assemblies (compress.rs:42-47, `ac_compress`):
padded, end-repaired strands  ->  k-mer table, unitigs, links, repeat expansion, renumbering, GFA text (ONE pipeline of B200 kernels)
->  the bytes of input_assemblies.gfa in pinned host memory.  Every timed run is gated on the oracle's committed SHA-256 of that file.

  python bench.py [--gpus N] [--steps K] [--warmup W]          the CUDA path through the C ABI (N > 1: torchrun, BASELINE config 5's first 8N assemblies)
  python bench.py --impl reference [...]                        the reference's CPU algorithm (oracle port, -O3 -march=native), 1 core, the SAME full-size input

`value`  : Mbp/s with the strands already resident in HBM when the timed region starts.
`e2e`    : the same, with the strands copied from pinned host memory inside the timed region (the call a user makes).
`roofline`: the hash-insert kernel alone (events right around its launch) against the measured HBM copy peak (MEASURED_PEAKS.json).
`cli_wall`: `autocycler compress` from process start to both files closed (stage A, CUDA context and file I/O included).

--dump-outputs DIR writes what the last timed step returned (dump_outputs), so that two builds can be compared output for output.
The bench writes nothing into the tree it runs from: the tree may be read-only.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "input-assembly Mbp/sec through compress->unitig GFA"
K = 51
WORKLOADS = {   # BASELINE.json configs (SURVEY.md §8d generator); the default is the config the metric is quoted on
    "cfg1": "cfg1: 3 synthetic 100 kbp assemblies",
    "cfg2": "cfg2: 8 synthetic E. coli-sized (4.64 Mbp) assemblies",
    "cfg3": "cfg3: 12 synthetic K. pneumoniae-sized assemblies (5.5 Mbp chromosome + 5 plasmids)",
    "cfg4": "cfg4: 24 synthetic 10 Mbp assemblies",
    "cfg5": "cfg5: 64 synthetic 5 Mbp assemblies, 8 per rank",
}
WORKLOAD = WORKLOADS["cfg2"] + ", k=51"


INSERT_BODY = "InsertBody"          # pipeline.cu: the k-mer hash insert, one window per thread, 32-byte slot groups


def measured_traffic(kernel):
    """DRAM bytes per launch of `kernel` from the committed `ncu --set full` capture (profiles/kernel_traffic.json, written by
    profiles/extract_traffic.py from the .ncu-rep): dram__bytes_read.sum + dram__bytes_write.sum.  None if no capture matches."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "kernel_traffic.json")))
        return t.get(kernel, {}).get("dram_bytes")
    except Exception:
        return None


def golden_for(key):
    """SHA-256 of the oracle's GFA for a named input (tests/golden/config_goldens.json, made by tests/golden/make_config_goldens.py)."""
    try:
        return json.load(open(os.path.join(ROOT, "tests", "golden", "config_goldens.json")))[key]["sha256"]
    except Exception:
        return None


DUMP_GFA_MAX = 15_000_000      # bytes of GFA text dumped as float32: 60 MB, under the 64 MB the dump may take


def dump_outputs(directory, gfa, counts):
    """What the timed path returned in its last step, as float arrays: gfa.npy holds the bytes of input_assemblies.gfa (all of them up
    to DUMP_GFA_MAX, else that many at positions drawn with a fixed seed from the file's length, in file order) and gfa_size.npy their
    number; graph_counts.npy holds the k-mers, unitigs, links and total unitig length of the graph."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    text = np.frombuffer(bytes(gfa), dtype=np.uint8)
    if text.size > DUMP_GFA_MAX:
        text = text[np.sort(np.random.default_rng(0).choice(text.size, DUMP_GFA_MAX, replace=False))]
    np.save(os.path.join(directory, "gfa.npy"), text.astype(np.float32))
    np.save(os.path.join(directory, "gfa_size.npy"), np.array([len(gfa)], dtype=np.float64))
    np.save(os.path.join(directory, "graph_counts.npy"), np.array(counts, dtype=np.float64))


def measured_peak():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md's clocks line).  NVML is polled from a
    thread every 5 ms (the timed region lasts a few hundred ms; `nvidia-smi -lms` needs longer than that to print its first
    line); if NVML is unavailable the recipe's `nvidia-smi --query-gpu` loop is used instead."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index=0):
        self.index, self.samples, self.proc, self.stop_flag, self.thread, self.max_mhz, self.source = index, [], None, False, None, None, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))

            def poll():
                while not self.stop_flag:
                    try:
                        mhz = int(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                        try:
                            mask = int(pynvml.nvmlDeviceGetCurrentClocksEventReasons(h))
                        except Exception:
                            mask = int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                        self.samples.append((mhz, mask))
                    except Exception:
                        pass
                    time.sleep(0.005)
            self.source = "nvml"
            self.thread = threading.Thread(target=poll, daemon=True); self.thread.start()
            return
        except Exception:
            self.source = None
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.source = "nvidia-smi"
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        inv = {v: k for k, v in self.REASONS.items()}
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            if len(f) >= 6 and f[0].isdigit():
                if f[1].isdigit():
                    self.max_mhz = max(self.max_mhz or 0, int(f[1]))
                self.samples.append((int(f[0]), sum(inv[names[i]] for i in range(4) if f[2 + i].lower().startswith("active"))))

    def stop(self):
        self.stop_flag = True
        if self.thread:
            self.thread.join(timeout=1)
        if self.proc:
            self.proc.terminate()
        sm = sorted(m for m, _ in self.samples)
        reasons = sorted({name for _, mask in self.samples for bit, name in self.REASONS.items() if mask & bit})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz, "reasons": reasons, "samples": len(sm), "source": self.source}


def bind_to_gpu_numa_node(index):
    """One process per GPU, kept on the CPU socket the GPU hangs off: the pinned result buffers are then local both to the DMA
    engine and to the host threads that edit them (what `numactl --cpunodebind` would do; the threads the library creates
    inherit the mask).  Returns the node, or None when the topology cannot be read (then nothing is changed)."""
    if os.environ.get("AC_BENCH_NO_NUMA_BIND"):
        return None
    try:
        import pynvml
        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(index)).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:                 # NVML prints an 8-digit PCI domain, sysfs a 4-digit one
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if len(cpus) < 8:
            return None
        os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


def prepare_sequences(assemblies, k, threads=8):
    """Stage A on the host (FASTA -> padded, end-repaired strands) happens once, outside the timed region, through
    the product's own loader; returns [Sequence]."""
    import tempfile
    from autocycler_b200 import api, synth
    with tempfile.TemporaryDirectory() as d:
        synth.write_assemblies(assemblies, d)
        kg, seqs, count = api.load_sequences(d, k, threads=threads)
    return kg, seqs, count


def run_gpu(args):
    import torch
    import torch.distributed as dist
    from autocycler_b200 import api, synth

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    numa_node = bind_to_gpu_numa_node(local)          # before the library creates threads or pinned memory
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the GPU path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run --nproc-per-node {args.gpus}")
    from autocycler_b200 import dist as acdist
    # Weak scaling: 8 assemblies of the cfg2 genome per rank (N=1 is exactly cfg2; N=8 is 64 assemblies, the shape of cfg5).
    # Every rank stages all sequences (SURVEY 8e: end repair needs all of them anyway) and owns a contiguous block.
    global K, WORKLOAD
    K = args.k
    # N = 1: the configuration the metric is quoted on (cfg2).  N > 1: BASELINE config 5 — the first 8N assemblies of the cfg5
    # generator, 8 per rank; N = 8 is cfg5 itself.  Every workload has a committed oracle hash (tests/golden/config_goldens.json).
    workload, per_rank, n_assemblies, golden_key, WORKLOAD = workload_for(args, world)
    args.workload = workload
    assemblies = synth.make_assemblies(workload, n_assemblies=n_assemblies)
    n_bases = synth.total_bases(assemblies)
    # One stream for everything that is timed: the library's kernels and copies, NCCL's ordering (ProcessGroupNCCL orders each collective
    # against the current stream) and the CUDA events.  A stream of its own rather than the default one: nothing else in the process can
    # serialise against it.
    stream = torch.cuda.Stream(device=local)
    torch.cuda.set_stream(stream)
    # stage A once, untimed: product loader + end repair, then a handle bound to torch's current stream
    _, seqs, count = prepare_sequences(assemblies, K)
    kg = api.KmerGraph(K, device=local, stream=stream.cuda_stream)
    kg.add_sequences(seqs, count, upload=False)          # strands staged in pinned host memory
    lib = kg._h.lib
    dev = torch.device("cuda", local)
    # sequences of assemblies [8*rank, 8*rank+8): contiguous because files are loaded in sorted order
    first_of = {}
    for i, sq in enumerate(seqs):
        first_of.setdefault(sq.filename, i)
    files = sorted(first_of, key=first_of.get)
    bounds = [first_of[f] for f in files] + [len(seqs)]
    seq_lo, seq_hi = bounds[per_rank * rank], bounds[per_rank * (rank + 1)]

    rank_bounds = [bounds[per_rank * r] for r in range(world)] + [len(seqs)]

    def step(upload):
        if upload and world == 1:
            kg.upload()
        elif upload:                 # every rank copies its own strands host -> device; the others' arrive over NVLink
            acdist.upload_sharded(kg, rank_bounds, dev)
        if world == 1:
            g = api.UnitigGraph.compress(kg)                 # compress.rs:42-47 in one call: k-mer graph -> unitig graph -> simplify -> GFA text
        else:
            st = {}
            # the same, sharded: one all-gather of k-mer buckets, rank 0 finishes the graph and prints H/S/L, every rank prints its own P lines
            g, lines = acdist.compress_distributed_split(kg, seq_lo, seq_hi, dev, stats=st)
            exchange_stats.append(st)
            return g, (g.gfa_view() if g is not None else memoryview(b""), lines.view())
        return g, (g.gfa_view(), memoryview(b""))

    exchange_stats = []
    step_walls = []          # host clock of every timed step, per loop: where a rank waits shows up as a long step on the OTHER ranks' stages

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    kg.upload()
    for _ in range(args.warmup):
        step(True)

    def timed(upload):
        exchange_stats.clear()
        ins, dev, launches0 = [], [], kg_launches()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        last = None
        walls = []
        for _ in range(args.steps):
            w0 = time.perf_counter()
            g, gfa = step(upload)
            t = api.AcTimings(); lib.ac_timings_get(kg._h.ptr, t)
            ins.append(t.insert_kernel or t.insert); dev.append(t.as_dict()); last = (g, gfa, t)      # the hash-insert kernel alone, CUDA events right around its launch on the library's stream
            walls.append(round((time.perf_counter() - w0) * 1e3, 3))
        step_walls.append(walls)
        e1.record(stream)
        barrier()
        ms = e0.elapsed_time(e1)
        for st in exchange_stats:
            acdist.finish_stats(st)
        if world > 1:
            tt = torch.tensor([ms], device="cuda"); dist.all_reduce(tt, op=dist.ReduceOp.MAX); ms = float(tt.item())
        return ms, ins, dev, last, kg_launches() - launches0, list(exchange_stats)

    def kg_launches():
        t = api.AcTimings(); lib.ac_timings_get(kg._h.ptr, t); return t.kernel_launches

    sampler = ClockSampler(local); sampler.start()
    if os.environ.get("AC_BENCH_E2E_FIRST"):                                   # comparison only: the two timed loops in the other order
        ms_e2e, _, _, last2, _, _ = timed(upload=True)
        ms_res, ins_ms, dev_t, last, launches, xstats = timed(upload=False)
    else:
        ms_res, ins_ms, dev_t, last, launches, xstats = timed(upload=False)      # inputs resident in HBM
        ms_e2e, _, _, last2, _, _ = timed(upload=True)                           # host buffers -> GFA bytes on the host
    clocks = sampler.stop()
    per_rank = None
    if world > 1:          # every rank's view of the sharded stages (rank 0 prints them): a stage that is long on one rank only is that rank waiting for another
        keys = [k2 for k2 in (xstats[0] if xstats else {}) if k2.endswith("_ms")]
        mine = {"rank": rank, "step_wall_ms": step_walls, **{k2: round(sum(st[k2] for st in xstats) / len(xstats), 3) for k2 in keys}}
        per_rank = [None] * world
        dist.all_gather_object(per_rank, mine)

    g, gfa, t = last
    parity = None

    def whole_file(parts):
        """input_assemblies.gfa of a step: rank 0's text followed by every rank's P lines in rank order (gathered to rank 0 for the check only)."""
        head, lines = parts
        if world == 1:
            return bytes(head)
        mine = torch.frombuffer(bytearray(bytes(lines)) or bytearray(1), dtype=torch.uint8).to(dev)
        n_mine = torch.tensor([len(lines)], dtype=torch.int64, device=dev)
        sizes = torch.zeros(world, dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(sizes, n_mine)
        sizes = [int(x) for x in sizes.tolist()]
        pad = torch.zeros(max(1, max(sizes)), dtype=torch.uint8, device=dev); pad[:mine.numel()] = mine
        got = [torch.empty_like(pad) for _ in range(world)] if rank == 0 else None
        dist.gather(pad, got, dst=0)
        if rank != 0:
            return None
        return bytes(head) + b"".join(bytes(got[r][:sizes[r]].cpu().numpy().tobytes()) for r in range(world))

    file1, file2 = whole_file(gfa), whole_file(last2[1])
    d2h_all = torch.tensor([float(last2[2].d2h_bytes) + len(last2[1][1])], device=dev)
    own_strand_bytes = sum(sq.length + K - 1 for sq in seqs[seq_lo:seq_hi]) + 24 * len(seqs)      # this rank's padded strands + the sequence table
    h2d_all = torch.tensor([float(last2[2].h2d_bytes) if world == 1 else float(own_strand_bytes)], device=dev)
    if world > 1:
        dist.all_reduce(d2h_all); dist.all_reduce(h2d_all)
    if rank == 0:      # every timed run is checked: SHA-256 of the last step's GFA against the oracle's committed hash
        import hashlib
        sha = hashlib.sha256(file1).hexdigest()
        sha2 = hashlib.sha256(file2).hexdigest()
        golden = golden_for(golden_key)
        parity = {"sha256": sha, "golden": golden, "golden_key": golden_key, "ok": bool(golden) and sha == golden and sha2 == golden,
                  "checked": "last step of the resident-input loop and of the host-buffer (e2e) loop" + ("" if world == 1 else "; the file is rank 0's H/S/L text followed by the ranks' P lines")}
        gfa = file1
        if args.dump_outputs:      # the last step of the host-buffer loop: the call a user makes
            c = last2[0].counts()
            dump_outputs(args.dump_outputs, file2, [c.n_kmers, c.n_unitigs, c.n_links, c.total_length])
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    W = (2 * K + 63) // 64
    bytes_per_window = 8 * W + 16           # SURVEY.md §8(d): 8W key read + 16 payload read-modify-write per inserted k-mer occurrence (one canonical insert per window)
    bytes_per_window_design = 8 * W + 20.25  # DESIGN.md §4, what this table moves: slot 8 read + representative k-mer 8W + slot 8 RMW + slot id 4 written + packed base 0.25
    insert_ms = sum(ins_ms) / len(ins_ms)
    peak, peak_kind = measured_peak()
    own_windows = sum(sq.length for sq in seqs[seq_lo:seq_hi])     # the insert kernel only hashes this rank's sequences
    achieved = own_windows * bytes_per_window / (insert_ms * 1e-3) / 1e9
    achieved_design = own_windows * bytes_per_window_design / (insert_ms * 1e-3) / 1e9
    value = n_bases * args.steps / (ms_res * 1e-3) / 1e6
    e2e = n_bases * args.steps / (ms_e2e * 1e-3) / 1e6
    mean = lambda key: sum(d[key] for d in dev_t) / len(dev_t)
    out = {
        "metric": METRIC, "value": round(value, 3), "unit": "Mbp/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(ms_res / args.steps, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u64", "data": "synthetic (splitmix64 genomes, SURVEY.md §8d)",
        "config": {"workload": WORKLOAD, "k": K, "input_bases": n_bases, "sequences": len(seqs),
                   "exchange": None if world == 1 else "all-gather of deduplicated k-mer entries (16 B each) over NCCL, gather of unitig occurrences (16 B each) to rank 0, scatter of path tokens (4 B per occurrence) back to the owners",
                   "l2": "working set per step (table %.0f MB at 8 B per slot + %.0f MB of per-position arrays) exceeds the 126 MB L2; the table is re-initialised and every array rewritten every step" % (t.table_capacity * 8 / 1e6, n_bases * 4.6 / 1e6),
                   "gfa_bytes": len(gfa), "unitigs": int(g.counts().n_unitigs), "numa_node": numa_node},
        "e2e": {"value": round(e2e, 3), "unit": "Mbp/s", "ms_per_step": round(ms_e2e / args.steps, 3),
                "h2d_bytes_per_step": int(h2d_all.item()), "d2h_bytes_per_step": int(d2h_all.item()),
                "copies": "h2d = every rank's own strands over its own PCIe link (the others' blocks are broadcast over NVLink), summed over the ranks; d2h = rank 0's H/S/L text + every rank's own P lines, each over its own link" if world > 1 else "one GPU"},
        "gpu_launches": int(launches),
        "parity": parity,
        "clocks": clocks,
        "roofline": {"kernel": "%s<%d> (k-mer hash insert)" % (INSERT_BODY, W), "bound": "hbm", "achieved": round(achieved, 2), "peak": peak, "unit": "GB/s",
                     "frac": round(achieved / peak, 4), "peak_kind": peak_kind,
                     "traffic": measured_traffic("%s<%d>:%s:k%d" % (INSERT_BODY, W, args.workload, K)) if world == 1 else None,
                     "limiter": ("integer ALU pipe (70 % busy, issue slots 64 %; DRAM 18 %, L2 43 %: profiles/kernels_r2.md) - the kernel moves about its algorithmic bytes and is bound by the instructions that hash, probe and compare"
                                 if t.table_capacity * 8 <= 126e6 else
                                 "DRAM latency: the table (%.0f MB) exceeds the 126 MB L2, every probe and most comparisons are random 32-byte DRAM sectors (3.7 x the algorithmic bytes, DRAM busy 35 %, issue slots 37 %: profiles/kernels_r2.md, config 4)" % (t.table_capacity * 8 / 1e6)),
                     "algorithmic_bytes_per_window": bytes_per_window, "windows_per_launch": int(own_windows), "kernel_ms": round(insert_ms, 3),
                     "timed": "CUDA events right around the kernel's launch on the library's stream, mean over the timed steps (stage_ms.insert also holds the table initialisation and the counter read-back)",
                     "accounting": "SURVEY 8(d): 8W+16 bytes per canonical window insert; by DESIGN.md's own count (8W+20.25) achieved %.1f GB/s = %.4f of peak; %.4f of the nominal 8 TB/s"
                                   % (achieved_design, achieved_design / peak, achieved / 8000.0)},
        "stage_ms": {k2: round(mean(k2), 3) for k2 in ("pack", "sample", "insert", "insert_kernel", "adjacency", "boundaries", "runs", "unitigs", "links", "seed_sort", "emit", "device_simplify", "device_gfa", "d2h", "device_total",
                                                        "host_graph", "host_simplify", "host_gfa")},
    }
    if world > 1 and xstats:       # rank 0's view of the sharded stages: where the step goes when it does not scale
        keys = [k2 for k2 in xstats[0] if k2.endswith("_ms")]
        out["stage_ms"].update({k2: round(sum(st[k2] for st in xstats) / len(xstats), 3) for k2 in keys})
        out["exchange"] = {k2: int(xstats[-1][k2]) for k2 in xstats[-1] if not k2.endswith("_ms")}
        tail = {k2: v for k2, v in out["stage_ms"].items() if k2 in ("unitigs", "links", "seed_sort", "emit", "device_simplify", "device_gfa", "d2h", "adjacency", "merge_ms", "exchange_ms", "gather_runs_ms", "path_lines_ms")}
        out["per_rank"] = per_rank
        out["limiting_stage"] = max(tail, key=tail.get) + " (rank 0's view; unitigs to device_gfa are the union graph finished by rank 0 alone)"
    if rank == 0:
        if not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline(sample_replicon=1_500_000)       # about 15 s of one core
        if world == 1 and not args.no_cli_wall:
            out["cli_wall"] = cli_wall(assemblies, K, n_bases, parity["golden"] if parity else None)
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()
    if rank == 0 and not parity["ok"] and not os.environ.get("AC_BENCH_ALLOW_UNCHECKED"):
        sys.stderr.write("bench.py: the timed GFA does not match the oracle's committed SHA-256 (%s)\n" % golden_key)
        sys.exit(3)


def workload_for(args, world):
    """-> (workload name, assemblies to generate, key of its committed oracle hash).  N = 1: the configuration the metric is quoted on
    (cfg2).  N > 1: BASELINE config 5 — the first 8N assemblies of the cfg5 generator, 8 per rank; N = 8 is cfg5 itself."""
    from autocycler_b200 import synth
    workload = args.workload or ("cfg2" if world == 1 else "cfg5")
    per_rank = 8 if workload == "cfg5" else synth.CONFIGS[workload][2]
    n_assemblies = per_rank * world
    whole = n_assemblies == synth.CONFIGS[workload][2] and workload != "cfg5"
    key = f"{workload}_k{args.k}" + ("" if whole else f"_n{n_assemblies}")
    label = f"{WORKLOADS[workload]}, k={args.k}" if n_assemblies == synth.CONFIGS[workload][2] else f"the first {n_assemblies} assemblies of {WORKLOADS[workload]}, k={args.k}"
    return workload, per_rank, n_assemblies, key, label


def cli_wall(assemblies, k, n_bases, golden):
    """The user's clock (compress.rs:34-49 and the process around it): `autocycler compress` from process start to both files closed, FASTA
    files on disk -> input_assemblies.gfa + .yaml on disk.  Run twice: the first run pays the CUDA context and a cold page cache for
    the library, the second is warm.  Stage A (load + end repair), the graph, and the file writes are all inside; the steady-state
    library numbers above (`value`, `e2e`) are per graph on a live handle."""
    import hashlib
    import tempfile
    from autocycler_b200 import synth
    exe = os.path.join(ROOT, "autocycler_b200", "bin", "autocycler")
    runs = []
    with tempfile.TemporaryDirectory() as d:
        src = os.path.join(d, "in")
        synth.write_assemblies(assemblies, src)
        for rep in range(2):
            dst = os.path.join(d, "out%d" % rep)
            t0 = time.perf_counter()
            try:
                r = subprocess.run([exe, "compress", "-i", src, "-a", dst, "--kmer", str(k)], capture_output=True, text=True, timeout=300)
            except Exception as e:     # noqa: BLE001 - reported, not fatal for the bench line
                return {"error": repr(e)[:200]}
            wall = time.perf_counter() - t0
            if r.returncode != 0:
                return {"error": r.stderr[-300:]}
            sha = hashlib.sha256(open(os.path.join(dst, "input_assemblies.gfa"), "rb").read()).hexdigest()
            runs.append({"wall_s": round(wall, 3), "Mbp_per_s": round(n_bases / wall / 1e6, 1), "gfa_ok": bool(golden) and sha == golden})
    return {"what": "autocycler compress, process start -> GFA and YAML closed (FASTA on disk in, files on disk out)", "cold": runs[0], "warm": runs[1]}


def oracle_inputs(workload, n_assemblies, k, replicon=None):
    """Stage A through the oracle (untimed, as in the GPU arm): the synthetic assemblies of `workload` -> padded, end-repaired strands."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import tempfile
    import oracle_lib as o
    from autocycler_b200 import synth
    assemblies = synth.make_assemblies(workload, n_assemblies=n_assemblies, replicon_lengths=[replicon] if replicon else None)
    with tempfile.TemporaryDirectory() as d:
        synth.write_assemblies(assemblies, d)
        count, seqs = o.load_sequences(d, k, threads=min(8, os.cpu_count() or 1))
    return o, seqs, count, synth.total_bases(assemblies)


def cpu_baseline(sample_replicon):
    """The repo arm's CPU leg: a bounded sample (same generator, divergence and assembly count as cfg2, shorter replicon)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib
    flags = oracle_lib.use_native()
    o, seqs, count, n_bases = oracle_inputs("cfg2", 8, K, replicon=sample_replicon)
    t0 = time.perf_counter()
    gfa, st, _ = o.compress_seqs(seqs, count, K)
    dt = time.perf_counter() - t0
    return {"value": round(n_bases / dt / 1e6, 4), "unit": "Mbp/s", "cores": 1, "kind": "port", "host_cores": os.cpu_count(), "build": flags,
            "sample": f"8 assemblies x {sample_replicon} bp (cfg2 generator), k={K}, {n_bases} bases in {dt:.1f} s; graph stages are single-threaded in the reference (SURVEY D5); "
                      "the full-size number is the --impl reference arm",
            "stage_s": {"kmer_graph": round(st.t_kmer_graph, 2), "unitig_graph": round(st.t_unitig_graph, 2), "simplify": round(st.t_simplify, 2), "gfa": round(st.t_gfa, 2)}}


def run_reference(args):
    """The reference's CPU algorithm (oracle port, built -O3 -march=native on this machine) on the SAME workload as the B200 arm at this N,
    at full size.  One pass over cfg2 takes about a minute, so the passes are counted against a time budget: at least one full-size
    pass is timed, never a smaller input (unless a single pass could not finish inside the driver's limit; the line then says so)."""
    import hashlib
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib
    flags = oracle_lib.use_native()
    global K
    K = args.k
    workload, per_rank, n_assemblies, golden_key, label = workload_for(args, args.gpus)
    budget_s = float(os.environ.get("AC_REF_BUDGET_S", "420"))          # for the timed passes together
    one_pass_limit_s = float(os.environ.get("AC_REF_PASS_LIMIT_S", "900"))
    from autocycler_b200 import synth
    full_n, note = n_assemblies, None
    est_rate = 0.24e6                                                     # bases per second (cfg5 in the build container): only used to avoid a pass that cannot end in time
    genome = sum(synth.CONFIGS[workload][1])
    while n_assemblies > 8 and n_assemblies * genome / est_rate > one_pass_limit_s:
        n_assemblies //= 2                                                # stays on a committed golden (cfg5_k51_n16 / _n32)
    if n_assemblies != full_n:
        note = f"one pass over all {full_n} assemblies would not end inside the limit on one core: the first {n_assemblies} are timed instead"
        golden_key = f"{workload}_k{K}_n{n_assemblies}"
    o, seqs, count, n_bases = oracle_inputs(workload, n_assemblies, K)
    t_start = time.perf_counter()
    warm = 0
    times, sha, st = [], None, None
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        gfa, st, _ = o.compress_seqs(seqs, count, K)
        dt = time.perf_counter() - t0
        if sha is None:
            sha = hashlib.sha256(gfa.encode()).hexdigest()
        # warm-up passes only while they are cheap: a pass over tens of Mbp touches gigabytes and is as cold the second time
        if i < args.warmup and dt * (args.warmup + 1) < 0.25 * budget_s:
            warm += 1
        else:
            times.append(dt)
        if len(times) >= args.steps or (times and sum(times) + dt > budget_s):
            break
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, gfa.encode(), [st.n_kmers, st.unitigs_after, st.links_after, st.length_after])
    total = sum(times)
    v = round(n_bases * len(times) / total / 1e6, 4)
    golden = golden_for(golden_key)
    sample = f"{len(times)} full-size pass(es) over {n_assemblies} assemblies, {n_bases} bases each ({warm} warm-up); {note or 'same input as the B200 arm'}"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "Mbp/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "steps_timed": len(times), "warmup_done": warm,
        "ms_per_step": round(total / len(times) * 1e3, 2), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
        "data": "synthetic (splitmix64 genomes, SURVEY.md §8d)",
        "config": {"workload": label if n_assemblies == full_n else f"the first {n_assemblies} assemblies of {WORKLOADS[workload]}, k={K}", "k": K, "input_bases": n_bases, "sequences": len(seqs), "sample": sample},
        "parity": {"sha256": sha, "golden": golden, "golden_key": golden_key, "ok": bool(golden) and sha == golden},
        "cpu_baseline": {"value": v, "unit": "Mbp/s", "cores": 1, "host_cores": os.cpu_count(), "kind": "port", "build": flags, "sample": sample +
                         "; oracle = C++ restatement of the reference's Rust path (the reference itself cannot be built here: no Rust toolchain); "
                         "its graph stages are single-threaded by construction (SURVEY D5); clock = compress.rs:42-47 (k-mer graph -> GFA text), stage A untimed in both arms",
                         "stage_s": {"kmer_graph": round(st.t_kmer_graph, 2), "unitig_graph": round(st.t_unitig_graph, 2), "simplify": round(st.t_simplify, 2), "gfa": round(st.t_gfa, 2)}},
        "e2e": {"value": v, "unit": "Mbp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS), help="BASELINE.json config to run (default: cfg2, the one the metric is quoted on, at N=1; cfg5's first 8N assemblies at N>1)")
    ap.add_argument("--k", type=int, default=51)
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU oracle leg and the CLI runs (profiling and A/B runs)")
    ap.add_argument("--no-cli-wall", action="store_true", help="skip the two `autocycler compress` process runs that report the CLI's wall clock")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write what the last timed step returned to DIR/<name>.npy (float32 / float64)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    args.no_cli_wall = args.no_cli_wall or args.no_cpu_baseline          # profiling and A/B runs: the device path only
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
