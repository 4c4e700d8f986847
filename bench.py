#!/usr/bin/env python3
"""bench.py — read pairs/s of the fusion-matching hot path on synthetic paired-end reads vs the cancer.csv-shaped panel.

  python bench.py --gpus N --steps K --warmup W            # our arm
  python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (C++ restatement in oracle/: there is
                                                           # no Rust toolchain in this image, see DESIGN.md)

Main leg = BASELINE.json configs[1] (2x150 bp, 10 M pairs per GPU, one rank per GPU under torchrun, weak scaling, index
replicated, no data-path collective): `value` is device-timed with the batch resident in HBM, `e2e` goes through the
reference-facing C-ABI call (gf_map_pairs) from pinned host memory, `parity` compares EVERY record of the timed workload with
the CPU oracle's (N = 1), `roofline` / `cpu_baseline` as the contract says.  `configs` holds the other BASELINE.json configs,
each with its own clocks sample, roofline and full-size parity: the read-length sweep (2x75 / 2x250, 50 M pairs), the 16-CSV
list call, raw FASTQ text through gf_map_fastq, config 3 (100 M pairs split over the ranks: strong scaling) and the Matcher
pass (gf_reference_create over a 1 Gbase synthetic reference).  --legs selects them (default: all at N = 1, main + config3
under torchrun).  Rank 0 prints ONE JSON line; a parity mismatch makes the run fail.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True     # the tree may be read-only: importing the package from it leaves no __pycache__ there

METRIC = "read_pairs_per_sec_matched"
UNIT = "pairs/s"
ALL_LEGS = ("main", "sweep75", "sweep250", "list16", "fastq", "config3", "matcher")
SEEDS = {75: 11, 150: 12, 250: 13}     # SURVEY 8(d)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--pairs", type=int, default=10_000_000, help="pairs per GPU per step (configs[1]: 10M)")
    ap.add_argument("--read-len", type=int, default=150)
    ap.add_argument("--seed", type=int, default=12)
    ap.add_argument("--panel-scale", type=float, default=1.0)
    ap.add_argument("--repeat-frac", type=float, default=0.0, help="fraction of the panel's bases in planted 2-5-copy blocks")
    ap.add_argument("--cpu-sample", type=int, default=0, help="pairs per step of the reference arm (0 = 2,000,000)")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU oracle (no cpu_baseline, no parity)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--legs", default=os.environ.get("GF_BENCH_LEGS", ""), help="comma list of " + ",".join(ALL_LEGS))
    ap.add_argument("--sweep-pairs", type=int, default=50_000_000)
    ap.add_argument("--total-pairs", type=int, default=100_000_000, help="config 3: pairs of the whole job, split over the ranks")
    ap.add_argument("--matcher-mbases", type=int, default=1024)
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the match records of the timed path "
                    "(main leg; --impl reference: the oracle's) as DIR/<gf_match field>.npy and their count as "
                    "DIR/n_records.npy, float64, in (pair_idx, source) order")
    return ap.parse_args()


def workload_name(a):
    return (f"synthetic 2x{a.read_len}bp, {a.pairs} pairs/GPU vs cancer.csv-shaped panel "
            f"(136 genes, {15.1 * a.panel_scale:.1f} Mbases) on synthetic contigs")


def config_dict(a):
    """identical in both arms (the driver compares them)"""
    P, L = a.pairs, a.read_len
    return {"workload": workload_name(a), "pairs_per_gpu": P, "read_len": L, "seed": a.seed,
            "panel_scale": a.panel_scale, "repeat_frac": a.repeat_frac,
            "l2": f"inputs ({4 * P * L / 1e9:.0f} GB/GPU) and table (0.5 GB) both exceed the 126 MB L2; no flush needed",
            "sharding": "pairs sharded by rank, index replicated, no data-path collective"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def stop(self, t_begin=None, t_end=None):
        """clocks of the samples that arrived inside [t_begin, t_end] (host clock); when the timed region is shorter than
        the sampling period the samples of the whole loaded phase (warm-up .. extra steps, the same kernels) are used and
        `window` says so"""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

        def summarise(lines):
            sm, mx, reasons = [], [], set()
            for _t, ln in lines:
                f = [x.strip() for x in ln.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1]))
                    mx.append(float(f[2]))
                except ValueError:
                    continue
                for nm, v in zip(names, f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            sm.sort()
            return sm, mx, sorted(reasons)
        window = "timed region"
        inside = [x for x in self.lines if t_begin is None or (t_begin - 0.01 <= x[0] <= t_end + 0.03)]
        sm, mx, reasons = summarise(inside)
        if len(sm) < 2:
            window = "warm-up + timed region + further identical steps (timed region shorter than the sampling period)"
            sm, mx, reasons = summarise(self.lines)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": reasons, "window": window}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic():
    """per-launch DRAM bytes of the dominant kernel from the committed ncu capture, if any"""
    p = os.path.join(ROOT, "profiles", "screen_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            return None
    return None


def cpu_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def host_topology():
    """what the e2e numbers depend on: NUMA nodes of the box and of this rank's GPU (a single-node KVM guest reports -1)"""
    import glob
    nodes = len(glob.glob("/sys/devices/system/node/node[0-9]*"))
    return {"numa_nodes": nodes, "cpus": cpu_threads()}


def _only_json_on_stdout():
    """Libraries (NCCL's version banner, nvcc) write to the C-level stdout; the contract is ONE JSON line there.
    Everything else goes to stderr; the JSON line is written to the saved descriptor."""
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    return os.fdopen(saved, "w")


def log(*a):
    print("[bench]", *a, file=sys.stderr, flush=True)


# ------------------------------------------------------------------------------------------------ oracle helpers
def match_dtype():
    import numpy as np
    return np.dtype([("pair_idx", "<u8"), ("read_break", "<i4"), ("l_pos", "<i4"), ("r_pos", "<i4"), ("gap", "<i4"),
                     ("l_dist", "<i4"), ("r_dist", "<i4"), ("seq_len", "<i4"), ("l_contig", "<i2"), ("r_contig", "<i2"),
                     ("merge_olen", "<i2"), ("merge_diff", "<i2"), ("source", "u1"), ("used_rc", "u1"), ("reversed", "u1"),
                     ("filter_flags", "u1")])


def oracle_scan_raw(oidx, batch, threads, pair_base=0):
    """CPU oracle over a host batch -> structured array of gf_match records in (pair_idx, source) order.
    (oracle/ is test infrastructure: here it is the CHECKER of the CUDA path's records and the timed CPU baseline.)"""
    import numpy as np
    import _oracle
    from genefuserust_b200._abi import gf_match
    cap = max(1 << 16, batch.n // 8)
    L = _oracle.lib()
    st = batch.as_struct()
    while True:
        buf = np.zeros(cap, dtype=match_dtype())
        n = L.orc_scan_pairs(oidx.h, C.byref(st), C.cast(buf.ctypes.data, C.POINTER(gf_match)), cap, threads)
        if n <= cap:
            break
        cap = int(n)
    out = buf[:n].copy()
    out["pair_idx"] += np.uint64(pair_base)
    return out


def gpu_records(torch, d_out, n):
    """device record buffer -> structured array sorted by (pair_idx, source)"""
    import numpy as np
    dt = match_dtype()
    raw = d_out[:n * dt.itemsize].cpu().numpy().view(dt)
    return np.sort(raw, order=["pair_idx", "source"])


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, recs):
    """records (structured, match_dtype order) -> one float64 .npy per field + n_records.npy.  Beyond DUMP_BYTES a fixed,
    seeded sample of the rows is written: the same rows whenever the record count is the same."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    fields = recs.dtype.names
    rows = np.arange(len(recs))
    cap = (DUMP_BYTES - 4096) // (8 * len(fields))      # (4096: the .npy headers)
    if len(rows) > cap:
        rows = np.sort(np.random.default_rng(0).choice(len(recs), cap, replace=False))
    np.save(os.path.join(out_dir, "n_records.npy"), np.array([len(recs)], dtype=np.float64))
    for f in fields:
        np.save(os.path.join(out_dir, f + ".npy"), recs[f][rows].astype(np.float64))
    log(f"dumped {len(rows)} of {len(recs)} records to {out_dir}")


def parity_record(got, want, pairs, what):
    import numpy as np
    same = len(got) == len(want) and got.tobytes() == want.tobytes()
    rec = {"pairs": int(pairs), "records": int(len(want)), "gpu_records": int(len(got)), "identical": bool(same),
           "checked_against": "CPU oracle (oracle/: C++ restatement of the reference's CPU path; its core has no reference "
                              "vector, see DESIGN.md) over " + what}
    if not same:
        k = 0
        m = min(len(got), len(want))
        while k < m and got[k].tobytes() == want[k].tobytes():
            k += 1
        rec["first_difference"] = {"index": k, "gpu": str(got[k]) if k < len(got) else None,
                                   "oracle": str(want[k]) if k < len(want) else None}
    return rec


# ------------------------------------------------------------------------------------------------ workload on the device
class DeviceWorkload:
    """Counter-based synthetic pairs [first, first + P) generated on the host in pieces (one reusable set of pinned buffers),
    uploaded into four device arenas; optionally every piece also goes through the CPU oracle (records kept, time summed).
    The LAST piece generated is pairs [0, piece) of this rank and stays in the pinned buffers for the e2e leg."""

    def __init__(self, torch, synth, panel, P, L, seed, first, dev, threads, oracle=None, oracle_threads=1):
        import numpy as np
        self.P, self.L = P, L
        piece = max(1, min(P, (6 << 30) // (4 * L)))
        piece = min(piece, 10_000_000 if L <= 150 else piece)
        self.piece = piece
        t0 = time.perf_counter()
        self.pinned = [torch.empty(piece * L, dtype=torch.uint8, pin_memory=True) for _ in range(4)]
        self.d_arr = [torch.empty(P * L, dtype=torch.uint8, device=dev) for _ in range(4)]
        self.oracle_records = [] if oracle is not None else None
        self.oracle_s = 0.0
        self.gen_s = 0.0
        starts = list(range(0, P, piece))
        for lo in reversed(starts):       # descending, so that the first piece is the one left in `pinned`
            cn = min(piece, P - lo)
            g0 = time.perf_counter()
            batch = synth.generate_pairs(panel, cn, read_len=L, seed=seed, first=first + lo, threads=threads,
                                         out=tuple(t.numpy()[:cn * L] for t in self.pinned))
            self.gen_s += time.perf_counter() - g0
            for dt_, pt in zip(self.d_arr, self.pinned):
                dt_[lo * L:(lo + cn) * L].copy_(pt[:cn * L], non_blocking=True)
            if oracle is not None:
                o0 = time.perf_counter()
                self.oracle_records.append((lo, oracle_scan_raw(oracle, batch, oracle_threads, pair_base=lo)))
                self.oracle_s += time.perf_counter() - o0
            torch.cuda.synchronize()
        self.batch = batch                # host view of pairs [0, cn0)
        off_host = torch.from_numpy(batch.off1.view(np.int64)).pin_memory()
        self.off_host = off_host
        batch.off1 = off_host.numpy().view(np.uint64)
        batch.off2 = batch.off1
        self.d_off = torch.arange(P + 1, dtype=torch.int64, device=dev) * L
        self.setup_s = time.perf_counter() - t0
        if self.oracle_records is not None:
            self.oracle_records.sort(key=lambda x: x[0])
            self.oracle_all = np.concatenate([r for _, r in self.oracle_records]) if self.oracle_records else None

    def gf_batch(self):
        from genefuserust_b200._abi import gf_batch
        db = gf_batch()
        db.n = self.P
        db.seq1, db.qual1, db.seq2, db.qual2 = (t.data_ptr() for t in self.d_arr)
        db.off1 = db.off2 = self.d_off.data_ptr()
        db.bytes1 = db.bytes2 = self.P * self.L
        db.max_len = self.L
        return db

    def free(self, torch):
        self.d_arr = self.pinned = self.d_off = None
        torch.cuda.empty_cache()


def time_device_steps(torch, lib, handles, db, out_cap, steps, warmup, local_rank, barrier, list_mode=False):
    """W warm-up + K timed steps of gf_map_pairs_device (or ONE gf_map_pairs_device_list call per step) with CUDA events on
    the launching stream; returns (ms_total, clocks, stats of the last step, d_out buffers, d_nout)"""
    from genefuserust_b200._abi import gf_map_stats, gf_match
    dev = torch.device("cuda", local_rank)
    K = len(handles)
    d_outs = [torch.empty(out_cap * C.sizeof(gf_match), dtype=torch.uint8, device=dev) for _ in range(K)]
    d_ns = torch.zeros(K, dtype=torch.int64, device=dev)
    stream = torch.cuda.current_stream()
    if list_mode:
        hs = (C.c_void_p * K)(*[h.value for h in handles])
        outs = (C.c_void_p * K)(*[t.data_ptr() for t in d_outs])
        nouts = (C.c_void_p * K)(*[d_ns.data_ptr() + 8 * k for k in range(K)])

        def step():
            rc = lib.gf_map_pairs_device_list(hs, K, C.byref(db), outs, out_cap, nouts, C.c_void_p(stream.cuda_stream))
            if rc != 0:
                raise RuntimeError(lib.gf_last_error().decode())
    else:
        def step():
            for k, h in enumerate(handles):
                rc = lib.gf_map_pairs_device(h, C.byref(db), d_outs[k].data_ptr(), out_cap, d_ns.data_ptr() + 8 * k,
                                             C.c_void_p(stream.cuda_stream))
                if rc != 0:
                    raise RuntimeError(lib.gf_last_error().decode())
    sampler = ClockSampler(local_rank).start()     # before the warm-up: nvidia-smi needs ~100 ms for its first line
    for _ in range(max(warmup, 3)):
        step()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_begin = time.perf_counter()
    ev0.record(stream)
    for _ in range(steps):
        step()
    ev1.record(stream)
    barrier()
    t_end = time.perf_counter()
    ms_total = ev0.elapsed_time(ev1)
    stats = []
    for h in handles:
        st = gf_map_stats()
        lib.gf_get_map_stats(h, C.byref(st))
        stats.append(st)
    # per-kernel durations of a few more single steps (the library's own events on the launching stream), and enough
    # samples for the clocks line when the timed region was shorter than the sampling period
    parts = []
    t_extra = time.perf_counter()
    k = 0
    while k < min(3, steps) or (len(sampler.lines) < 4 and time.perf_counter() - t_extra < 1.0):
        step()
        s2 = gf_map_stats()
        lib.gf_get_map_stats(handles[-1], C.byref(s2))
        parts.append((s2.ms_screen, s2.ms_exact, s2.ms_prep, s2.ms_seed, s2.ms_diag, s2.ms_scan))
        k += 1
    clocks = sampler.stop(t_begin, t_end)
    return ms_total, clocks, stats, parts, d_outs, d_ns, step


def roofline_block(stats, parts, ms_step, P, L, n_records, peak, peak_src, traffic=None, whole_step_mult=0):
    """SURVEY 8(d) yardstick + what it hides.  achieved = algorithmic bytes (bases of every mapped sequence + one 32-byte
    sector per pass-1 probe) / the screen's measured duration; frac_compulsory = the bytes that MUST cross HBM once (both
    mates' bases, two 8-byte offsets per pair, the emitted records) / the same time: the streaming bound of this path."""
    st = stats
    alg_bytes = st.seq_bytes + 32 * st.n_probes_pass1
    k_ms = sum(p[0] for p in parts) / len(parts)
    ex_ms = sum(p[1] for p in parts) / len(parts)
    if whole_step_mult:   # list mode: `mult` indices per step, only the whole step is timed as one unit
        alg_bytes *= whole_step_mult
        k_ms = ms_step
    achieved = alg_bytes / (k_ms / 1000.0) / 1e9
    compulsory = 2 * P * L + 16 * P + 48 * n_records
    names = ("k_prep", "k_seed", "k_diag", "k_scan")
    per_kernel = {}
    for i, nm in enumerate(names):
        e = {"ms": sum(p[2 + i] for p in parts) / len(parts)}
        if traffic and nm in traffic.get("kernels", {}):
            e.update(traffic["kernels"][nm])
            if e["ms"] > 0 and "dram_bytes" in e:
                e["dram_gbs_live"] = e["dram_bytes"] / (e["ms"] / 1000.0) / 1e9
        per_kernel[nm] = e
    dram = traffic["dram_bytes_per_launch"] if traffic else None
    return {"bound": "hbm",
            "kernel": "screen = k_prep + k_seed + k_diag + k_scan (fast_merge + conservative pass 1 of Indexer::map_read for "
                      "every pair; 4 launches per step, timed together with CUDA events on the launching stream)",
            "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
            "traffic": dram, "algorithmic_bytes_per_launch": int(alg_bytes), "kernel_ms": k_ms,
            "compulsory_bytes_per_launch": int(compulsory),
            "frac_compulsory": compulsory / (k_ms / 1000.0) / 1e9 / peak,
            "frac_compulsory_whole_step": compulsory / (ms_step / 1000.0) / 1e9 / peak,
            "dram_frac": (dram / (k_ms / 1000.0) / 1e9 / peak) if dram else None,
            "per_kernel": per_kernel,
            "note": "frac is the SURVEY 8(d) yardstick (one 32-byte HBM sector charged per pass-1 probe).  The probes are "
                    "answered from an L2-resident filter + 2-bit gene planes, so the yardstick can exceed 1 and is not what "
                    "to optimise against: frac_compulsory (bases + offsets + records that must stream from HBM once, over the "
                    "same time) is the distance to the streaming bound, dram_frac the measured DRAM traffic (ncu, profiles/) "
                    "over the same time.",
            "kernel_share_of_step": k_ms / ms_step, "exact_verify_ms": ex_ms}


# ================================================================================================ reference arm
def reference_arm(a, json_out, rank):
    """CPU only, rank 0 only; loads oracle/ and the synthetic-data helper, never the CUDA library."""
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from genefuserust_b200 import synth
    import _oracle
    synth.build()
    _oracle.build_oracle()
    panel = synth.make_panel(scale=a.panel_scale, repeat_frac=a.repeat_frac)
    threads = cpu_threads()
    n_sample = min(a.pairs, a.cpu_sample or 2_000_000)
    batch = synth.generate_pairs(panel, n_sample, read_len=a.read_len, seed=a.seed, threads=threads)
    oidx = _oracle.OracleIndex(panel.genes())
    for _ in range(a.warmup):
        oidx.scan(batch.slice(0, min(20000, batch.n)), threads=threads)
    t0 = time.perf_counter()
    for _ in range(a.steps):
        recs = oracle_scan_raw(oidx, batch, threads)
    dt = time.perf_counter() - t0
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, recs)
    val = batch.n * a.steps / dt
    sample = (f"each step = the first {batch.n} pairs of the workload (bounded sample of its {a.pairs} pairs), "
              f"{a.steps} steps; C++ restatement of the Rust CPU path (oracle/), packs of 1000 pairs over all host threads")
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": 1000 * dt / a.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8/int64", "data": "synthetic", "config": config_dict(a),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    json_out.write(json.dumps(line) + "\n")
    json_out.flush()


# ================================================================================================ our arm
def main():
    a = parse_args()
    json_out = _only_json_on_stdout()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    # the ranks of one box share its host cores: each packs its uploads (csrc/gf_pack.cpp) with its share of them
    os.environ.setdefault("GF_PACK_THREADS", str(max(1, min(64, (cpu_threads() - cpu_threads() // 4) // world))))
    if a.impl == "reference":
        return reference_arm(a, json_out, rank)

    import numpy as np
    import torch
    import torch.distributed as dist
    import __graft_entry__ as ge
    from genefuserust_b200 import synth
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ge.build()
    from genefuserust_b200._abi import gf_map_stats, gf_match
    from genefuserust_b200.host import FusionMapper
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    legs = [x for x in (a.legs.split(",") if a.legs else (ALL_LEGS if world == 1 else ("main", "config3"))) if x]
    for x in legs:
        if x not in ALL_LEGS:
            raise SystemExit(f"unknown leg {x!r}")
    if a.dump_outputs and "main" not in legs:
        raise SystemExit("--dump-outputs writes the main leg's records: select the main leg")
    dev = torch.device("cuda", local_rank)
    threads = max(1, cpu_threads() // max(1, world))
    want_oracle = (not a.no_cpu_baseline) and world == 1
    peak, peak_src = measured_peak()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def all_max(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def all_sum(x):
        t = torch.tensor([float(x)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    panel = synth.make_panel(scale=a.panel_scale, repeat_frac=a.repeat_frac)
    genes = panel.genes()
    # the first create also pays CUDA context + module load; time a second one for the steady-state index build
    t0 = time.perf_counter()
    FusionMapper.from_gene_spans(genes, device=local_rank).close()
    t_first = time.perf_counter() - t0
    t0 = time.perf_counter()
    mapper = FusionMapper.from_gene_spans(genes, device=local_rank)
    t_index = time.perf_counter() - t0
    info = mapper.m_indexer.info()
    lib, h = mapper.lib, mapper.m_indexer.h
    oracle = None
    t_oidx = 0.0
    if want_oracle:
        import _oracle
        t0 = time.perf_counter()
        oracle = _oracle.OracleIndex(genes)
        t_oidx = time.perf_counter() - t0
    failures = []
    line = {}

    # -------------------------------------------------------------------------------------------- main leg
    if "main" in legs:
        P, L = a.pairs, a.read_len
        log(f"main leg: {P} pairs 2x{L}")
        wl = DeviceWorkload(torch, synth, panel, P, L, a.seed, rank * P, dev, threads, oracle, cpu_threads())
        out_cap = max(1 << 16, P // 4)
        db = wl.gf_batch()
        ms_total, clocks, stats, parts, d_outs, d_ns, step = time_device_steps(torch, lib, [h], db, out_cap, a.steps, a.warmup,
                                                                               local_rank, barrier)
        st = stats[0]
        n_matches = int(d_ns[0].item())
        ms_total_max = all_max(ms_total)
        value = world * P * a.steps / (ms_total_max / 1000.0)
        matches_all = all_sum(n_matches)
        parity = None
        cpu = None
        if a.dump_outputs and rank == 0:
            dump_outputs(a.dump_outputs, gpu_records(torch, d_outs[0], n_matches))
        if oracle is not None:
            got = gpu_records(torch, d_outs[0], n_matches)
            parity = parity_record(got, wl.oracle_all, P, f"all {P} pairs of the timed workload")
            if not parity["identical"]:
                failures.append("main leg: GPU records differ from the oracle's")
            cpu = {"value": P / wl.oracle_s, "unit": UNIT, "cores": cpu_threads(), "kind": "port",
                   "sample": f"all {P} pairs of the same workload, {wl.oracle_s:.1f} s; C++ restatement of the Rust CPU path (no "
                             f"Rust toolchain here), packs of 1000 pairs over all host threads; index build {t_oidx:.1f} s not "
                             "included; its records are the parity reference"}
        # ---- end to end through the public C-ABI call with HOST (pinned) buffers: H2D + kernels + D2H inside
        e2e = None
        if not a.no_e2e:
            hb = wl.batch.as_struct()
            out_host = (gf_match * out_cap)()
            n_out = C.c_uint64(0)

            def step_host():
                rc = lib.gf_map_pairs(h, C.byref(hb), out_host, out_cap, C.byref(n_out))
                if rc != 0:
                    raise RuntimeError(lib.gf_last_error().decode())
            step_host()
            step_host()
            barrier()
            e2e_steps = max(10, min(a.steps, 20))
            per_call = []
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                c0 = time.perf_counter()
                step_host()
                per_call.append(time.perf_counter() - c0)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            dt_max = all_max(dt)
            if wl.piece >= P and int(n_out.value) != n_matches:
                failures.append(f"e2e call returned {n_out.value} records, the device path {n_matches}")
            hs_ = gf_map_stats()
            lib.gf_get_map_stats(h, C.byref(hs_))
            # the records of the host call against the oracle's (the packed upload is a different input path into k_prep)
            e2e_parity = None
            if oracle is not None and wl.piece >= P:
                import numpy as np
                got_h = np.frombuffer(out_host, dtype=match_dtype(), count=int(n_out.value)).copy()
                e2e_parity = parity_record(got_h, wl.oracle_all, P, f"all {P} pairs, records returned by gf_map_pairs")
                if not e2e_parity["identical"]:
                    failures.append("e2e leg: records of gf_map_pairs differ from the oracle's")
            # the same call with the packed upload switched off (ASCII arenas copied as they are), for comparison
            ascii_ms = None
            if hs_.packed_upload:
                os.environ["GF_HOST_PACK"] = "0"
                step_host()
                tt = []
                for _ in range(5):
                    c0 = time.perf_counter()
                    step_host()
                    tt.append(time.perf_counter() - c0)
                del os.environ["GF_HOST_PACK"]
                ascii_ms = 1e3 * sorted(tt)[len(tt) // 2]
            per_call.sort()
            med = per_call[len(per_call) // 2]
            e2e = {"value": world * wl.batch.n * e2e_steps / dt_max, "unit": UNIT,
                   "h2d_bytes_per_step": int(hs_.h2d_bytes), "d2h_bytes_per_step": int(hs_.d2h_bytes),
                   "zero_copy_qualities": bool(hs_.zero_copy_qual),
                   "packed_upload": bool(hs_.packed_upload),
                   "upload": {0: "ASCII sequence arenas copied", 1: "every chunk as 2-bit planes built by the host threads",
                              2: "some chunks as 2-bit planes built by the host threads (csrc/gf_pack.cpp) while the copy engine "
                                 "moves the others as ASCII; the ASCII stays in pinned memory for the survivors"}[int(hs_.packed_upload)],
                   "ms_host_pack_per_step": float(hs_.ms_host_pack),
                   "pack_threads": int(os.environ.get("GF_PACK_THREADS", 0)) or cpu_threads(),
                   "ms_per_call_median_ascii_upload": ascii_ms,
                   "parity": e2e_parity,
                   "host_buffer_bytes_per_step": 4 * wl.batch.n * L + 2 * 8 * (wl.batch.n + 1),
                   "pairs_per_step": int(wl.batch.n), "steps": e2e_steps,
                   "ms_per_call_min": 1e3 * per_call[0], "ms_per_call_median": 1e3 * med, "ms_per_call_max": 1e3 * per_call[-1],
                   "h2d_gbs_this_rank_median": hs_.h2d_bytes / med / 1e9,
                   "value_from_median_call": world * wl.batch.n / all_max(med),
                   "timing": "host wall clock around the synchronous C-ABI calls (2 warm-up calls, then the timed calls back to "
                             "back), max over ranks"}
        if rank == 0:
            ms_step = ms_total_max / a.steps
            line = {
                "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3),
                "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "u8/int64", "data": "synthetic", "config": config_dict(a),
                "index": {"keys": info.n_keys, "sites": info.n_sites, "table_bytes": info.table_bytes,
                          "device_bytes": info.device_bytes, "build_ms": info.build_ms},
                "matches_per_step": matches_all, "survivors_per_step": int(st.n_survivors),
                "clocks": clocks, "e2e": e2e, "gpu_launches": int(st.kernel_launches) * a.steps,
                "parity": parity,
                "roofline": roofline_block(st, parts, ms_step, P, L, n_matches, peak, peak_src, ncu_traffic()),
                "cpu_baseline": cpu,
                "setup": {"host": host_topology(), "index_create_s": t_index, "first_index_create_s_incl_cuda_init": t_first,
                          "generate_s": wl.gen_s, "host_threads": threads},
            }
        del d_outs, d_ns
        wl.free(torch)
        del wl

    configs = {}

    def run_sweep(tag, L, P):
        log(f"{tag}: {P} pairs 2x{L}")
        wl = DeviceWorkload(torch, synth, panel, P, L, SEEDS[L], 0, dev, threads, oracle, cpu_threads())
        out_cap = max(1 << 16, P // 4)
        db = wl.gf_batch()
        ms_total, clocks, stats, parts, d_outs, d_ns, _ = time_device_steps(torch, lib, [h], db, out_cap, a.steps, a.warmup,
                                                                            local_rank, barrier)
        n = int(d_ns[0].item())
        ms_step = ms_total / a.steps
        rec = {"workload": f"read-length sweep: synthetic 2x{L}bp, {P} pairs vs the cancer.csv-shaped panel, 1 B200 "
                           "(BASELINE.json configs[4])",
               "pairs": P, "value": P / (ms_step / 1e3), "unit": UNIT, "ms_per_step": ms_step, "steps": a.steps,
               "matches": n, "survivors": int(stats[0].n_survivors), "clocks": clocks,
               "roofline": roofline_block(stats[0], parts, ms_step, P, L, n, peak, peak_src)}
        if oracle is not None:
            rec["parity"] = parity_record(gpu_records(torch, d_outs[0], n), wl.oracle_all, P, f"all {P} pairs")
            rec["cpu_baseline"] = {"value": P / wl.oracle_s, "unit": UNIT, "cores": cpu_threads(), "kind": "port",
                                   "sample": f"all {P} pairs, {wl.oracle_s:.1f} s"}
            if not rec["parity"]["identical"]:
                failures.append(f"{tag}: GPU records differ from the oracle's")
        del d_outs, d_ns
        wl.free(torch)
        return rec

    if "sweep75" in legs and rank == 0:
        configs["sweep_2x75"] = run_sweep("sweep75", 75, a.sweep_pairs)
    if "sweep250" in legs and rank == 0:
        configs["sweep_2x250"] = run_sweep("sweep250", 250, a.sweep_pairs)

    # -------------------------------------------------------------------------------------------- list mode, 16 CSVs
    if "list16" in legs and rank == 0:
        K, P, L = 16, a.pairs, 150
        log(f"list16: {K} indices x {P} pairs")
        sub = genes[:40]
        mappers = [FusionMapper.from_gene_spans(genes if k % 2 == 0 else sub, device=local_rank) for k in range(K)]
        handles = [m.m_indexer.h for m in mappers]
        o_sub = None
        if oracle is not None:
            import _oracle
            o_sub = _oracle.OracleIndex(sub)
        wl = DeviceWorkload(torch, synth, panel, P, L, 12, 0, dev, threads, oracle, cpu_threads())
        want_sub = oracle_scan_raw(o_sub, wl.batch, cpu_threads()) if (o_sub is not None and wl.piece >= P) else None
        out_cap = max(1 << 16, P // 4)
        db = wl.gf_batch()
        ms_total, clocks, stats, parts, d_outs, d_ns, _ = time_device_steps(torch, lib, handles, db, out_cap, a.steps, a.warmup,
                                                                            local_rank, barrier, list_mode=True)
        ms_job = ms_total / a.steps
        ns = [int(x) for x in d_ns.tolist()]
        rec = {"workload": f"list mode: {K} fusion CSVs (alternating the 136-gene panel and a 40-gene subset, the shape of "
                           f"benchmark_res/hg38_fusion_csv_list.txt) x {P} pairs 2x150, ONE gf_map_pairs_device_list call per "
                           "step, 1 B200 (BASELINE.json configs[3])",
               "pairs": P, "csvs": K, "value": P * K / (ms_job / 1e3), "unit": "pair x CSV / s",
               "pairs_per_s_whole_list": P / (ms_job / 1e3), "ms_per_step": ms_job, "steps": a.steps, "clocks": clocks,
               "index_bytes_total": sum(int(m.m_indexer.info().device_bytes) for m in mappers),
               "roofline": roofline_block(stats[0], parts, ms_job, P, L, sum(ns), peak, peak_src, whole_step_mult=K),
               "roofline_note": "achieved / frac: 16 x the SURVEY 8(d) bytes of one index over the whole list step (exact path "
                                "included); per_kernel are the LAST index's launches (k_prep runs once, for the first index); "
                                "frac_compulsory charges the reads once for the whole list job"}
        if oracle is not None and want_sub is not None:
            ok = True
            for k in range(K):
                got = gpu_records(torch, d_outs[k], ns[k])
                want = wl.oracle_all if k % 2 == 0 else want_sub
                ok = ok and len(got) == len(want) and got.tobytes() == want.tobytes()
            rec["parity"] = {"pairs": P, "indices": K, "records": int(sum(ns)), "identical": bool(ok),
                             "checked_against": "CPU oracle, one index per distinct panel, every record of all 16 outputs"}
            if not ok:
                failures.append("list16: GPU records differ from the oracle's")
        # end to end: one gf_list_map_pairs call from pinned host memory
        if not a.no_e2e and wl.piece >= P:
            cap_h = max(4096, P // 64)
            bufs = [(gf_match * cap_h)() for _ in range(K)]
            outs_h = (C.POINTER(gf_match) * K)(*[C.cast(b_, C.POINTER(gf_match)) for b_ in bufs])
            caps_h = (C.c_uint64 * K)(*([cap_h] * K))
            nout_h = (C.c_uint64 * K)()
            hs_arr = (C.c_void_p * K)(*[x.value for x in handles])
            hst = wl.batch.as_struct()
            walls = []
            for it in range(4):
                t0 = time.perf_counter()
                rc = lib.gf_list_map_pairs(hs_arr, K, C.byref(hst), outs_h, caps_h, nout_h)
                walls.append(time.perf_counter() - t0)
                if rc != 0:
                    raise RuntimeError(lib.gf_last_error().decode())
            walls = sorted(walls[1:])
            rec["e2e"] = {"value": P * K / walls[len(walls) // 2], "unit": "pair x CSV / s", "ms_per_list_call_median": 1e3 * walls[len(walls) // 2],
                          "calls": 3, "what": "gf_list_map_pairs from pinned host memory: one upload, one k_prep, 16 indices"}
        del d_outs, d_ns
        wl.free(torch)
        for m in mappers:
            m.close()
        if o_sub is not None:
            o_sub.close()
        configs["list16"] = rec

    # -------------------------------------------------------------------------------------------- raw FASTQ text
    if "fastq" in legs and rank == 0:
        P, L = 1_000_000, 150
        log(f"fastq: {P} pairs of raw text")
        batch = synth.generate_pairs(panel, P, read_len=L, seed=12, threads=threads)

        def fastq_text(seq, qual, mate):
            name = np.frombuffer(b"@SYN:12:000000000 %d:N:0:ACGT\n" % mate, dtype=np.uint8)
            rec = len(name) + L + 1 + 2 + L + 1
            t = torch.empty(P * rec, dtype=torch.uint8, pin_memory=True)
            out = t.numpy().reshape(P, rec)
            out[:, :len(name)] = name
            idx = np.arange(P, dtype=np.int64)
            for k in range(9):                                   # zero-padded decimal pair index
                out[:, 8 + 8 - k] = 48 + (idx // 10 ** k) % 10
            o = len(name)
            out[:, o:o + L] = seq.reshape(P, L)
            out[:, o + L] = 10
            out[:, o + L + 1] = 43
            out[:, o + L + 2] = 10
            out[:, o + L + 3:o + 2 * L + 3] = qual.reshape(P, L)
            out[:, o + 2 * L + 3] = 10
            return t
        t1 = fastq_text(batch.seq1, batch.qual1, 1)
        t2 = fastq_text(batch.seq2, batch.qual2, 2)
        cap = max(1 << 16, P // 4)
        out = np.zeros(cap, dtype=match_dtype())
        n, nrec = C.c_uint64(0), C.c_uint64(0)

        def call():
            rc = lib.gf_map_fastq(h, C.cast(t1.data_ptr(), C.c_char_p), t1.numel(), C.cast(t2.data_ptr(), C.c_char_p), t2.numel(),
                                  C.cast(out.ctypes.data, C.POINTER(gf_match)), cap, C.byref(n), C.byref(nrec))
            if rc != 0:
                raise RuntimeError(lib.gf_last_error().decode())
        sampler = ClockSampler(local_rank).start()
        call()
        call()
        walls = []
        s = gf_map_stats()
        t_begin = time.perf_counter()
        for _ in range(10):
            t0 = time.perf_counter()
            call()
            walls.append(time.perf_counter() - t0)
        t_end = time.perf_counter()
        lib.gf_get_map_stats(h, C.byref(s))
        clocks = sampler.stop(t_begin, t_end)
        walls.sort()
        med = walls[len(walls) // 2]
        text_bytes = t1.numel() + t2.numel()
        rec = {"workload": f"raw FASTQ text, {P} pairs 2x150 ({text_bytes} bytes in pinned host memory) through gf_map_fastq: "
                           "H2D of the text, record splitting and mapping on the device (SURVEY 8(f) #2)",
               "pairs": P, "value": P / med, "unit": UNIT, "what": "end to end, host wall clock around the C-ABI call, median of 10",
               "ms_per_call_median": 1e3 * med, "ms_per_call_min": 1e3 * walls[0], "device_ms_total": s.ms_total,
               "ingest_ms": s.ms_ingest, "text_gbs_through_the_call": text_bytes / med / 1e9, "clocks": clocks,
               "roofline": {"bound": "hbm", "kernel": "k_nl_count + k_nl_write + k_records (text scanned twice, 8 B per line written)",
                            "note": "the call is PCIe-bound: the text arrives at the H2D rate; the device-side split is "
                                    f"{max(0.0, s.ms_ingest - text_bytes / 55.6e6):.2f} ms of the {s.ms_ingest:.2f} ms ingest at 55.6 GB/s"}}
        if oracle is not None:
            want = oracle_scan_raw(oracle, batch, cpu_threads())
            got = out[:n.value]
            rec["parity"] = parity_record(got, want, P, f"all {P} records")
            if not rec["parity"]["identical"] or nrec.value != P:
                failures.append("fastq: GPU records differ from the oracle's")
        configs["fastq_text"] = rec
        # ---- the same reads as .fq.gz files fed as byte streams (gf_fastq_stream_*, SURVEY 8(f) #2: fastq_reader.rs:39-69,149-179):
        # one gzip member per file (inflate is sequential: one host thread per mate) and BGZF (what bgzip / bcl2fastq write:
        # members of <= 64 KB: their compressed payloads cross PCIe and the device inflates them, one warp per member)
        import gzip as _gzip
        from genefuserust_b200.host import bgzf_compress
        Pz = 250_000                                   # (compressing the bench input in Python is the slow part)
        rec_bytes = t1.numel() // P
        raw1, raw2 = bytes(t1.numpy()[:Pz * rec_bytes]), bytes(t2.numpy()[:Pz * rec_bytes])
        want_z = None
        if oracle is not None:
            want_z = want[want["pair_idx"] < Pz]
        gz_rec = {"workload": f"{Pz} pairs 2x150 as two .fq.gz byte streams through gf_fastq_stream_feed (8 MiB pieces): "
                              "gzip_single_member = host inflate (zlib, one thread per mate) + H2D of the text; bgzf = H2D of the "
                              "compressed members + inflate on the device (k_bgzf_inflate, a warp per member; GF_BGZF_DEVICE=0: "
                              "all host threads); then record splitting + mapping", "pairs": Pz, "unit": UNIT,
                  "bgzf_inflate": "host" if os.environ.get("GF_BGZF_DEVICE") == "0" else "device"}
        for kind, enc in (("gzip_single_member", lambda d: _gzip.compress(d, compresslevel=1)), ("bgzf", lambda d: bgzf_compress(d))):
            e1, e2 = enc(raw1), enc(raw2)
            k1, k2 = np.frombuffer(e1, dtype=np.uint8), np.frombuffer(e2, dtype=np.uint8)
            b1, b2 = k1.ctypes.data, k2.ctypes.data
            # one stream, the files fed three times over (a gzip file may be several files concatenated: MultiGzDecoder): the
            # first pass pays for the pinned text buffers, the passes after it are what a long file costs per record
            sh = C.c_void_p()
            if lib.gf_fastq_stream_create(h, 1, 1, 0, C.byref(sh)) != 0:
                raise RuntimeError(lib.gf_last_error().decode())
            piece = 8 << 20
            passes = []
            for _ in range(3):
                t0 = time.perf_counter()
                for p0 in range(0, max(len(e1), len(e2)), piece):      # (pointers into the files' bytes: no Python-side copies)
                    n1, n2 = max(0, min(piece, len(e1) - p0)), max(0, min(piece, len(e2) - p0))
                    a1 = C.cast(b1 + p0, C.c_char_p) if n1 else None
                    a2 = C.cast(b2 + p0, C.c_char_p) if n2 else None
                    if lib.gf_fastq_stream_feed(sh, a1, n1, a2, n2) != 0:
                        raise RuntimeError(lib.gf_last_error().decode())
                passes.append(time.perf_counter() - t0)
            t0 = time.perf_counter()
            if lib.gf_fastq_stream_finish(sh) != 0:
                raise RuntimeError(lib.gf_last_error().decode())
            nz = C.c_uint64(0)
            outz = np.zeros(3 * cap, dtype=match_dtype())
            rcz = lib.gf_fastq_stream_take(sh, C.cast(outz.ctypes.data, C.POINTER(gf_match)), 3 * cap, C.byref(nz))
            t_fin = time.perf_counter() - t0
            lib.gf_fastq_stream_destroy(sh)
            if rcz != 0:
                raise RuntimeError(lib.gf_last_error().decode())
            best = min(passes[1:]) + t_fin / 3      # (the text is mapped when 256 MiB have accumulated or at finish)
            sub = {"value": Pz / best, "ms_per_pass": 1e3 * best, "ms_first_pass_incl_pinned_buffers": 1e3 * passes[0],
                   "compressed_bytes": len(e1) + len(e2), "inflated_gbs": 2 * len(raw1) / best / 1e9}
            if want_z is not None:
                gotz = outz[:nz.value]
                sub["parity"] = parity_record(gotz[gotz["pair_idx"] < Pz], want_z, Pz, f"all {Pz} records of the first pass; "
                                              f"the three passes returned {int(nz.value)} records = 3 x {len(want_z)}")
                if int(nz.value) != 3 * len(want_z):
                    failures.append(f"fastq_gz {kind}: record count of the repeated passes")
                if not sub["parity"]["identical"]:
                    failures.append(f"fastq_gz {kind}: GPU records differ from the oracle's")
            gz_rec[kind] = sub
        configs["fastq_gz"] = gz_rec
        del t1, t2

    # -------------------------------------------------------------------------------------------- config 3: 100 M pairs, strong
    if "config3" in legs:
        from genefuserust_b200.sharding import shard_range
        total = a.total_pairs
        first, hi3 = shard_range(total, rank, world)      # contiguous shards, sizes differ by at most one pair
        P3 = hi3 - first
        log(f"config3: {total} pairs over {world} rank(s), rank {rank}: [{first}, {hi3})")
        do_oracle = oracle if world == 1 else None
        wl = DeviceWorkload(torch, synth, panel, P3, 150, 12, first, dev, threads, do_oracle, cpu_threads())
        out_cap = max(1 << 16, P3 // 4)
        db = wl.gf_batch()
        barrier()
        ms_total, clocks, stats, parts, d_outs, d_ns, _ = time_device_steps(torch, lib, [h], db, out_cap, a.steps, a.warmup,
                                                                            local_rank, barrier)
        ms_max = all_max(ms_total)
        n = int(d_ns[0].item())
        n_all = all_sum(n)
        ms_step = ms_max / a.steps
        rec = {"workload": f"synthetic 2x150bp, {total} pairs in all, split over {world} B200 (~{total // world} pairs per rank, index "
                           "replicated, no exchange step) (BASELINE.json configs[2])",
               "pairs_total": total, "n_gpus": world, "scaling": "strong", "value": total / (ms_step / 1e3), "unit": UNIT,
               "ms_per_step": ms_step, "steps": a.steps, "matches": n_all, "clocks": clocks,
               "roofline": roofline_block(stats[0], parts, ms_step, P3, 150, n, peak, peak_src),
               "device_bytes_inputs_per_rank": 4 * P3 * 150}
        if do_oracle is not None:
            rec["parity"] = parity_record(gpu_records(torch, d_outs[0], n), wl.oracle_all, P3, f"all {P3} pairs")
            if not rec["parity"]["identical"]:
                failures.append("config3: GPU records differ from the oracle's")
        else:
            rec["parity"] = None
        del d_outs, d_ns
        wl.free(torch)
        if rank == 0:
            configs["config3_100M_strong"] = rec

    # -------------------------------------------------------------------------------------------- Matcher pass
    if "matcher" in legs and rank == 0:
        from genefuserust_b200.host import Matcher
        nb = a.matcher_mbases << 20
        log(f"matcher: {nb} reference bases")
        # 24 contigs like a genome's chromosomes; soft-masked stretches, N runs and poly-A every few Mbases
        rng = np.random.default_rng(7)
        host_ref = torch.empty(nb, dtype=torch.uint8, pin_memory=True)
        arr = host_ref.numpy()
        synth.lib().gfs_random_bases(20240202, arr.ctypes.data, nb)
        for s0 in rng.integers(0, nb - 70000, nb >> 18):       # one gap / soft-masked stretch / poly-A per 256 kbases
            arr[s0:s0 + 3000] |= 0x20
            arr[s0 + 4000:s0 + 4100] = ord("N")
            arr[s0 + 5000:s0 + 5040] = ord("A")
        cuts = [0] + sorted(int(x) for x in rng.integers(1 << 20, nb - (1 << 20), 23)) + [nb]
        contigs = [arr[cuts[i]:cuts[i + 1]] for i in range(24)]
        seqs = [b"ACGTTGCAAGCTTAGC" * 10, b"acgtnnACGT" * 15]
        sampler = ClockSampler(local_rank).start()
        Matcher(contigs, device=local_rank).close()       # warm-up (module load, pinned tables)
        t_begin = time.perf_counter()
        walls, infos = [], []
        for _ in range(3):
            t0 = time.perf_counter()
            m = Matcher(contigs, device=local_rank)
            walls.append(time.perf_counter() - t0)
            infos.append(m.info())
            flags, res, rc_m = m.remove_alignables(seqs)
            m.close()
        # resident reference: the scan kernel alone, inputs in HBM
        d_ref = host_ref.to(dev)
        torch.cuda.synchronize()
        dcontigs = [(d_ref.data_ptr() + cuts[i], cuts[i + 1] - cuts[i]) for i in range(24)]
        dinf = []
        for _ in range(4):
            m = Matcher(dcontigs, device=local_rank)
            dinf.append(m.info())
            dres = m.remove_alignables(seqs)[1]
            m.close()
        t_end = time.perf_counter()
        clocks = sampler.stop(t_begin, t_end)
        scan_ms = sorted(i.ms_scan for i in dinf[1:])[1]
        inf = infos[-1]
        wall = sorted(walls)[1]
        rec = {"workload": f"Matcher pass (FusionMapper::remove_alignables, matcher.rs): {nb} reference bases in 24 contigs "
                           "(pinned host memory) streamed through gf_reference_create; SURVEY 8(a) row M / 8(f) #4b",
               "bases": nb, "value": nb / wall, "unit": "reference bases/s end to end (host wall clock, H2D inside)",
               "ms_per_pass_e2e": 1e3 * wall, "ms_pass_device_span": inf.ms_total, "ms_scan_kernels": inf.ms_scan,
               "h2d_bytes": int(inf.h2d_bytes),
               "h2d_gbs": inf.h2d_bytes / wall / 1e9, "kernel_launches": int(inf.kernel_launches),
               "key_positions": [int(x) for x in inf.key_positions], "clocks": clocks,
               "reference_cost_of_the_same_pass": "13-18 s of the reference's wall clock on hg19 / hg38 (benchmark_res/bench_res.md:8-9)",
               "roofline": {"bound": "hbm", "kernel": "k_ref_scan (reference resident in HBM, 1 byte per base read, nothing written)",
                            "achieved": nb / (scan_ms / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                            "frac": nb / (scan_ms / 1e3) / 1e9 / peak, "kernel_ms": scan_ms, "peak_source": peak_src,
                            "algorithmic_bytes_per_launch": nb}}
        if oracle is not None:
            import _oracle
            t0 = time.perf_counter()
            oflags, ores, orc_rc = _oracle.remove_alignables([c.tobytes() for c in contigs], seqs)
            o_s = time.perf_counter() - t0
            ok = (rc_m, res.astuple()) == (orc_rc, ores.astuple()) and dres.astuple() == ores.astuple()
            rec["parity"] = {"bases": nb, "identical": bool(ok), "gpu": list(res.astuple()), "oracle": list(ores.astuple()),
                             "checked_against": "literal CPU restatement of matcher.rs (oracle/gf_oracle_matcher.cpp)"}
            rec["cpu_baseline"] = {"value": nb / o_s, "unit": "reference bases/s", "cores": 1, "kind": "port",
                                   "sample": f"the same {nb} bases, {o_s:.1f} s"}
            if not ok:
                failures.append("matcher: GPU result differs from the oracle's")
        configs["matcher_pass"] = rec
        del d_ref, host_ref

    if rank == 0:
        if not line:     # main leg not selected: still one well-formed line
            line = {"metric": METRIC, "value": None, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3),
                    "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/int64", "data": "synthetic",
                    "config": config_dict(a)}
        line["configs"] = configs
        line["legs"] = legs
        if failures:
            line["failures"] = failures
        json_out.write(json.dumps(line) + "\n")
        json_out.flush()
    if oracle is not None:
        oracle.close()
    mapper.close()
    if world > 1:
        dist.destroy_process_group()
    if failures:
        log("FAILED:", failures)
        sys.exit(1)


if __name__ == "__main__":
    main()
