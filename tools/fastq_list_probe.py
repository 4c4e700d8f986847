#!/usr/bin/env python3
"""developer tool: one FASTQ stream against a list of indices (gf_fastq_stream_create_list) against one stream per index.

The shape of the bench's `list16` leg on the bench's FASTQ inputs (full panel, 2x150 reads, seed 12): K = 16 indices, alternating
the full panel and its 40-gene subset, and two workloads, the 250 k-pair `fastq_gz` workload as BGZF and the 1 M-pair
`fastq_text` workload as plain text.  Two arms per workload:
  list     one stream over the K indices: every chunk copied, inflated, split and converted once, then mapped per index;
  singles  K streams, one per index, each fed the same pieces (so every chunk is copied, inflated, split and converted K times).
A pass is the whole workload on one arm: the files fed in 8 MiB pieces, the streams finished (every record of the files is
mapped, in the same chunks every pass: 256 MiB of text per mate, the rest at the finish), every index's records taken.  The arms
alternate, one full warm-up pass each (pinned buffers, device workspaces) and then `--passes` timed passes each; every index's
records (with --keep-reads also its descriptors and lines) must be identical between the arms in every pass.  Then K = 1: a list
stream of one against gf_fastq_stream_create, the same way.  Prints one JSON line with the median and mean ms per pass and the
GPU's name and power limit, read in the same run.
usage: python tools/fastq_list_probe.py [--passes 8] [--keep-reads]"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np  # noqa: E402

import __graft_entry__ as ge  # noqa: E402

ge.build()
from fastq_reads_probe import fastq_text  # noqa: E402
from genefuserust_b200 import synth  # noqa: E402
from genefuserust_b200._abi import GF_OK, gf_fastq_read_pair, gf_match  # noqa: E402
from genefuserust_b200.host import FusionMapper, bgzf_compress  # noqa: E402


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                              text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # (reported, not fatal)
        return f"unknown ({e})"


def check(lib, rc):
    if rc != GF_OK:
        raise RuntimeError(lib.gf_last_error().decode())


class Arm:
    """streams over `handles`: one list stream (gf_fastq_stream_create_list) or one stream per handle (gf_fastq_stream_create)"""

    def __init__(self, lib, handles, fmt, as_list, keep):
        self.lib, self.keep, self.n = lib, keep, len(handles)
        self.streams = []
        groups = [handles] if as_list else [[h] for h in handles]
        for g in groups:
            sh = C.c_void_p()
            if as_list:
                check(lib, lib.gf_fastq_stream_create_list((C.c_void_p * len(g))(*g), len(g), 1, fmt, 0, C.byref(sh)))
            else:
                check(lib, lib.gf_fastq_stream_create(g[0], 1, fmt, 0, C.byref(sh)))
            if keep:
                check(lib, lib.gf_fastq_stream_keep_reads(sh))
            self.streams.append((sh, len(g)))

    def one_pass(self, k1, k2, bufs):
        lib = self.lib
        out_m, pairs, text = bufs
        piece = 8 << 20
        got = []
        t0 = time.perf_counter()
        for sh, nh in self.streams:
            for p0 in range(0, max(len(k1), len(k2)), piece):
                n1, n2 = max(0, min(piece, len(k1) - p0)), max(0, min(piece, len(k2) - p0))
                check(lib, lib.gf_fastq_stream_feed(sh, C.cast(k1.ctypes.data + p0, C.c_char_p) if n1 else None, n1,
                                                    C.cast(k2.ctypes.data + p0, C.c_char_p) if n2 else None, n2))
            check(lib, lib.gf_fastq_stream_finish(sh))
            for h in range(nh):
                n, npair, ntext = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
                if self.keep:
                    check(lib, lib.gf_fastq_stream_take_reads_index(sh, h, out_m, len(out_m), C.byref(n), pairs, len(pairs),
                                                                    C.byref(npair), C.cast(text.ctypes.data, C.c_void_p), len(text),
                                                                    C.byref(ntext)))
                else:
                    check(lib, lib.gf_fastq_stream_take_index(sh, h, out_m, len(out_m), C.byref(n)))
                # (copied inside the timed region: the same bytes in both arms)
                got.append((bytes(C.string_at(C.addressof(out_m), C.sizeof(gf_match) * n.value)),
                            bytes(C.string_at(C.addressof(pairs), C.sizeof(gf_fastq_read_pair) * npair.value)),
                            text[:ntext.value].tobytes()))
        return time.perf_counter() - t0, got

    def calls(self):
        c = C.c_uint64(0)
        total = 0
        for sh, _ in self.streams:
            self.lib.gf_fastq_stream_get_counts(sh, None, None, C.byref(c))
            total += int(c.value)
        return total

    def close(self):
        for sh, _ in self.streams:
            self.lib.gf_fastq_stream_destroy(sh)


def compare(lib, handles, name, fmt, e1, e2, passes, keep, bufs):
    """list stream against single-index streams, alternating; returns the workload's record"""
    k1, k2 = np.frombuffer(e1, dtype=np.uint8), np.frombuffer(e2, dtype=np.uint8)
    arms = {"list": Arm(lib, handles, fmt, True, keep), "singles": Arm(lib, handles, fmt, False, keep)}
    times = {k: [] for k in arms}
    for k in arms:                      # warm-up: a whole pass that maps every chunk
        arms[k].one_pass(k1, k2, bufs)
    calls0 = {k: a.calls() for k, a in arms.items()}
    records = 0
    for _ in range(passes):
        got = {}
        for k, a in arms.items():
            dt, got[k] = a.one_pass(k1, k2, bufs)
            times[k].append(dt)
        if got["list"] != got["singles"]:
            raise RuntimeError(f"{name}: the list stream's output differs from the single-index streams'")
        records = sum(len(r) // C.sizeof(gf_match) for r, _p, _t in got["list"])
    calls = {k: (a.calls() - calls0[k]) / passes for k, a in arms.items()}
    for a in arms.values():
        a.close()
    med = {k: 1e3 * sorted(v)[len(v) // 2] for k, v in times.items()}
    mean = {k: 1e3 * sum(v) / len(v) for k, v in times.items()}
    return {"indices": len(handles), "ms_per_pass_median": {k: round(v, 2) for k, v in med.items()},
            "ms_per_pass_mean": {k: round(v, 2) for k, v in mean.items()},
            "singles_over_list_median": round(med["singles"] / med["list"], 3),
            "singles_over_list_mean": round(mean["singles"] / mean["list"], 3),
            "map_calls_per_pass": calls, "records_per_pass_all_indices": records, "identical": True,
            "ms_per_pass_all": {k: [round(1e3 * t, 2) for t in v] for k, v in times.items()}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--passes", type=int, default=8)
    ap.add_argument("--keep-reads", action="store_true", help="gather the matched pairs' lines too (compared as well)")
    a = ap.parse_args()
    P, Pz, L, K = 1_000_000, 250_000, 150, 16
    panel = synth.make_panel()
    genes = panel.genes()
    batch = synth.generate_pairs(panel, P, read_len=L, seed=12, threads=os.cpu_count())
    t1, t2 = fastq_text(batch.seq1, batch.qual1, 1, P, L), fastq_text(batch.seq2, batch.qual2, 2, P, L)
    rec = len(t1) // P
    work = [("fastq_gz bgzf 250k pairs", 1, bgzf_compress(t1[:Pz * rec]), bgzf_compress(t2[:Pz * rec])),
            ("fastq_text 1M pairs", 0, t1, t2)]
    mappers = [FusionMapper.from_gene_spans(genes if k % 2 == 0 else genes[:40]) for k in range(K)]
    lib = mappers[0].lib
    handles = [m.m_indexer.h for m in mappers]
    bufs = ((gf_match * (1 << 21))(), (gf_fastq_read_pair * (1 << 21))(), np.zeros(1 << 29, dtype=np.uint8))
    res = {"gpu": gpu_info(), "passes": a.passes, "keep_reads": a.keep_reads, "workloads": {}}
    for name, fmt, e1, e2 in work:
        res["workloads"][name] = {"K16": compare(lib, handles, name, fmt, e1, e2, a.passes, a.keep_reads, bufs),
                                  "K1": compare(lib, handles[:1], name, fmt, e1, e2, a.passes, a.keep_reads, bufs)}
    for m in mappers:
        m.close()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
