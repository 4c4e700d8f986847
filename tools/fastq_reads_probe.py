#!/usr/bin/env python3
"""developer tool: what keeping the reads (gf_fastq_stream_keep_reads) costs a FASTQ stream.

The bench's FASTQ inputs (full panel, 2x150 reads, seed 12): the 1 M-pair `fastq_text` workload fed as a plain stream, and the
250 k-pair `fastq_gz` workload as one gzip member per file and as BGZF.  Per workload one stream keeps the reads and one does
not.  A pass is the whole workload on one of them: the files fed in 8 MiB pieces, the stream finished (so every record of the
files is mapped, in the same chunks every pass: 256 MiB of text per mate, the rest at the finish), the records taken.  The
streams are used alternately, one full warm-up pass each (pinned buffers, device workspaces, the arena of the lines) and then
`--passes` timed passes each.  Prints one JSON line: the median and mean ms per pass with and without the reads, the mapping
calls, matched pairs and bytes the reads add per pass, and the GPU's name and power limit.
usage: python tools/fastq_reads_probe.py [--passes 5]"""
import argparse
import ctypes as C
import gzip
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

import __graft_entry__ as ge  # noqa: E402

ge.build()
from genefuserust_b200 import synth  # noqa: E402
from genefuserust_b200._abi import GF_OK, gf_fastq_read_pair, gf_match  # noqa: E402
from genefuserust_b200.host import FusionMapper, bgzf_compress  # noqa: E402


def fastq_text(seq, qual, mate, P, L):
    name = np.frombuffer(b"@SYN:12:000000000 %d:N:0:ACGT\n" % mate, dtype=np.uint8)
    rec = len(name) + L + 1 + 2 + L + 1
    out = np.empty((P, rec), dtype=np.uint8)
    out[:, :len(name)] = name
    idx = np.arange(P, dtype=np.int64)
    for k in range(9):
        out[:, 8 + 8 - k] = 48 + (idx // 10 ** k) % 10
    o = len(name)
    out[:, o:o + L] = seq.reshape(P, L)
    out[:, o + L] = 10
    out[:, o + L + 1] = 43
    out[:, o + L + 2] = 10
    out[:, o + L + 3:o + 2 * L + 3] = qual.reshape(P, L)
    out[:, o + 2 * L + 3] = 10
    return out.tobytes()


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                              text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # (reported, not fatal)
        return f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--passes", type=int, default=5)
    a = ap.parse_args()
    P, Pz, L = 1_000_000, 250_000, 150
    panel = synth.make_panel()
    batch = synth.generate_pairs(panel, P, read_len=L, seed=12, threads=os.cpu_count())
    t1, t2 = fastq_text(batch.seq1, batch.qual1, 1, P, L), fastq_text(batch.seq2, batch.qual2, 2, P, L)
    rec = len(t1) // P
    z1, z2 = t1[:Pz * rec], t2[:Pz * rec]
    work = [("fastq_text", 0, t1, t2),
            ("fastq_gz gzip_single_member", 1, gzip.compress(z1, compresslevel=1), gzip.compress(z2, compresslevel=1)),
            ("fastq_gz bgzf", 1, bgzf_compress(z1), bgzf_compress(z2))]
    m = FusionMapper.from_gene_spans(panel.genes())
    lib, h = m.lib, m.m_indexer.h
    cap = 1 << 20
    out_m = (gf_match * cap)()
    pairs = (gf_fastq_read_pair * cap)()
    text = np.zeros(1 << 28, dtype=np.uint8)
    res = {"gpu": gpu_info(), "passes": a.passes, "workloads": {}}
    for name, fmt, e1, e2 in work:
        k1, k2 = np.frombuffer(e1, dtype=np.uint8), np.frombuffer(e2, dtype=np.uint8)
        streams = {}
        for keep in (False, True):
            sh = C.c_void_p()
            assert lib.gf_fastq_stream_create(h, 1, fmt, 0, C.byref(sh)) == GF_OK
            if keep:
                assert lib.gf_fastq_stream_keep_reads(sh) == GF_OK
            streams[keep] = sh
        times = {False: [], True: []}
        got = {False: [], True: []}
        extra = {"pairs": 0, "bytes": 0}

        def one_pass(keep):
            sh = streams[keep]
            piece = 8 << 20
            t0 = time.perf_counter()
            for p0 in range(0, max(len(e1), len(e2)), piece):
                n1, n2 = max(0, min(piece, len(e1) - p0)), max(0, min(piece, len(e2) - p0))
                rc = lib.gf_fastq_stream_feed(sh, C.cast(k1.ctypes.data + p0, C.c_char_p) if n1 else None, n1,
                                              C.cast(k2.ctypes.data + p0, C.c_char_p) if n2 else None, n2)
                if rc != GF_OK:
                    raise RuntimeError(lib.gf_last_error().decode())
            if lib.gf_fastq_stream_finish(sh) != GF_OK:
                raise RuntimeError(lib.gf_last_error().decode())
            n, npair, ntext = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
            if keep:
                rc = lib.gf_fastq_stream_take_reads(sh, out_m, cap, C.byref(n), pairs, cap, C.byref(npair),
                                                    C.cast(text.ctypes.data, C.c_void_p), len(text), C.byref(ntext))
            else:
                rc = lib.gf_fastq_stream_take(sh, out_m, cap, C.byref(n))
            dt = time.perf_counter() - t0
            if rc != GF_OK:
                raise RuntimeError(lib.gf_last_error().decode())
            return dt, [out_m[i].astuple() for i in range(n.value)], int(npair.value), int(ntext.value)

        def calls(keep):
            c = C.c_uint64(0)
            lib.gf_fastq_stream_get_counts(streams[keep], None, None, C.byref(c))
            return int(c.value)
        for keep in (False, True):          # warm-up: a whole pass that maps every chunk
            one_pass(keep)
        calls0 = {k: calls(k) for k in (False, True)}
        for _ in range(a.passes):
            for keep in (False, True):
                dt, recs, npair, ntext = one_pass(keep)
                times[keep].append(dt)
                got[keep] += recs
                if keep:
                    extra["pairs"] += npair
                    extra["bytes"] += npair * C.sizeof(gf_fastq_read_pair) + ntext
        per_pass_calls = {k: (calls(k) - calls0[k]) / a.passes for k in (False, True)}
        for keep in (False, True):
            lib.gf_fastq_stream_destroy(streams[keep])
        med = {k: 1e3 * sorted(v)[len(v) // 2] for k, v in times.items()}
        mean = {k: 1e3 * sum(v) / len(v) for k, v in times.items()}
        same = got[False] == got[True]
        res["workloads"][name] = {
            "ms_per_pass_median": {"reads_not_kept": round(med[False], 2), "reads_kept": round(med[True], 2)},
            "overhead_pct_of_median": round(100 * (med[True] / med[False] - 1), 2),
            "ms_per_pass_mean": {"reads_not_kept": round(mean[False], 2), "reads_kept": round(mean[True], 2)},
            "overhead_pct_of_mean": round(100 * (mean[True] / mean[False] - 1), 2),
            "map_calls_per_pass": per_pass_calls,
            "ms_per_pass_all": {"reads_not_kept": [round(1e3 * t, 2) for t in times[False]],
                                "reads_kept": [round(1e3 * t, 2) for t in times[True]]},
            "matched_pairs_per_pass": extra["pairs"] // a.passes, "bytes_returned_per_pass": extra["bytes"] // a.passes,
            "records_per_pass": len(got[True]) // a.passes, "records_identical": same}
    m.close()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
