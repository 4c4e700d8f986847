"""bench.py --dump-outputs: the records of the timed path as float64 .npy files, identical from run to run.  On the CPU the
reference arm (the oracle) is the timed path; the main leg writes through the same function."""
import os
import subprocess
import sys

import numpy as np

import _oracle as orc
from genefuserust_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARGS = ["--impl", "reference", "--steps", "2", "--warmup", "1", "--pairs", "30000", "--panel-scale", "0.05", "--seed", "7"]


def run_dump(out):
    subprocess.check_call([sys.executable, os.path.join(ROOT, "bench.py")] + ARGS + ["--dump-outputs", out],
                          stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    return {f[:-4]: np.load(os.path.join(out, f)) for f in sorted(os.listdir(out))}


def test_dump_outputs_reproducible_and_exact(tmp_path):
    a = run_dump(str(tmp_path / "a"))
    b = run_dump(str(tmp_path / "b"))
    assert sorted(a) == sorted(b) and all(np.array_equal(a[k], b[k]) for k in a)
    assert all(v.dtype == np.float64 for v in a.values())
    panel = synth.make_panel(scale=0.05)
    batch = synth.generate_pairs(panel, 30000, read_len=150, seed=7)
    want = orc.OracleIndex(panel.genes()).scan(batch, threads=4)
    assert len(want) > 5 and a["n_records"].tolist() == [len(want)]
    fields = ["pair_idx", "source", "used_rc", "reversed", "read_break", "l_contig", "l_pos", "r_contig", "r_pos", "gap",
              "l_dist", "r_dist", "seq_len", "merge_olen", "merge_diff", "filter_flags"]
    assert sorted(a) == sorted(fields + ["n_records"])
    got = list(zip(*(a[f].astype(np.int64).tolist() for f in fields)))
    assert got == [tuple(r) for r in want]


def test_dump_outputs_samples_large_outputs(tmp_path, monkeypatch):
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 1 << 20)
    recs = np.zeros(100_000, dtype=bench.match_dtype())
    recs["pair_idx"] = np.arange(len(recs))
    recs["l_pos"] = -np.arange(len(recs))
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), recs)
    a, b = (str(tmp_path / d) for d in ("a", "b"))
    assert sum(os.path.getsize(os.path.join(a, f)) for f in os.listdir(a)) <= 1 << 20
    assert np.load(os.path.join(a, "n_records.npy")).tolist() == [len(recs)]
    rows = np.load(os.path.join(a, "pair_idx.npy"))
    assert 1000 < len(rows) < len(recs) and np.all(np.diff(rows) > 0)          # a sample, in record order
    assert np.array_equal(rows, np.load(os.path.join(b, "pair_idx.npy")))        # the same sample every time
    assert np.array_equal(np.load(os.path.join(a, "l_pos.npy")), -rows)          # the fields of the same rows
