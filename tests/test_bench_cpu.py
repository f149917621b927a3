"""CPU-only checks of bench.py: the reference arm runs (it is the one bench leg that needs no GPU),
prints one well-formed JSON line, and the interval/traffic helpers behave."""
import importlib.util
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent


def _bench():
    spec = importlib.util.spec_from_file_location("bench_mod", ROOT / "bench.py")
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_union_of_overlapping_kernel_intervals():
    b = _bench()
    assert b.union_ms([]) == 0
    assert b.union_ms([(0, 10), (5, 20), (30, 40)]) == 30
    assert b.union_ms([(3, 4), (0, 10)]) == 10


def test_traffic_is_read_from_committed_ncu_summaries():
    b = _bench()
    tr = b.ncu_traffic()
    if tr is not None:       # K1 reads the batch once, K3 (bulk + long kernel) reads it again: 2.0 x the algorithmic bytes
        assert 1.9 < tr["ratio_to_algorithmic"] < 2.1 and "profiles/" in tr["source"]
        assert abs(tr["total"] - (tr["K1_scan"] + tr["K3_sha_bulk"] + tr["K3_sha_long"])) < 1


def test_instruction_ceiling_counts_every_sm():
    b = _bench()
    c = b.instr_ceiling(148, 1965.0, 500.0)
    assert c["sm_count"] == 148 and 950 < c["alu_pipe_GBps"] < 1000 and abs(c["frac_of_alu_pipe"] - 500.0 / c["alu_pipe_GBps"]) < 1e-9
    assert b.instr_ceiling(148, None, 1.0) is None


def test_cfg4_expected_entries_are_found_by_shape(tmp_path, monkeypatch):
    b = _bench()
    (tmp_path / "profiles").mkdir()
    (tmp_path / "profiles" / "r02_cfg4_expected.json").write_text(json.dumps({"entries": [
        {"world": 2, "files_per_rank": 1024, "file_mib": 64, "chunks": 10, "known": 3}]}))
    monkeypatch.setattr(b, "ROOT", tmp_path)
    assert b.expected_cfg4_hits(2, 1024, 64)["known"] == 3
    assert b.expected_cfg4_hits(4, 1024, 64) is None


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--file-mib", "1"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "GiB/s" and d["value"] > 0 and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]


def test_dump_outputs_writes_the_last_step_records(tmp_path):
    """--dump-outputs: the records of the last timed step as float .npy files, equal to the oracle's for the same
    corpus, and the same files from a second run with the same arguments."""
    import numpy as np

    import oracle
    dumps = []
    for run in ("a", "b"):
        out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                              "--file-mib", "1", "--dump-outputs", str(tmp_path / run)], capture_output=True, text=True,
                             timeout=600)
        assert out.returncode == 0, out.stderr[-2000:]
        dumps.append({n: np.load(tmp_path / run / f"{n}.npy") for n in ("row", "stream", "end_off", "digest", "known")})
    a, b = dumps
    assert all(a[n].dtype in (np.float32, np.float64) for n in a) and sum(a[n].nbytes for n in a) <= 64_000_000
    assert all(np.array_equal(a[n], b[n]) for n in a)
    n_files = int(a["stream"].max()) + 1
    files = oracle.corpus_files(oracle.corpus(seed=2, file_len=1 << 20), 0, n_files)
    ref = oracle.chunk_digest_streams(oracle.config(4 << 20), files)
    assert a["row"].tolist() == list(range(len(ref)))
    assert a["stream"].tolist() == ref["stream"].tolist() and a["end_off"].tolist() == ref["end_off"].tolist()
    assert (a["digest"] == ref["digest"]).all() and not a["known"].any()


def test_dump_outputs_samples_a_large_step(tmp_path, monkeypatch):
    import numpy as np
    b = _bench()
    rec = np.zeros(5000, dtype=[("stream", "<u4"), ("flags", "<u4"), ("end_off", "<u8"), ("digest", "u1", (32,))])
    rec["end_off"] = np.arange(5000) * 7
    rec["digest"] = np.random.default_rng(1).integers(0, 256, (5000, 32))
    known = np.arange(5000) % 3 == 0
    monkeypatch.setattr(b, "DUMP_LIMIT", 156 * 1000)
    for d in ("a", "b"):
        b.dump_outputs(str(tmp_path / d), rec, known)
    rows = np.load(tmp_path / "a" / "row.npy")
    assert len(rows) == 1000 and (np.diff(rows) > 0).all() and (rows == np.load(tmp_path / "b" / "row.npy")).all()
    idx = rows.astype(np.int64)
    assert (np.load(tmp_path / "a" / "end_off.npy") == idx * 7).all()
    assert (np.load(tmp_path / "a" / "digest.npy") == rec["digest"][idx]).all()
    assert (np.load(tmp_path / "a" / "known.npy") == known[idx]).all()
    assert sum((tmp_path / "a" / f).stat().st_size for f in ("row.npy", "stream.npy", "end_off.npy", "digest.npy", "known.npy")) \
        <= b.DUMP_LIMIT + 5 * 128


def test_reference_arm_nonzero_rank_is_silent():
    import os
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"],
                         capture_output=True, text=True, timeout=120, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""
