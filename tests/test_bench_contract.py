"""bench.py's JSON contract, checked on CPU through the reference arm (the oracle on the host cores) and statically for the
GPU arm's line; on a GPU, the arrays --dump-outputs writes."""
import json
import os
import re
import subprocess
import sys

import pytest

from conftest import ROOT

REQUIRED = ["metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
            "data", "config", "e2e", "cpu_baseline"]


def tree_state():
    """(path, size, mtime) of every file of the working tree outside .git"""
    state = set()
    for dp, dns, fns in os.walk(ROOT):
        dns[:] = [d for d in dns if d != ".git"]
        for f in fns:
            st = os.stat(os.path.join(dp, f))
            state.add((os.path.join(dp, f), st.st_size, st.st_mtime_ns))
    return state


def test_reference_arm_prints_one_json_line(orc):
    """and it writes nothing into the tree as build() left it (the oracle fixture builds the oracle first)"""
    before = tree_state()
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--ref-sample-mib", "2"], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr
    assert tree_state() == before, "bench.py wrote into the source tree"       # the tree may be read-only where it runs
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in REQUIRED + ["impl"]:
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "GB/s" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["config"]["workload"].startswith("single 10 GiB-per-GPU synthetic slot (163840 blocks")
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"], capture_output=True, text=True,
                         env=env, timeout=120)
    assert res.returncode == 0 and res.stdout.strip() == ""


def test_gpu_arm_line_has_every_contract_key():
    src = open(os.path.join(ROOT, "bench.py")).read()
    body = src[src.index("        line = {\n            \"metric\""):]
    for k in REQUIRED + ["gpu_launches", "clocks", "roofline", "perms_per_s"]:
        assert f'"{k}"' in body, k
    roof = src[src.index("    roofline = {"):src.index("    traffic_file")]
    for k in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert f'"{k}"' in roof, k
    assert re.search(r'"sm_mhz".*"sm_max_mhz".*"reasons"', src, re.S)


def test_steps_must_be_positive():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"], capture_output=True,
                         text=True, timeout=120)
    assert res.returncode != 0 and "--steps" in res.stderr and res.stdout == ""


@pytest.mark.gpu
def test_gpu_arm_dumps_what_the_last_step_committed(pkg, orc, tmp_path):
    """--dump-outputs on a 1 GiB slot: the root, every block hash and a seeded sample of 32-cell windows of the cell hashes
    the last timed step committed, as float64 limbs; they agree with the JSON line and with the oracle over the same bytes"""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    before = tree_state()
    out = tmp_path / "dump"
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--slot-gib", "1", "--steps", "2", "--warmup", "1", "--no-extras",
                          "--no-e2e", "--no-cpu", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stderr
    assert tree_state() == before, "bench.py wrote into the source tree"
    line = json.loads(res.stdout)
    assert line["steps"] == 2 and line["warmup"] == 1
    d = {f[:-4]: np.load(out / f) for f in os.listdir(out)}
    assert sorted(d) == ["block_hashes", "block_hashes_index", "cell_hashes", "cell_hashes_index", "slot_root"]
    assert all(a.dtype == np.float64 for a in d.values()) and sum(a.nbytes for a in d.values()) <= 64 << 20

    def felts(a):
        return [int.from_bytes(row.astype("<u4").tobytes(), "little") for row in a]
    n_blocks = 16384
    root = felts(d["slot_root"])[0]
    assert hex(root) == line["slot_root"]
    assert d["block_hashes_index"].tolist() == list(range(n_blocks))
    bh = felts(d["block_hashes"])
    assert orc.merkle_root(bh) == root
    idx = d["cell_hashes_index"].astype(np.int64)
    assert len(idx) == bench.DUMP_MAX_NODES < 32 * n_blocks                   # more cells than the cap: a sample of whole blocks
    assert (idx[::32] % 32 == 0).all() and (np.diff(idx[::32]) > 0).all() and (idx.reshape(-1, 32) - idx[::32, None] == np.arange(32)).all()
    ch = felts(d["cell_hashes"])
    for w in (0, 1, len(idx) // 64, len(idx) // 32 - 1):                     # four sampled blocks, re-hashed by the oracle
        b = int(idx[32 * w]) // 32
        raw = bench.synthetic_bytes_host(bench.SEED, b * bench.BLOCK // 8, bench.BLOCK).tobytes()
        cells = [orc.hash_bytes(raw[i * bench.CELL:(i + 1) * bench.CELL]) for i in range(32)]
        assert ch[32 * w:32 * w + 32] == cells, b
        assert orc.merkle_root(cells) == bh[b], b


def test_work_model_matches_the_survey_appendix():
    sys.path.insert(0, ROOT)
    import bench
    assert bench.total_perms(64) == 71679                      # config 1, one slot
    assert bench.total_perms(16384) == 18350079                # 1 GiB
    assert bench.total_perms(163840) == 183500801              # 10 GiB (odd nodes at 5 -> 3 -> 2 -> 1)
    assert bench.total_perms(1638400) == 1835008002            # 100 GiB
    assert bench.total_perms(2097152) == 2348810239            # 128 GiB
