"""CPU tier: the parts of bench.py that do not need a GPU — argument surface, workload inventories of the BASELINE configs, the CPU arm
(--impl reference) end to end on the small workload, and the one-JSON-line contract of that arm."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from tools import synth  # noqa: E402


def args_for(*argv):
    old = sys.argv
    sys.argv = ["bench.py", *argv]
    try:
        return bench.parse()
    finally:
        sys.argv = old


def test_defaults_follow_the_contract():
    a = args_for()
    assert (a.gpus, a.impl, a.workload, a.fanout) == (1, "ours", "llama3-8b", "p2p") and a.warmup >= 3 and a.steps >= 1  # fan-out only matters at N > 1
    assert not (a.nvls_compare or a.kernel_only or a.no_secondary) and a.qtype == "Q4_K"
    assert args_for("--workload", "gpt2").fanout == "p2p" and args_for("--fanout", "raw").fanout == "raw" and args_for("--fanout", "pull").fanout == "pull"


def test_workload_inventories_match_the_baseline_configs():
    """SURVEY.md §8(d): Llama-3-8B = 291 tensors / 16,060,522,496 B; Llama-3-70B = 723 tensors / 141,107,412,992 B; GPT-2-small = 148 tensors /
    497,759,232 B; Mixtral-8x7B merged experts = 323 tensors."""
    s = bench.workload_spec(args_for("--workload", "llama3-8b"))
    assert len(s["tensors"]) == 291 and synth.total_bytes(s["tensors"]) == 16_060_522_496 and s["mode"] == "broadcast"
    s = bench.workload_spec(args_for("--workload", "llama3-70b-scatter"))
    assert len(s["tensors"]) == 723 and synth.total_bytes(s["tensors"]) == 141_107_412_992 and s["mode"] == "scatter"
    s = bench.workload_spec(args_for("--workload", "gpt2"))
    assert len(s["tensors"]) == 148 and synth.total_bytes(s["tensors"]) == 497_759_232
    s = bench.workload_spec(args_for("--workload", "mixtral-q4k"))
    assert len(s["tensors"]) == 323 and "q4_k" in s["name"]
    q = synth.total_bytes(s["tensors"])
    assert 26.2e9 < q < 26.4e9  # ~26.27 GB of Q4_K blocks + F32 norms / routers
    s6 = bench.workload_spec(args_for("--workload", "mixtral-q4k", "--qtype", "Q6_K", "--layers", "2"))
    assert "q6_k" in s6["name"] and "REDUCED to 2 layers" in s6["name"] and {t[1] for t in s6["tensors"]} == {"Q6_K", "F32"}
    with pytest.raises(SystemExit):
        bench.workload_spec(args_for("--workload", "mixtral-q4k", "--qtype", "F32"))


def test_reference_arm_prints_one_json_line(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "gpt2", "--layers", "2", "--steps", "1", "--warmup", "1",
                        "--data-dir", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == bench.METRIC and d["unit"] == bench.UNIT and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"] > 0
    assert d["e2e"] == {"value": d["value"], "unit": bench.UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0} and d["gpu_launches"] == 0
    assert d["config"]["workload"].startswith("GPT-2-small") and d["n_gpus"] == 1 and d["steps"] == 1
    assert d["config"]["same_config"] is True and "whole checkpoint" in d["cpu_baseline"]["sample"]


def test_dump_outputs_writes_every_pool_tensor_and_samples_large_ones_by_seed(tmp_path, monkeypatch):
    """bench.dump_outputs (--dump-outputs) over an oracle pool: a tensor that fits its share comes out whole, in its shape, value for value;
    a larger one as runs of DUMP_RUN consecutive elements of the tensor; a second dump is identical; the files stay within the budget."""
    import numpy as np

    from oracle import oracle
    from tests import helpers
    p = str(tmp_path / "m.safetensors")
    helpers.mixed_safetensors(p)
    shards, recs = oracle.index_path(p)
    pool, plan = oracle.expected_pool(shards, recs)
    tensors = [dict(name=t["name"], dtype=t["dtype"], shape=t["shape"], offset=t["pool_offset"], nbytes=t["nbytes"]) for t in plan]
    monkeypatch.setattr(bench, "DUMP_BYTES", 512 << 10)  # h.bf16.big (716,800 values) is sampled, the rest fits
    monkeypatch.setattr(bench, "DUMP_RUN", 256)
    for k in ("a", "b"):
        bench.dump_outputs(str(tmp_path / k), tensors, lambda off, n: pool[off:off + n].copy())
    assert sorted(os.listdir(tmp_path / "a")) == sorted(t["name"] + ".npy" for t in tensors)
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= (512 << 10) + 128 * len(tensors)
    for t in tensors:
        a, b = np.load(tmp_path / "a" / (t["name"] + ".npy")), np.load(tmp_path / "b" / (t["name"] + ".npy"))
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b, equal_nan=True)
        raw = pool[t["offset"]:t["offset"] + t["nbytes"]]
        full = {"BF16": lambda: (raw.view(np.uint16).astype(np.uint32) << 16).view(np.float32), "F32": lambda: raw.view(np.float32),
                "I64": lambda: raw.view(np.int64).astype(np.float64), "U8": lambda: raw.astype(np.float64), "BOOL": lambda: raw.astype(np.float64)}[t["dtype"]]()
        if t["name"] == "h.bf16.big":
            runs = full.reshape(-1, 256)
            assert a.ndim == 1 and a.size and a.size % 256 == 0 and a.size < full.size
            assert all(any(np.array_equal(r, q, equal_nan=True) for q in runs) for r in a.reshape(-1, 256))
        else:
            assert a.shape == tuple(t["shape"]) and np.array_equal(a.reshape(-1), full, equal_nan=True)


def test_pending_gpu_scripts_point_at_things_that_exist():
    """The GPU command files still to be spent (tools/r02/*.sh; spent ones move to tools/history/) each cost box minutes: they must parse and
    every script they run must exist and parse."""
    import ast
    import glob
    import re
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for sh in sorted(glob.glob(os.path.join(root, "tools", "r02", "*.sh"))):
        assert subprocess.run(["bash", "-n", sh]).returncode == 0, sh
        text = open(sh).read()
        for rel in sorted(set(re.findall(r"\b((?:tools|tests)/[\w/]+\.py)\b", text))):
            path = os.path.join(root, rel)
            assert os.path.exists(path), (sh, rel)
            ast.parse(open(path).read(), rel)


def test_page_cache_warm_up_stripes_every_byte_over_the_ranks(tmp_path):
    """bench.warm_page_cache: the ranks' stripes (32 MiB blocks dealt round-robin) cover every byte of every file exactly once; hidden files
    (the .complete marker) are not data."""
    d = tmp_path / "ck"
    d.mkdir()
    (d / "a.bin").write_bytes(b"x" * (70 << 20))
    (d / "b.bin").write_bytes(b"y" * (5 << 20))
    (d / ".complete").write_text("ok")
    per_rank = [bench.warm_page_cache(str(d), r, 3, passes=1, threads=2) for r in range(3)]
    assert sum(per_rank) == (70 << 20) + (5 << 20) and all(per_rank)
    assert bench.warm_page_cache(str(d), 0, 1, passes=1, threads=3) == (75 << 20)
