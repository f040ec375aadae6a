"""The reference arm of bench.py (`--impl reference`) needs no GPU: it times the CPU port of the path and must print one
JSON line with the contract's keys."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "3",
                          "--records", "20000"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert key in d, key
    assert d["impl"] == "reference" and d["unit"] == "records/s" and d["higher_is_better"] is True and d["steps"] == 2
    assert d["value"] > 0 and d["gpu_launches"] == 0 and d["vs_baseline"] is None and d["dtype"] == "u8"
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and 1 <= cb["cores"] <= (os.cpu_count() or 1) and cb["value"] == d["value"] and "sample" in cb
    # both of the reference's chunk settings are timed (its own NUM_CHUNKS = 8, and 4 chunks per usable core)
    assert [s["num_chunks"] for s in cb["settings"]] == [8, 4 * cb["cpus"]["usable"]]
    assert cb["cpus"]["usable"] <= cb["cpus"]["affinity"]
    # the same configuration keys as the GPU arm (the driver compares the two lines' `config`)
    assert d["config"]["records_per_gpu"] == 20000 and d["config"]["num_chunks"] == 8 and "workload" in d["config"]


def test_usable_cores_respects_affinity_and_quota():
    sys.path.insert(0, ROOT)
    import bench
    n, aff, quota = bench.usable_cores()
    assert 1 <= n <= aff
    if quota is not None:
        assert n <= max(1, int(quota + 0.999))


def test_steps_below_one_is_an_error():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"], capture_output=True,
                         text=True, timeout=120, cwd=ROOT)
    assert out.returncode != 0 and "--steps" in out.stderr


@pytest.mark.parametrize("workload", ["kafka", "flat", "wide"])
def test_dump_flattening_keeps_every_value(workload, coracle):
    """`--dump-outputs` writes each column through bench.flatten_arrow: float32/float64 arrays from which the rows can be
    read back exactly (here from batches the C oracle decodes, sliced so that the arrays carry offsets)."""
    import numpy as np
    import pyarrow as pa
    sys.path.insert(0, ROOT)
    import bench
    import workloads
    from oracle import pyoracle as po
    n = 3000
    sj, data, off = workloads.generate(workload, n, seed=5)
    recs = [data[off[i]:off[i + 1]].tobytes() for i in range(n)]
    batch = po.canon_to_batch(coracle.decode(sj, recs), po.to_arrow_schema(po.parse_schema(sj))).slice(1000, 1500)
    out = {}
    for name, col in zip(batch.schema.names, batch.columns):
        bench.flatten_arrow(name, col, out)
    assert all(a.dtype in (np.float32, np.float64) for a in out.values())
    assert 0 < sum(a.nbytes for a in out.values()) < 64 * 1500 * 1024

    def text(prefix, row):
        lens = out[prefix + ".len"].astype(np.int64)
        start = int(lens[:row].sum())
        return bytes(out[prefix + ".bytes"][start:start + lens[row]].astype(np.uint8)).decode()

    def i64(prefix, row):
        hi, lo = out[prefix][row]
        return int(hi) * 2 ** 32 + int(lo)

    rows = batch.to_pylist()
    for r in (0, 1, 777, 1499):
        want = rows[r]
        if workload == "flat":
            assert (out["i"][r], i64("l", r), out["f"][r], out["d"][r], out["b"][r]) == (want["i"], want["l"], want["f"], want["d"], want["b"])
            assert text("s", r) == want["s"]
        elif workload == "kafka":
            assert i64("created_at", r) == want["created_at"] and text("class", r) == want["class"]
            assert out["name.valid"][r] == (want["name"] is not None) and (want["name"] is None or text("name", r) == want["name"])
            assert out["emails.len"][r] == len(want["emails"]) and out["phone_numbers.len"][r] == len(want["phone_numbers"])
        else:
            assert i64("id", r) == want["id"] and out["ml.len"][r] == len(want["ml"])
    if workload == "kafka":
        assert len(out["emails.item.valid"]) == sum(len(x["emails"]) for x in rows)
        assert len(out["phone_numbers.item.keys.len"]) == sum(len(x["phone_numbers"]) for x in rows)


def test_roofline_traffic_comes_from_a_committed_capture():
    """`roofline.traffic` of the bench line is the DRAM byte count of a committed ncu capture of the fused kernel for the
    bench's own workload and size (the first, current, entry of profiles/traffic.json) and names that capture."""
    sys.path.insert(0, ROOT)
    import bench
    traffic, capture = bench.traffic_of("kafka", 10_000_000)
    assert isinstance(traffic, int) and traffic > 0
    algorithmic = 1_170_821_397 + 80_000_008 + 1_670_247_592          # SURVEY 8(d): input + offsets + Arrow buffers
    assert 0.9 * algorithmic < traffic < 1.2 * algorithmic             # the fused pass reads the input once
    assert capture and os.path.exists(os.path.join(ROOT, capture.split(" ")[0]))
    assert bench.traffic_of("kafka", 123) == (None, None)              # no capture for other sizes: reported as null
