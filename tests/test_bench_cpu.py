"""bench.py pieces that need no GPU: the response bytes the timed decode consumes are what the oracle builds, the workloads'
request/response units are what BASELINE.json's configs say, the CPU legs run the UNMODIFIED reference and return well-formed
records, the reference arm prints one JSON line with the contract's keys and honours --steps / --warmup."""
import json
import os
import subprocess
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
import bench  # noqa: E402
from oracle import wire_oracle  # noqa: E402


def test_response_wire_parts_are_the_oracles_bytes():
    x = np.random.default_rng(0).standard_normal((64, 48)).astype(np.float32)
    pre, suf = bench.response_wire_parts(b"y", (64, 48), x.nbytes)
    assert pre + x.tobytes() + suf == wire_oracle.build_predict_response([("y", x)])
    head = bench.request_wire_parts(b"x", (64, 48), x.nbytes)
    assert head + x.tobytes() == wire_oracle.encode_predict_request("default", 1, [("x", x)])


def test_workload_units_follow_the_configs():
    c2, c3, c4, c5 = bench.C2(), bench.C3(), bench.C4(), bench.C5()
    m, v, ins, rk, rx = c2.unit(1)
    assert (m, v, rk) == ("default", 1, "y") and ins[0][0] == "x" and ins[0][1].shape == (1024, 1024) and ins[0][1].dtype == np.float32
    assert rx is ins[0][1] and c2.batch == 256 and c2.scaling == "weak"
    # every float32 tensor carries the sNaN probe, and the expected decode has it quieted (SURVEY Q3)
    assert ins[0][1].view(np.uint32)[0, 0] == 0x7F800001 and bench.quiet_f32(rx).view(np.uint32)[0, 0] == 0x7FC00001
    m, v, ins, rk, rx = c3.unit(7)
    assert [k for k, _ in ins] == ["image", "label"] and ins[0][1].shape == (3, 224, 224) and ins[1][1].tolist() == [7] and ins[1][1].dtype == np.int64
    assert rk == "scores" and rx.shape == (1000,) and c3.batch == 256
    m, v, ins, rk, rx = c4.unit(0)
    assert ins[0][1].dtype == np.float16 and ins[0][1].shape == (8, 512, 1024) and rx.dtype == np.float32 and c4.wire_dtype == 1 and c4.out_dtype == 19
    assert c4.expected_decoded(0, rx).tobytes() == ins[0][1].tobytes()         # fp16 -> fp32 -> fp16: exact
    assert c5.batch == 8192 and c5.sharded and c5.scaling == "strong" and c5.unit(3)[2][0][0] == "image"


def test_c5_request_is_the_golden_one_apart_from_the_probe():
    """Request 3 of C5 without the sNaN probe is tests/golden/requests.json `c5_req3` (what the unmodified reference emits)."""
    import hashlib

    with open(os.path.join(REPO, "tests", "golden", "requests.json")) as fh:
        gold = json.load(fh)["cases"]["c5_req3"]
    x = np.random.default_rng(3).standard_normal((3, 224, 224), dtype=np.float32)
    wire = wire_oracle.encode_predict_request("default", 1, [("image", x)])
    assert len(wire) == gold["wire"]["len"] and hashlib.sha256(wire).hexdigest() == gold["wire"]["sha256"]
    y = bench.C5().unit(3)[2][0][1]
    assert np.array_equal(y.reshape(-1)[4:], x.reshape(-1)[4:])


def test_cpu_baseline_leg_runs_the_unmodified_reference():
    r = bench.cpu_baseline("c2", budget_s=0.5, max_units=2)
    assert r["cores"] == 1 and r["unit"] == "GB/s" and 0 < r["value"] < 1.0
    assert r["sample"].startswith("2 request/response units of c2")
    from baseline import ref_loader

    if ref_loader.available():
        assert r["kind"] == "reference"
        t, origin = ref_loader.load()
        assert "reference" in origin and not t.__file__.startswith(os.path.join(REPO, "min-tfs-client_b200"))
    assert bench.cpu_c_oracle(1)["value"] > r["value"]          # plain C beats per-element Python


def test_host_cores_is_sane():
    h = bench.host_cores()
    assert 1 <= h["used"] <= h["affinity"]


def test_numa_binding_is_best_effort():
    assert isinstance(bench.bind_to_gpu_numa_node(0), str)       # no GPU here: says why it did nothing


def test_reference_arm_prints_one_contract_line():
    env = dict(os.environ, RANK="0", B200TFS_REF_WORKERS="2")
    out = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1", "--workload", "c3"],
                         capture_output=True, text=True, env=env, timeout=600).stdout.strip().splitlines()
    assert len(out) == 1
    line = json.loads(out[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "config", "cpu_baseline", "e2e"):
        assert key in line
    assert line["impl"] == "reference" and line["e2e"]["h2d_bytes_per_step"] == 0
    assert line["steps"] == 2 and line["warmup"] == 1                      # honoured, not clamped
    assert line["config"]["workload"] == bench.C3().title                   # the same workload string as the GPU arm's line
    cb = line["cpu_baseline"]
    assert cb["cores"] == 2 and cb["kind"] in ("reference", "port") and 0 < cb["parallel_efficiency"] <= 1.5 and cb["one_core_gbs"] > 0
    # a rank other than 0 does no work and prints nothing
    out1 = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--steps", "1"], capture_output=True, text=True,
                          env=dict(os.environ, RANK="1"), timeout=60)
    assert out1.returncode == 0 and out1.stdout.strip() == ""
