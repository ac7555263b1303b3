"""bench.py's contract surface that needs no GPU: it refuses to run its own arm without a CUDA device (no CPU path),
non-zero ranks of the reference arm exit quietly, both arms name the same workload, and the roofline `traffic` keys it
reads exist in this round's ncu summary (profiles/ncu_traffic.json, written by tools/ncu_traffic.py)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, **env):
    e = dict(os.environ, CUDA_VISIBLE_DEVICES="", **env)
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, env=e, capture_output=True, text=True,
                          timeout=300)


def test_own_arm_fails_loudly_without_a_gpu():
    r = _run(["--steps", "1", "--no-extras", "--no-cpu-baseline"])
    assert r.returncode != 0
    assert "no CUDA device" in (r.stderr + r.stdout) and "no CPU path" in (r.stderr + r.stdout)
    assert not [ln for ln in r.stdout.splitlines() if ln.startswith("{")]      # no result line from a run that did not happen


def test_reference_arm_runs_on_rank_zero_only():
    r = _run(["--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"], RANK="1", WORLD_SIZE="2",
             LOCAL_RANK="1")
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_both_arms_name_the_same_workload_and_the_traffic_keys_exist():
    sys.path.insert(0, ROOT)
    import bench
    cfg = bench.workload_config(1)
    assert cfg == bench.workload_config(1) and "workload" in cfg and "model" not in cfg
    assert bench.workload_config(8)["workload"] == cfg["workload"]
    t = bench.ncu_traffic()
    for key in ("decode_attn_kernel", "decode_attn_kernel_96_rows", "gemm_bf16_2cta_kernel", "source"):
        assert key in t, key
    # traffic is per launch, like the algorithmic bytes it is compared with (SURVEY.md section 8d: 7.68 MB per row and layer)
    assert 1.0 <= t["decode_attn_kernel"] / (24 * 7.68e6) < 1.05
    assert 1.0 <= t["decode_attn_kernel_96_rows"] / (96 * 7.68e6) < 1.05
    json.dumps(t)


def test_dump_outputs_writes_the_rows_as_float_arrays(tmp_path):
    """--dump-outputs: one row of token ids per window of the last timed step, -1 after its end, plus the row lengths;
    a run that cannot happen (no GPU) writes nothing."""
    import numpy as np
    r = _run(["--steps", "1", "--no-extras", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / "none")])
    assert r.returncode != 0 and not (tmp_path / "none").exists()
    sys.path.insert(0, ROOT)
    import bench
    rows = [[50258, 50259, 50360, 50365, 51865, 50414], [50258, 50259, 50360]]
    bench.dump_outputs(str(tmp_path / "out"), rows)
    ids, counts = np.load(tmp_path / "out" / "token_ids.npy"), np.load(tmp_path / "out" / "token_counts.npy")
    assert ids.dtype == counts.dtype == np.float32 and ids.shape == (2, 6) and counts.tolist() == [6, 3]
    assert [row[:int(n)].astype(np.int64).tolist() for row, n in zip(ids, counts)] == rows
    assert (ids[1, 3:] == -1).all()
