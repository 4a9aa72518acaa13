"""bench.py contract, the part that runs without a GPU: the reference arm (CPU restatement of the step, oracle port)
prints ONE JSON line with the keys the driver reads, on the same config object as our arm."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    env = dict(os.environ, VTP_CPU_THREADS="4")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--cpu-batch", "1", "--gpus", "1"], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"].startswith("images/sec") and d["unit"] == "images/sec"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["value"] > 0 and d["vs_baseline"] is None
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] == 4 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # same workload description as our arm (bench.workload_config), plus the bounded sample
    sys.path.insert(0, ROOT)
    import argparse

    import bench

    args = argparse.Namespace(batch=256, model="small", prototypes=65536, no_lpips=False)
    ours = bench.workload_config(args, 1, d["config"]["flops_per_image"])
    assert {k: d["config"][k] for k in ours} == ours and "sample" in d["config"]


def test_dump_sample_follows_parameters_not_store_layout():
    """`bench.py --dump-outputs` samples the same parameter elements whatever order and padding the flat parameter store
    gives them, so that two builds can be compared output for output."""
    import torch

    sys.path.insert(0, ROOT)
    import bench
    from vtp_b200.train import ParamStore

    def store(specs):
        st = ParamStore("cpu")
        for name, shape in specs:
            st.add(name, shape)
        st.finalize()
        for name in st.offset:
            v = st.f32(name)
            v.copy_(torch.arange(v.numel()).view_as(v) + 1000.0 * ord(name))
        return st

    specs = [("a", (3, 5)), ("b", (7,)), ("c", (4, 4))]
    s1, s2 = store(specs), store(specs[::-1])
    assert s1.offset != s2.offset
    i1, i2 = (bench._canonical_sample(s, s.offset, 500) for s in (s1, s2))
    assert torch.equal(s1.p[i1], s2.p[i2])
    assert (s1.p[i1] >= 1000.0 * ord("a")).all()                  # never the zero padding between parameters
    assert set(s1.p[i1].div(1000, rounding_mode="floor").long().tolist()) == {ord("a"), ord("b"), ord("c")}
