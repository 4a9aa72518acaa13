"""Config 5 of BASELINE.json: encode+decode inference throughput sweep (bf16 autocast mode).  GPU only.  (Latents parity
against the reference lives in tests/test_model_gpu.py — tools never touch oracle/.)
  python tools/infer_sweep.py --model large --batches 1,8,64,256 [--graphs] [--image-size 512]
--graphs also times CUDA-graph replays (VTPModel.enable_cuda_graphs) — the small-batch serving path."""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from vtp_b200.config import preset
from vtp_b200.flops import encode_decode_flops
from vtp_b200.model import VTPModel

ap = argparse.ArgumentParser()
ap.add_argument("--model", default="large")
ap.add_argument("--batches", default="1,8,64,256")
ap.add_argument("--graphs", action="store_true")
ap.add_argument("--image-size", type=int, default=256, help="square input size (256: BASELINE config 5)")
a = ap.parse_args()
cfg = preset(a.model)
torch.manual_seed(0)
m = VTPModel(cfg).cuda()
fl = encode_decode_flops(cfg, a.image_size)
out = {"model": a.model, "image_size": a.image_size, "gflop_per_image": fl / 1e9, "rows": []}
for B in [int(b) for b in a.batches.split(",")]:
    x = torch.randn(B, 3, a.image_size, a.image_size, device="cuda")
    with torch.autocast("cuda", dtype=torch.bfloat16):
        for _ in range(3):
            rec = m.get_latents_decoded_images(m.get_reconstruction_latents(x))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 10 if B >= 8 else 30
        torch.cuda.synchronize()
        e0.record()
        for _ in range(reps):
            rec = m.get_latents_decoded_images(m.get_reconstruction_latents(x))
        e1.record()
        torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    row = {"batch": B, "ms": ms, "img_per_s": B / ms * 1e3, "tflops": fl * B / ms / 1e9}
    if a.graphs:
        m.enable_cuda_graphs()
        with torch.autocast("cuda", dtype=torch.bfloat16):
            for _ in range(2):
                rec_g = m.get_latents_decoded_images(m.get_reconstruction_latents(x))
            torch.cuda.synchronize()
            e0.record()
            for _ in range(reps):
                rec_g = m.get_latents_decoded_images(m.get_reconstruction_latents(x))
            e1.record()
            torch.cuda.synchronize()
        m.enable_cuda_graphs(False)
        row["ms_graphs"] = e0.elapsed_time(e1) / reps
        row["graphs_equal_eager"] = bool(torch.equal(rec_g, rec))
    out["rows"].append(row)
    print(f"{a.model} B={B:4d}: {ms:8.2f} ms  {B / ms * 1e3:9.1f} img/s  {fl * B / ms / 1e9:7.1f} TFLOP/s"
          + (f"   graphs: {row['ms_graphs']:8.2f} ms" if a.graphs else ""), flush=True)
print(json.dumps(out))
