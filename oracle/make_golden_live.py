"""TEST INFRASTRUCTURE ONLY — records what the tests once compared against the reference live, so that they run
without a reference checkout (see oracle/ref_harness.py for where it is imported from):

    python -m oracle.make_golden_live

Writes tests/golden/live_ref.json + live_ref.npz:
  * tiny_latents_fp32: `VTPModel.get_reconstruction_latents` of the reference on the "tiny" golden inputs;
  * cosine: `CosineScheduler(**kw)[i]` for i in 0 .. total_iters + 2, per case of CASES;
  * drop_single / drop_ranks: (batch, ratio, kept rows, residual scale) from `get_branges_scales`, in one process
    and on each of 2 gloo ranks (the reference allocates on rank 0 and broadcasts)."""
from __future__ import annotations

import json
import os
import socket
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_harness as rh  # noqa: E402
from tests.util import golden_inputs, load_golden  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")

COSINE_CASES = [dict(base_value=1e-3, final_value=1e-6, total_iters=50, warmup_iters=5, start_warmup_value=1e-7, freeze_iters=0),
                dict(base_value=0.994, final_value=1.0, total_iters=20),
                dict(base_value=0.04, final_value=0.2, total_iters=12, warmup_iters=3, start_warmup_value=0.0, freeze_iters=2)]
DROP_SINGLE = [(8, 0.3), (5, 0.5), (3, 0.9), (256, 0.25), (1, 0.5)]
DROP_RANKS = [(8, 0.3), (5, 0.5), (3, 0.9), (16, 0.1)]


def _branges(blk, cases):
    out = []
    for b, ratio in cases:
        br, scale = blk.get_branges_scales(torch.zeros(b, 2, 4), ratio)
        out.append([b, ratio, int(br.numel()), float(scale)])
    return out


def _drop_worker(rank, world, port, out):
    import torch.distributed as dist

    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    rh.import_reference()
    import vtp.models.layers.block as blk

    out[rank] = _branges(blk, DROP_RANKS)
    dist.destroy_process_group()


def main():
    import torch.multiprocessing as mp

    rh.import_reference()
    import vtp.models.layers.block as blk
    from vtp.models.utils.text_utils import CosineScheduler
    from vtp.models.vtp_hf import VTPConfig, VTPModel

    meta, g = load_golden("tiny")
    sd, x, _ = golden_inputs(meta)
    m = VTPModel(VTPConfig(**meta["config"])).eval()
    m.load_state_dict(sd)
    with torch.no_grad():
        lat = m.get_reconstruction_latents(x)
    cosine = []
    for kw in COSINE_CASES:
        s = CosineScheduler(**kw)
        cosine.append([float(s[i]) for i in range(kw["total_iters"] + 3)])
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    out = mp.Manager().dict()
    mp.spawn(_drop_worker, args=(2, port, out), nprocs=2, join=True)
    rec = {"cosine_cases": COSINE_CASES, "cosine": cosine, "drop_single": _branges(blk, DROP_SINGLE),
           "drop_ranks": [out[0], out[1]]}
    with open(os.path.join(OUT, "live_ref.json"), "w") as f:
        json.dump(rec, f, indent=1)
    np.savez_compressed(os.path.join(OUT, "live_ref.npz"), tiny_latents_fp32=lat.numpy())
    print("live_ref: latents vs tiny golden", float((lat - g["latents_fp32"]).norm() / g["latents_fp32"].norm()))


if __name__ == "__main__":
    main()
