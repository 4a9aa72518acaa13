"""TEST INFRASTRUCTURE ONLY — golden vectors for images above 256 patch tokens (tests/golden/tiny_rect.*, small512.*),
produced by the REAL reference (imported from /root/reference, see oracle/ref_harness.py) on seeded weights/inputs
(oracle/seeded.py).  Run in the dev container:

    python -m oracle.make_golden_hires [name ...]

Same content as oracle/make_golden.py (reference outputs in fp32 and under torch.autocast("cpu", bfloat16), the
state-dict spec, the reference's own 1e-6-perturbation sensitivity) for non-square sizes, recorded as `image_hw`.  To
keep the files small the reconstructed images are stored on every RECON_STRIDE-th row and column only (`recon_stride`
in the JSON); the sensitivity of `recon` is measured on the same subsample."""
from __future__ import annotations

import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_harness as rh  # noqa: E402
from oracle.seeded import seeded_images, seeded_state_dict  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
RECON_STRIDE = 4

TINY = dict(vision_embed_dim=128, vision_depth=2, vision_num_heads=2, text_embed_dim=128, text_num_heads=2, text_depth=2,
            decoder_embed_dim=128, decoder_num_heads=2, decoder_depth=2, text_vocab_size=1000)
SMALL = dict(vision_embed_dim=384, vision_depth=12, vision_num_heads=6, text_embed_dim=384, text_num_heads=6,
             text_depth=12, decoder_embed_dim=384, decoder_num_heads=6, decoder_depth=12, text_vocab_size=2048)
CONFIGS = {
    # name: (VTPConfig kwargs, B, (height, width), store patch tokens)
    # 272x400 -> 17x25 = 425 patches: ragged (not a multiple of 8 or 128), non-square, T = 426 in the trunk
    "tiny_rect": (TINY, 2, (272, 400), True),
    # VTP-Small at 512x512 -> 32x32 = 1024 patches, T = 1025
    "small512": (SMALL, 1, (512, 512), False),
}


def main():
    rh.import_reference()
    from vtp.models.vtp_hf import VTPConfig, VTPModel

    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(os.cpu_count())
    only = set(sys.argv[1:])
    s = RECON_STRIDE
    for name, (kw, B, hw, with_patch) in CONFIGS.items():
        if only and name not in only:
            continue
        m = VTPModel(VTPConfig(**kw)).eval()
        spec = {k: list(v.shape) for k, v in m.state_dict().items()}
        m.load_state_dict(seeded_state_dict(spec, seed=0))
        x = seeded_images(B, *hw)
        out = {}
        with torch.no_grad():
            for tag, ctx in (("fp32", torch.autocast("cpu", enabled=False)),
                             ("bf16", torch.autocast("cpu", dtype=torch.bfloat16))):
                with ctx:
                    lat = m.get_reconstruction_latents(x)
                    out[f"latents_{tag}"] = lat.float().numpy()
                    out[f"recon_{tag}"] = m.get_latents_decoded_images(lat)[..., ::s, ::s].float().numpy()
                    out[f"img_feat_{tag}"] = m.get_clip_image_feature(x).float().numpy()
                    feats = m.get_last_layer_feature(x)
                    out[f"cls_{tag}"] = feats["cls_token"].float().numpy()
                    if with_patch and tag == "fp32":  # (the bf16 mode is held to latents / cls / img_feat)
                        out[f"patch_{tag}"] = feats["patch_tokens"].float().numpy()
            xp = x * (1 + 1e-6)
            relf = lambda a, b: float(((a.float() - torch.from_numpy(b)).norm() / torch.from_numpy(b).norm()))
            latp = m.get_reconstruction_latents(xp)
            sens = {"latents": relf(latp, out["latents_fp32"]),
                    "recon": relf(m.get_latents_decoded_images(latp)[..., ::s, ::s], out["recon_fp32"]),
                    "img_feat": relf(m.get_clip_image_feature(xp), out["img_feat_fp32"]),
                    "cls": relf(m.get_last_layer_feature(xp)["cls_token"], out["cls_fp32"])}
        out["x_checksum"] = np.array([x.double().sum().item(), x.double().abs().sum().item()])
        np.savez_compressed(os.path.join(OUT, f"{name}.npz"), **out)
        with open(os.path.join(OUT, f"{name}.json"), "w") as f:
            json.dump({"config": kw, "batch": B, "image_hw": list(hw), "recon_stride": s, "spec": spec,
                       "reference_commit": "5ce1eb6", "torch": torch.__version__, "seed_opts": {},
                       "ref_sensitivity_1e-6": sens}, f)
        print(name, "reference sensitivity to 1e-6 input perturbation:", sens)


if __name__ == "__main__":
    main()
