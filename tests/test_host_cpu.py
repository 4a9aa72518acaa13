"""CPU: host-side logic — state-dict/ABI compatibility with the reference, config defaults, packing layouts."""
import ctypes
import os
import re

import pytest
import torch

from tests.util import load_golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_abi_exports_every_declared_symbol():
    from vtp_b200 import lib

    hdr = open(os.path.join(ROOT, "include", "vtp_b200.h")).read()
    declared = set(re.findall(r"\b(vtp_[a-z0-9_]+)\s*\(", hdr))
    declared -= {"vtp_stream_t"}
    assert declared, "no declarations parsed"
    assert os.path.exists(lib.LIB_PATH), "libvtp_b200.so missing: run python -m vtp_b200.build"
    so = ctypes.CDLL(lib.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(so, name), f"{name} declared in include/vtp_b200.h but not exported"
    assert declared == set(lib.SIGNATURES), declared ^ set(lib.SIGNATURES)
    assert lib.load().vtp_version() >= 100


@pytest.mark.parametrize("name", ["tiny", "small"])
def test_state_dict_keys_match_reference(name):
    from vtp_b200.config import VTPConfig
    from vtp_b200.model import VTPModel

    meta, _ = load_golden(name)
    m = VTPModel(VTPConfig(**meta["config"]))
    mine = {k: list(v.shape) for k, v in m.state_dict().items()}
    assert mine == meta["spec"]  # spec was dumped from the real reference's state_dict()


def test_config_defaults_match_reference():
    from vtp_b200.config import VTPConfig

    c = VTPConfig()
    assert (c.vision_embed_dim, c.vision_depth, c.vision_num_heads) == (768, 12, 12)
    assert (c.vision_norm_layer, c.vision_ffn_layer, c.decoder_norm_layer) == ("rmsnorm", "swiglu", "layernorm")
    assert c.vision_feature_bottleneck == 64 and c.vision_bottleneck_ae_only and c.vision_clip_feat == "cls"
    assert c.text_context_length == 77 and c.text_vocab_size == 49408 and c.model_type == "vtp"


def test_cpu_call_fails_loudly():
    from vtp_b200 import lib
    from vtp_b200.config import preset
    from vtp_b200.model import VTPModel

    m = VTPModel(preset("tiny"))
    with pytest.raises(lib.VtpError):
        m.get_reconstruction_latents(torch.zeros(1, 3, 64, 64))


def test_save_load_roundtrip(tmp_path):
    from vtp_b200.config import preset
    from vtp_b200.model import VTPModel

    m = VTPModel(preset("tiny"))
    m.save_pretrained(str(tmp_path))
    m2 = VTPModel.from_pretrained(str(tmp_path))
    for (k, a), (_, b) in zip(m.state_dict().items(), m2.state_dict().items()):
        assert torch.equal(a, b), k


def test_interleave8_layout():
    from vtp_b200.engine import interleave8

    w1 = torch.arange(32).float().view(16, 2)
    w2 = -w1
    p = interleave8(w1, w2)
    assert torch.equal(p[:8], w1[:8]) and torch.equal(p[8:16], w2[:8]) and torch.equal(p[16:24], w1[8:])


def test_rope_table_matches_oracle():
    from oracle import vtp_oracle as vo
    from vtp_b200.rope import rope_periods, rope_sincos

    per = rope_periods(64)
    assert torch.equal(per, vo.rope_periods(64))
    s, c = rope_sincos(16, 16, per)
    so, co = vo.rope_table(16, 16, per)
    assert torch.equal(s, so) and torch.equal(c, co) and s.dtype == torch.bfloat16


def test_compat_shim_serves_reference_import_path():
    """`from vtp.models.vtp_hf import VTPModel` (tools/test_reconstruction_hf.py:37) resolves to this implementation when
    <repo>/compat is first on the path; the rest of the `vtp` namespace is left to the reference checkout."""
    import subprocess
    import sys
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r); "
            "from vtp.models.vtp_hf import VTPModel, VTPConfig, VTPPreTrainedModel; "
            "import vtp_b200.model as m; assert VTPModel is m.VTPModel and issubclass(VTPModel, VTPPreTrainedModel); "
            "c = VTPConfig(); assert c.model_type == 'vtp'; print('ok')") % (ROOT, os.path.join(ROOT, "compat"))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr[-2000:]


def test_center_crop_matches_adm_definition():
    """vtp_b200/image_utils.py vs the ADM procedure written out with numpy slicing (vtp/utils/image_utils.py:5-31)."""
    import numpy as np
    from PIL import Image

    from vtp_b200.image_utils import center_crop_arr

    rng = np.random.default_rng(0)
    for (w, h), size in (((700, 520), 256), ((300, 260), 256), ((1030, 2051), 224), ((256, 256), 256)):
        im = Image.fromarray(rng.integers(0, 256, (h, w, 3), dtype=np.uint8))
        ref = im
        while min(*ref.size) >= 2 * size:
            ref = ref.resize(tuple(x // 2 for x in ref.size), resample=Image.BOX)
        sc = size / min(*ref.size)
        ref = ref.resize(tuple(round(x * sc) for x in ref.size), resample=Image.BICUBIC)
        a = np.array(ref)
        cy, cx = (a.shape[0] - size) // 2, (a.shape[1] - size) // 2
        out = np.array(center_crop_arr(im, size))
        assert out.shape == (size, size, 3) and np.array_equal(out, a[cy:cy + size, cx:cx + size])


def test_tokenizer_normalisation_constants():
    from vtp_b200.generation import VTP_Tokenizer

    t = VTP_Tokenizer.__new__(VTP_Tokenizer)
    t._setup_normalization("imagenet")
    assert t.norm_mean == [0.485, 0.456, 0.406] and t.norm_std == [0.229, 0.224, 0.225]
    assert abs(t.inv_mean[0] + 0.485 / 0.229) < 1e-12 and abs(t.inv_std[2] - 1 / 0.225) < 1e-12
    t._setup_normalization("half")
    assert t.inv_mean == [-1.0, -1.0, -1.0] and t.inv_std == [2.0, 2.0, 2.0]
    import pytest
    with pytest.raises(ValueError):
        t._setup_normalization("other")


def test_cosine_schedule_matches_reference_table():
    """vtp_b200.schedules.CosineSchedule restates the reference's CosineScheduler (models/utils/text_utils.py:160-207):
    against values recorded from it: a few points per case (fixture below), and every iteration (live_ref.json)."""
    import numpy as np

    from vtp_b200.schedules import CosineSchedule

    cases = [dict(base_value=1e-3, final_value=1e-6, total_iters=50, warmup_iters=5, start_warmup_value=1e-7, freeze_iters=0),
             dict(base_value=0.994, final_value=1.0, total_iters=20),
             dict(base_value=0.04, final_value=0.2, total_iters=12, warmup_iters=3, start_warmup_value=0.0, freeze_iters=2)]
    # recorded from the reference's CosineScheduler (commit 5ce1eb6): [it 0, 1, 4, 7, total-1, total, total+5] per case
    recorded = [[1e-07, 0.000250075, 0.001, 0.0009951389003364144, 2.2167568952178134e-06, 1e-06, 1e-06],
                [0.994, 0.9940369349782145, 0.9945729490168752, 0.9956380285007813, 0.9999630650217854, 1.0, 1.0],
                [0.0, 0.0, 0.04, 0.07012081585130131, 0.19207750943219354, 0.2, 0.2]]
    for kw, rec in zip(cases, recorded):
        s = CosineSchedule(**kw)
        T = kw["total_iters"]
        got = [s[i] for i in (0, 1, 4, 7, T - 1, T, T + 5)]
        assert np.allclose(got, rec, rtol=1e-12, atol=0), (kw, got, rec)
        assert s.table().dtype == np.float32 and s.table().size == T + 1 and s.table()[-1] == np.float32(kw["final_value"])
    meta, _ = load_golden("live_ref")
    assert meta["cosine_cases"] == cases
    for kw, ref in zip(cases, meta["cosine"]):
        s = CosineSchedule(**kw)
        assert [s[i] for i in range(kw["total_iters"] + 3)] == ref, kw


def test_from_pretrained_sharded_and_strict_arguments(tmp_path):
    """HF sharded layout (model.safetensors.index.json) loads; unsupported from_pretrained arguments raise instead of being
    dropped silently; torch_dtype converts the parameters but keeps the bf16 RoPE periods buffer."""
    import json

    import pytest
    from safetensors.torch import save_file

    from vtp_b200 import VTPConfig, VTPModel

    cfg = VTPConfig(vision_embed_dim=128, vision_depth=1, vision_num_heads=2, text_embed_dim=128, text_num_heads=2, text_depth=1,
                    decoder_embed_dim=128, decoder_num_heads=2, decoder_depth=1, text_vocab_size=64)
    m = VTPModel(cfg)
    m.save_pretrained(str(tmp_path))
    sd = {k: v.detach().clone().contiguous() for k, v in m.state_dict().items()}
    keys = sorted(sd)
    a, b = keys[: len(keys) // 2], keys[len(keys) // 2:]
    os.remove(os.path.join(tmp_path, "model.safetensors"))
    save_file({k: sd[k] for k in a}, os.path.join(tmp_path, "model-00001-of-00002.safetensors"))
    save_file({k: sd[k] for k in b}, os.path.join(tmp_path, "model-00002-of-00002.safetensors"))
    with open(os.path.join(tmp_path, "model.safetensors.index.json"), "w") as f:
        json.dump({"weight_map": {**{k: "model-00001-of-00002.safetensors" for k in a},
                                  **{k: "model-00002-of-00002.safetensors" for k in b}}}, f)
    m2 = VTPModel.from_pretrained(str(tmp_path))
    assert all(torch.equal(v, m2.state_dict()[k]) for k, v in sd.items())
    m3 = VTPModel.from_pretrained(str(tmp_path), torch_dtype=torch.bfloat16)
    assert m3.trunk.cls_token.dtype == torch.bfloat16 and m3.trunk.rope_embed.periods.dtype == torch.bfloat16
    with pytest.raises(TypeError):
        VTPModel.from_pretrained(str(tmp_path), low_cpu_mem_usage=True)
    with pytest.raises(NotImplementedError):
        VTPModel.from_pretrained(str(tmp_path), device_map="auto")
    with pytest.raises(FileNotFoundError):
        VTPModel.from_pretrained("MiniMaxAI/VTP-Large-f16d64")


def test_crop_box_sampling_follows_torchvision_get_params():
    """vtp_b200.data.random_resized_crop_boxes restates torchvision RandomResizedCrop.get_params (area scale x log-uniform
    aspect ratio, 10 tries, centre-crop fallback): boxes inside the image, areas / ratios inside the requested ranges, and
    the same distribution as torchvision's own sampler (mean area / mean log-ratio within sampling error)."""
    import math

    import numpy as np
    from torchvision.transforms import RandomResizedCrop

    from vtp_b200.data import random_resized_crop_boxes

    H, W = 300, 400
    rng = np.random.default_rng(0)
    for scale in ((0.32, 1.0), (0.05, 0.32), (0.9, 1.0)):
        b = random_resized_crop_boxes(rng, 6000, H, W, scale)
        assert (b[:, 0] >= 0).all() and (b[:, 1] >= 0).all() and (b[:, 0] + b[:, 2] <= W).all() and (b[:, 1] + b[:, 3] <= H).all()
        area = b[:, 2] * b[:, 3] / (H * W)
        assert area.min() >= scale[0] * 0.95 and area.max() <= min(1.0, scale[1] * 1.02)
        torch.manual_seed(0)
        img = torch.zeros(3, H, W)
        tv = np.array([RandomResizedCrop.get_params(img, list(scale), [3 / 4, 4 / 3]) for _ in range(3000)], dtype=np.float64)  # i, j, h, w
        tv_area = tv[:, 2] * tv[:, 3] / (H * W)
        tv_lr = np.log(tv[:, 3] / tv[:, 2])
        lr = np.log(b[:, 2] / b[:, 3])
        assert abs(area.mean() - tv_area.mean()) < 0.02 and abs(lr.mean() - tv_lr.mean()) < 0.02
        assert abs(lr.std() - tv_lr.std()) < 0.02
    # an image so elongated that no ratio in [3/4, 4/3] fits at this scale: centre-crop fallback, clipped to the ratio range
    fb = random_resized_crop_boxes(np.random.default_rng(1), 10, 100, 1000, (0.9, 1.0))
    assert (fb[:, 3] == 100).all() and (np.abs(fb[:, 2] / fb[:, 3] - 4 / 3) < 0.02).all()


def test_tokenizer_img_transform_matches_torchvision_pipeline():
    """`VTP_Tokenizer.img_transform` (one callable) == the torchvision pipeline the reference composes
    (generation/tokenizer/vtp_tokenizer.py:75-82): same crop, same flips under the same seed, same normalisation."""
    np = pytest.importorskip("numpy")
    tvt = pytest.importorskip("torchvision.transforms")
    from PIL import Image

    from vtp_b200.generation import VTP_Tokenizer
    from vtp_b200.image_utils import center_crop_arr

    tok = VTP_Tokenizer.__new__(VTP_Tokenizer)   # no model / GPU needed for the host-side transform
    tok.img_size = 64
    for kind in ("imagenet", "half"):
        tok._setup_normalization(kind)
        assert tok.inv_mean == [-m / s for m, s in zip(tok.norm_mean, tok.norm_std)]
        ref = tvt.Compose([tvt.Lambda(lambda im: center_crop_arr(im, 64)), tvt.RandomHorizontalFlip(p=0.5), tvt.ToTensor(),
                           tvt.Normalize(mean=tok.norm_mean, std=tok.norm_std, inplace=True)])
        ours = tok.img_transform(0.5)
        rng = np.random.RandomState(0)
        for i in range(6):
            img = Image.fromarray((rng.rand(90 + 7 * i, 140 - 5 * i, 3) * 255).astype("uint8"))
            torch.manual_seed(i)
            a = ours(img)
            torch.manual_seed(i)
            b = ref(img)
            assert torch.equal(a, b)
    with pytest.raises(ValueError):
        tok._setup_normalization("other")


def test_every_env_switch_is_documented():
    """Every `VTP_*` environment variable the library, bench.py or the entry points read is listed in INTEGRATION.md §4."""
    import re

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    pat = re.compile(r'getenv\("(VTP_[A-Z0-9_]+)"\)|environ(?:\.get)?[\(\[]\s*"(VTP_[A-Z0-9_]+)"')
    names = set()
    srcs = [os.path.join(root, "bench.py"), os.path.join(root, "__graft_entry__.py")]
    for d, _, files in os.walk(os.path.join(root, "vtp_b200")):
        srcs += [os.path.join(d, f) for f in files if f.endswith((".cu", ".cuh", ".h", ".py"))]
    for path in srcs:
        for m in pat.finditer(open(path, encoding="utf-8", errors="ignore").read()):
            names.add(m.group(1) or m.group(2))
    assert len(names) > 20
    doc = open(os.path.join(root, "INTEGRATION.md"), encoding="utf-8").read()
    missing = sorted(n for n in names if n not in doc)
    assert not missing, missing
