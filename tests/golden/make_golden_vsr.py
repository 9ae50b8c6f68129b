"""Generate the golden vectors that pin ``oracle/vsr_oracle.py`` (SURVEY 8f row N2) to the reference.

Run ONLY inside the build container (needs /root/reference, read-only):

    python tests/golden/make_golden_vsr.py

Imports the UNMODIFIED ``UNet3DVSRModel`` from /root/reference/vsr/models with the stand-ins of tests/golden/shims/,
builds it from the reference's own vsr/configs/unet_3d_config.json, loads the deterministic synthetic weights with
``load_state_dict(strict=True)`` (which proves the 1158-key table of ``lavie_b200.config.param_spec(VSR_CONFIG)``), runs
the forward on CPU in fp32 and stores inputs, output and two intermediate taps (forward hooks on the reference modules).
"""
import hashlib
import json
import os
import sys
import time
import zlib

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(HERE, "shims"))
sys.path.insert(0, "/root/reference/vsr")

import torch  # noqa: E402

from lavie_b200.config import VSR_CONFIG, param_spec  # noqa: E402
from lavie_b200.synthetic import synthetic_state_dict  # noqa: E402
from models.unet import UNet3DVSRModel  # noqa: E402  (the reference's VSR UNet)

CASES = {
    # name: (batch, frames, height, width, timestep, text tokens, noise levels)
    "vsr_b2_f4_16x16": (2, 4, 16, 16, 500, 77, (20, 50)),
    "vsr_b1_f3_24x8": (1, 3, 24, 8, 37, 20, (250,)),
}
# kept under 1 MB: the text embedding as the digest of its bytes (tests/conftest.py:load_golden draws it again)
LEAN = {"vsr_b2_f4_16x16"}


def main():
    torch.set_num_threads(os.cpu_count())
    cfg = json.load(open("/root/reference/vsr/configs/unet_3d_config.json"))
    ref = UNet3DVSRModel.from_config(cfg).eval()
    sd = synthetic_state_dict(VSR_CONFIG, seed=0)
    assert set(ref.state_dict().keys()) == set(param_spec(VSR_CONFIG).keys())
    ref.load_state_dict(sd, strict=True)
    taps = {}
    ref.down_temporal_blocks[0].register_forward_hook(lambda m, i, o: taps.__setitem__("down0", o.detach().clone()))
    ref.mid_temporal_block.register_forward_hook(lambda m, i, o: taps.__setitem__("mid", o.detach().clone()))
    for name, (b, f, h, w, t, ntok, levels) in CASES.items():
        g = torch.Generator().manual_seed(zlib.crc32(name.encode()))
        sample = torch.randn(b, 4, f, h, w, generator=g)
        low_res = torch.randn(b, 3, f, h, w, generator=g)
        text = torch.randn(b, ntok, 1024, generator=g)
        labels = torch.tensor(levels, dtype=torch.long)
        t0 = time.time()
        with torch.no_grad():
            out = ref(sample, t, low_res, encoder_hidden_states=text, class_labels=labels).sample
        blob = {"sample": sample, "low_res": low_res, "timestep": t, "text": text, "class_labels": labels, "out": out,
                "down0": taps["down0"], "mid": taps["mid"], "weights_seed": 0, "shape": (b, f, h, w)}
        if name in LEAN:
            blob["text_shape"] = tuple(text.shape)
            blob["text_sha256"] = hashlib.sha256(blob.pop("text").numpy().tobytes()).hexdigest()
        torch.save(blob, os.path.join(HERE, f"{name}.pt"))
        print(f"{name}: out {tuple(out.shape)} std {out.std():.4f} in {time.time() - t0:.1f}s")


if __name__ == "__main__":
    main()
