"""Generate the golden vectors that pin ``oracle/unet3d_oracle.py`` to the reference.

Run ONLY inside the build container (needs /root/reference, read-only):

    python tests/golden/make_golden.py

It imports the UNMODIFIED reference model code from /root/reference/base/models with
stand-ins (tests/golden/shims/) for the two third-party packages the reference does not
vendor (diffusers==0.16.0, rotary_embedding_torch), loads the deterministic synthetic
weights of ``lavie_b200.synthetic`` with ``load_state_dict(strict=True)`` (which also proves
the 830-key table of ``lavie_b200.config.param_spec``), runs the reference forward on CPU in
fp32 and stores inputs, a few intermediate activations (forward hooks) and the output.
Nothing under tests/, bench.py or smoke() reads /root/reference at run time; they read the
.pt files written here.
"""
import hashlib
import os
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(HERE, "shims"))
sys.path.insert(0, "/root/reference/base")

import torch  # noqa: E402

from lavie_b200.config import BASE_CONFIG  # noqa: E402
from lavie_b200.synthetic import synthetic_inputs, synthetic_state_dict  # noqa: E402
from models.unet import UNet3DConditionModel  # noqa: E402  (the reference)

CASES = {
    # name: (batch, frames, height, width, timestep)
    "b2_f16_8x8": (2, 16, 8, 8, 500),
    "b1_f3_16x24": (1, 3, 16, 24, 37),
}
TAPS = {
    "conv_in": "conv_in",
    "down0_res0": "down_blocks.0.resnets.0",
    "down0_attn0": "down_blocks.0.attentions.0",
    "mid": "mid_block",
}
# kept under 1 MB: taps at every 16th channel instead of every 8th, the text embedding as the digest of its bytes
# (tests/conftest.py:load_golden draws it again from the inputs seed)
LEAN = {"b2_f16_8x8"}


def main():
    torch.manual_seed(0)
    torch.set_num_threads(os.cpu_count())
    ref = UNet3DConditionModel.from_config(BASE_CONFIG.to_dict()).eval()
    sd = synthetic_state_dict(seed=0)
    ref.load_state_dict(sd, strict=True)
    mods = dict(ref.named_modules())
    for name, (b, f, h, w, t) in CASES.items():
        sample, _, text = synthetic_inputs(b, f, h, w, seed=1)
        stride = 16 if name in LEAN else 8
        got = {}
        hooks = []
        for tap, modname in TAPS.items():
            def hook(_m, _i, out, tap=tap):
                out = out.sample if hasattr(out, "sample") else out
                got[tap] = out.detach()[:, ::stride].contiguous().clone()   # a channel subset keeps the fixture small
            hooks.append(mods[modname].register_forward_hook(hook))
        t0 = time.time()
        with torch.no_grad():
            out = ref(sample, t, encoder_hidden_states=text).sample
        dt = time.time() - t0
        for hk in hooks:
            hk.remove()
        blob = {"sample": sample, "timestep": t, "text": text, "out": out, "taps": got,
                "weights_seed": 0, "inputs_seed": 1, "shape": (b, f, h, w)}
        if name in LEAN:
            blob["text_sha256"] = hashlib.sha256(blob.pop("text").numpy().tobytes()).hexdigest()
        torch.save(blob, os.path.join(HERE, f"{name}.pt"))
        print(f"{name}: out std {out.std():.4f} in {dt:.1f}s -> {name}.pt")
    # one timestep passed as a [B] tensor with different values per batch item
    b, f, h, w, _ = CASES["b2_f16_8x8"]
    sample, _, text = synthetic_inputs(b, 2, h, w, seed=2)
    tt = torch.tensor([981, 1])
    with torch.no_grad():
        out = ref(sample, tt, encoder_hidden_states=text).sample
    torch.save({"sample": sample, "timestep": tt, "text": text, "out": out, "taps": {},
                "weights_seed": 0, "inputs_seed": 2, "shape": (b, 2, h, w)},
               os.path.join(HERE, "b2_f2_8x8_tvec.pt"))
    print("b2_f2_8x8_tvec done")


if __name__ == "__main__":
    main()
