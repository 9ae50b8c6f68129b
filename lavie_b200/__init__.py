"""lavie_b200: B200-native (sm_100a) implementation of LaVie's per-step denoisers and the encoders around them.

Public surface = the reference's module APIs for this path:

    from lavie_b200 import UNet3DConditionModel            # base T2V and (INTERP_CONFIG) frame-interpolation denoiser
    unet = UNet3DConditionModel().to("cuda"); unet.load_state_dict(torch.load("lavie_base.pt"))
    noise = unet(latents, t, encoder_hidden_states=prompt_embeds).sample

    from lavie_b200 import UNet3DVSRModel                   # x4 video super-resolution denoiser
    from lavie_b200 import CLIPTextEncoder, VAEDecoder      # text_encoder(ids)[0], vae.decode(z).sample
    from lavie_b200 import VAEEncoder                       # vae.encode(x).latent_dist, vae.encode_video(frames)
    from lavie_b200 import VSRSampler                       # the VSR stage: VSRSampler(vsr_unet).upscale(frames, text, vae_x4)
"""
from .clip import CLIPTextConfig, CLIPTextEncoder  # noqa: F401
from .config import BASE_CONFIG, INTERP_CONFIG, VSR_CONFIG, UNetConfig, param_spec  # noqa: F401
from .pipeline import VSRSampler  # noqa: F401
from .unet import UNet3DConditionModel, UNet3DConditionOutput  # noqa: F401
from .vae import VAEDecoder, VAEEncoder  # noqa: F401
from .vsr import UNet3DVSRModel  # noqa: F401

__all__ = ["UNet3DConditionModel", "UNet3DConditionOutput", "UNet3DVSRModel", "VSRSampler", "CLIPTextEncoder", "CLIPTextConfig",
           "VAEDecoder", "VAEEncoder", "UNetConfig", "BASE_CONFIG", "INTERP_CONFIG", "VSR_CONFIG", "param_spec"]
