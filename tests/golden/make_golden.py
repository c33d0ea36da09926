"""Generates tests/golden/* by running the reference's OWN Python files (an unchanged teticio/audio-diffusion checkout,
imported through the audio_diffusion_b200/compat shim) on the CPU.  Run from the repo root:

    python tests/golden/make_golden.py /path/to/audio-diffusion

 * vae_key_map.json — output of audiodiffusion/utils.py::convert_ldm_vae_checkpoint on an ldm-format checkpoint of the
   config/ldm_autoencoder_kl.yaml shape: [hf key, shape] in the order the reference writes them.  Pins the parameter
   table of libb200ad's AutoencoderKL (b200ad_vae_param_name / _shape).
 * vae_ldm_to_hf.json — the same converter's key mapping: [ldm key, hf key, hf shape] for every tensor it writes (the
   attention projections go from 1x1 conv to linear shape), read off by feeding it tensors tagged with their index.
 * reference_pipeline_cpu.npz — the uint8 images of the reference AudioDiffusionPipeline.__call__ driving the CPU oracle
   U-Net of tests/test_cpu_dropin.py with the product's schedulers: unconditional (`shim_<ddpm|ddim>`) and the
   audio-conditioned / in-painting path (`cond_<ddpm|ddim>`); plus its DDIM inversion (`encode_ddim`) and `slerp`.
 * mel_host_logic.json — audiodiffusion/mel.py's slicing / padding bookkeeping on seeded audio: sizes, dtype and
   SHA-256 of the padded audio and of its slices.
 * pipeline_ddpm_small.npz — audiodiffusion/pipeline_audio_diffusion.py::AudioDiffusionPipeline.__call__ (the reference
   file, on the import shim) driving the fp32 CPU oracle U-Net (seeded synthetic weights, oracle/unet_oracle.py) and the
   ORACLE's DDPM scheduler (oracle/schedulers_oracle.py - nothing of the product computes a number in this fixture; the
   product's own scheduler gives bit-identical images, which the generator asserts) for 6 steps from a given noise tensor
   with a CPU step generator: the uint8 images it returns.
   The GPU pipeline must reproduce them within the stated tolerance (tests/test_gpu_pipeline.py).
The numerical content is the oracle's (diffusers cannot be imported here); what the fixtures pin is the reference
files' own logic: key mapping, loop order, noise draws, float->uint8 conversion.
"""
import hashlib
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
GOLDEN = os.path.join(ROOT, "tests", "golden")

SMALL = dict(in_channels=1, out_channels=1, layers_per_block=2, block_out_channels=(128, 256),
             down_block_types=("DownBlock2D", "AttnDownBlock2D"), up_block_types=("AttnUpBlock2D", "UpBlock2D"))


def vae_key_map():
    from audiodiffusion.utils import convert_ldm_vae_checkpoint
    from oracle.vae_oracle import VAEConfig, init_weights
    from test_cpu_dropin import _hf_to_ldm_vae
    w = init_weights(VAEConfig(), seed=0)
    conv = convert_ldm_vae_checkpoint(_hf_to_ldm_vae(w), None)
    out = [[k, list(v.shape)] for k, v in conv.items()]
    with open(os.path.join(ROOT, "tests", "golden", "vae_key_map.json"), "w") as f:
        json.dump({"source": "audiodiffusion/utils.py:156-291 convert_ldm_vae_checkpoint", "keys": out}, f, indent=0)
    print("vae_key_map.json", len(out))


def pipeline_small():
    from audiodiffusion.pipeline_audio_diffusion import AudioDiffusionPipeline as RefPipe
    from diffusers import DDPMScheduler as ProductDDPM      # the import shim = the product's scheduler (cross-check only)
    from oracle.schedulers_oracle import OracleDDPM
    from oracle.unet_oracle import UNetConfig, init_weights, unet_forward

    class OracleUNet:
        def __init__(self):
            self.cfg = UNetConfig(sample_size=(32, 32), **SMALL)
            self.w = init_weights(self.cfg, seed=11)
            self.sample_size = (32, 32)
            self.in_channels = 1

        def __call__(self, x, t):
            return {"sample": unet_forward(self.w, self.cfg, x, t)}

    class FakeMel:
        x_res, y_res, hop_length = 32, 32, 512

        def get_sample_rate(self):
            return 22050

        def image_to_audio(self, image):
            return np.zeros((self.x_res - 1) * self.hop_length, dtype=np.float32)

    noise = torch.randn(2, 1, 32, 32, generator=torch.Generator().manual_seed(42))

    def run(scheduler):
        pipe = RefPipe(vqvae=None, unet=OracleUNet(), mel=FakeMel(), scheduler=scheduler)
        pipe.set_progress_bar_config(disable=True)
        images, _ = pipe(batch_size=2, steps=6, noise=noise.clone(), step_generator=torch.Generator().manual_seed(7),
                         return_dict=False)
        return np.stack([np.asarray(im) for im in images]).astype(np.uint8)
    arr = run(OracleDDPM())
    assert np.array_equal(arr, run(ProductDDPM())), "the product's DDPMScheduler disagrees with the oracle's"

    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "pipeline_ddpm_small.npz"), noise=noise.numpy(), images=arr,
                        steps=6, weight_seed=11, step_seed=7)
    print("pipeline_ddpm_small.npz", arr.shape, arr.mean())


def vae_ldm_to_hf():
    from audiodiffusion.utils import convert_ldm_vae_checkpoint
    from oracle.vae_oracle import VAEConfig, init_weights
    from test_cpu_dropin import _hf_to_ldm_vae
    ldm = _hf_to_ldm_vae(init_weights(VAEConfig(), seed=3))
    names = list(ldm)
    tagged = {k: torch.full(v.shape, float(i)) for i, (k, v) in enumerate(ldm.items())}
    conv = convert_ldm_vae_checkpoint(tagged, None)
    out = [[names[int(v.flatten()[0])], k, list(v.shape)] for k, v in conv.items()]
    with open(os.path.join(GOLDEN, "vae_ldm_to_hf.json"), "w") as f:
        json.dump({"source": "audiodiffusion/utils.py:156-291 convert_ldm_vae_checkpoint", "map": out}, f, indent=0)
    print("vae_ldm_to_hf.json", len(out))


def reference_pipeline_cpu():
    from PIL import Image

    from audiodiffusion.pipeline_audio_diffusion import AudioDiffusionPipeline as RefPipe
    from diffusers import DDIMScheduler, DDPMScheduler
    from test_cpu_dropin import FakeMel, OracleUNet, ScriptedMel, cond_call

    def u8(images):
        return np.stack([np.asarray(im) for im in images]).astype(np.uint8)
    out = {}
    for sched, cls in (("ddpm", DDPMScheduler), ("ddim", DDIMScheduler)):
        pipe = RefPipe(vqvae=None, unet=OracleUNet(), mel=FakeMel(), scheduler=cls())
        pipe.set_progress_bar_config(disable=True)
        out[f"shim_{sched}"] = u8(pipe(batch_size=2, steps=4, generator=torch.Generator().manual_seed(42)).images)
        pipe = RefPipe(vqvae=None, unet=OracleUNet(), mel=ScriptedMel(), scheduler=cls())
        pipe.set_progress_bar_config(disable=True)
        images, _ = pipe(**cond_call(sched))
        out[f"cond_{sched}"] = u8(images)
    rng = np.random.default_rng(9)
    pil = [Image.fromarray(rng.integers(0, 256, (16, 16), dtype=np.uint8)) for _ in range(2)]
    pipe = RefPipe(vqvae=None, unet=OracleUNet(), mel=ScriptedMel(), scheduler=DDIMScheduler())
    pipe.set_progress_bar_config(disable=True)
    out["encode_ddim"] = pipe.encode(pil, steps=5).numpy()
    a = torch.randn(4, 4, generator=torch.Generator().manual_seed(1))
    b = torch.randn(4, 4, generator=torch.Generator().manual_seed(2))
    out["slerp"] = RefPipe.slerp(a, b, 0.3).numpy()
    np.savez_compressed(os.path.join(GOLDEN, "reference_pipeline_cpu.npz"), **out)
    print("reference_pipeline_cpu.npz", {k: v.shape for k, v in out.items()})


def mel_host_logic():
    from audiodiffusion.mel import Mel as RefMel
    from test_cpu_dropin import MEL_CASES
    rng = np.random.default_rng(0)
    cases = []
    for (x_res, y_res, hop) in MEL_CASES:
        for n in [10, x_res * hop - 1, x_res * hop, 3 * x_res * hop + 17]:
            a = RefMel(x_res=x_res, y_res=y_res, hop_length=hop)
            a.load_audio(raw_audio=rng.standard_normal(n).astype(np.float32))
            slices = hashlib.sha256()
            for s in range(a.get_number_of_slices()):
                slices.update(a.get_audio_slice(s).tobytes())
            cases.append({"x_res": x_res, "y_res": y_res, "hop_length": hop, "n": n, "slice_size": a.slice_size,
                          "n_mels": a.n_mels, "sample_rate": a.get_sample_rate(), "slices": a.get_number_of_slices(),
                          "audio_len": len(a.audio), "audio_dtype": str(a.audio.dtype),
                          "audio_sha256": hashlib.sha256(a.audio.tobytes()).hexdigest(),
                          "slices_sha256": slices.hexdigest()})
        a.set_resolution(32, 16)
        cases[-1]["after_set_resolution_32_16"] = [a.x_res, a.y_res, a.n_mels, a.slice_size]
    with open(os.path.join(GOLDEN, "mel_host_logic.json"), "w") as f:
        json.dump({"source": "audiodiffusion/mel.py:80-133 (Mel.load_audio / get_audio_slice / set_resolution)",
                   "cases": cases}, f, indent=0)
    print("mel_host_logic.json", len(cases))


if __name__ == "__main__":
    if len(sys.argv) != 2 or not os.path.isdir(os.path.join(sys.argv[1], "audiodiffusion")):
        raise SystemExit("usage: python tests/golden/make_golden.py /path/to/audio-diffusion")
    sys.path[:0] = [ROOT, os.path.join(ROOT, "audio_diffusion_b200", "compat"), os.path.abspath(sys.argv[1]),
                    os.path.join(ROOT, "tests")]
    vae_key_map()
    pipeline_small()
    vae_ldm_to_hf()
    reference_pipeline_cpu()
    mel_host_logic()
