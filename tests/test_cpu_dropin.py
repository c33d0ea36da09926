"""CPU tests of the drop-in boundary: the product's pipeline, schedulers, Mel, VAE loader and import shim
(`audio_diffusion_b200/compat`) against what the UNCHANGED reference files compute, and the N>1 path's host logic
(weight broadcast + batch sharding) over gloo with world_size 2.

The reference's results are stored under tests/golden/ (written by tests/golden/make_golden.py, which runs the reference
files on the import shim); these tests need no reference checkout.
"""
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


class OracleUNet:
    """Stand-in with the duck type the reference pipeline needs (callable, sample_size, in_channels), CPU oracle inside."""

    def __init__(self):
        from oracle.unet_oracle import UNetConfig, init_weights
        self.cfg = UNetConfig(sample_size=(16, 16), block_out_channels=(128, 128),
                              down_block_types=("DownBlock2D", "DownBlock2D"), up_block_types=("UpBlock2D", "UpBlock2D"),
                              layers_per_block=1)
        self.w = init_weights(self.cfg, seed=0)
        self.sample_size = 16
        self.in_channels = 1

    def __call__(self, x, t):
        from oracle.unet_oracle import unet_forward
        return {"sample": unet_forward(self.w, self.cfg, x, t)}


class FakeMel:
    x_res, y_res, hop_length = 16, 16, 512

    def get_sample_rate(self):
        return 22050

    def image_to_audio(self, image):
        return np.zeros((self.x_res - 1) * self.hop_length, dtype=np.float32)


def _golden_images(key):
    return np.load(os.path.join(GOLDEN, "reference_pipeline_cpu.npz"))[key]


def _host_u8_pipeline(monkeypatch):
    """The product's AudioDiffusionPipeline with its float->uint8 CUDA kernel replaced by the same torch expression, so
    that it runs on the CPU around the oracle U-Net (it then takes its unfused branch)."""
    from audio_diffusion_b200.pipeline import AudioDiffusionPipeline
    monkeypatch.setattr(AudioDiffusionPipeline, "images_to_u8",
                        staticmethod(lambda x: ((x / 2 + 0.5).clamp(0, 1) * 255).round().to(torch.uint8)))
    return AudioDiffusionPipeline


def _scheduler(sched):
    from audio_diffusion_b200.schedulers import DDIMScheduler, DDPMScheduler
    return DDIMScheduler() if sched == "ddim" else DDPMScheduler()


@pytest.mark.parametrize("sched", ["ddpm", "ddim"])
def test_unchanged_reference_pipeline_runs_on_the_shim(sched, monkeypatch):
    """`shim_<sched>` of tests/golden/reference_pipeline_cpu.npz holds the images the unchanged reference pipeline file
    returned on the import shim (the product's schedulers, the CPU oracle U-Net, batch 2, 4 steps, generator seed 42).
    The same loop by hand with the oracle schedulers, and the product's own pipeline on the same call, give those bytes."""
    from oracle.schedulers_oracle import OracleDDIM, OracleDDPM
    from oracle.unet_oracle import unet_forward
    gold = _golden_images(f"shim_{sched}")
    is_ddim = sched == "ddim"
    unet = OracleUNet()
    g = torch.Generator().manual_seed(42)
    x = torch.randn((2, 1, 16, 16), generator=g)
    o = OracleDDIM() if is_ddim else OracleDDPM()
    o.set_timesteps(4)
    for t in o.timesteps:
        eps = unet_forward(unet.w, unet.cfg, x, t)
        x = (o.step(eps, t, x, eta=0, generator=g) if is_ddim else o.step(eps, t, x, generator=g))["prev_sample"]
    ref = ((x / 2 + 0.5).clamp(0, 1).permute(0, 2, 3, 1).numpy() * 255).round().astype("uint8")[..., 0]
    assert np.array_equal(gold, ref), np.abs(gold.astype(int) - ref.astype(int)).max()
    pipe = _host_u8_pipeline(monkeypatch)(vqvae=None, unet=unet, mel=FakeMel(), scheduler=_scheduler(sched))
    assert pipe.get_default_steps() == (50 if is_ddim else 1000)
    pipe.set_progress_bar_config(disable=True)
    out = pipe(batch_size=2, steps=4, generator=torch.Generator().manual_seed(42))
    assert len(out.images) == 2 and out.images[0].size == (16, 16) and out.audios.shape == (2, 1, 15 * 512)
    got = np.stack([np.asarray(im) for im in out.images])
    assert np.array_equal(got, gold), np.abs(got.astype(int) - gold.astype(int)).max()


def _worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from audio_diffusion_b200.parallel import broadcast_parameters, shard_noise
    torch.manual_seed(100 + rank)                       # ranks start with different weights
    params = [torch.nn.Parameter(torch.randn(5, 3)), torch.nn.Parameter(torch.randn(7))]
    broadcast_parameters(params, src=0)
    full = torch.randn(8, 1, 4, 4, generator=torch.Generator().manual_seed(42))
    mine = shard_noise((8, 1, 4, 4), torch.Generator().manual_seed(42), rank, world, device="cpu")
    q.put((rank, [p.detach().clone() for p in params], mine, full))
    dist.barrier()
    dist.destroy_process_group()


def test_weight_broadcast_and_noise_sharding_gloo_world2():
    """⑤ multi-GPU host logic: one broadcast of the weights, batch rows sliced from ONE global RNG stream so that
    results are shard-count invariant (SURVEY §8e)."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=120) for _ in procs], key=lambda r: r[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    (r0, p0, m0, full), (r1, p1, m1, _) = res
    assert all(torch.equal(a, b) for a, b in zip(p0, p1))            # weights identical after the broadcast
    assert torch.equal(torch.cat([m0, m1]), full)                    # shards tile the global noise stream


def _hf_to_ldm_vae(w, num_blocks=4):
    """Inverse of the reference's key mapping: an `ldm` AutoencoderKL state dict (CompVis naming: down.{i}.block.{j},
    mid.block_1 / attn_1 / block_2, up.{i} counted from the LOW-resolution end, 1x1-conv attention projections)."""
    out = {}
    for k, v in w.items():
        n = k
        n = n.replace("conv_norm_out", "norm_out")
        for i in range(num_blocks):
            n = n.replace(f"encoder.down_blocks.{i}.resnets.", f"encoder.down.{i}.block.")
            n = n.replace(f"encoder.down_blocks.{i}.downsamplers.0.", f"encoder.down.{i}.downsample.")
        if n.startswith("decoder.up_blocks."):
            i = int(n.split(".")[2])
            n = n.replace(f"decoder.up_blocks.{i}.resnets.", f"decoder.up.{num_blocks - 1 - i}.block.")
            n = n.replace(f"decoder.up_blocks.{i}.upsamplers.0.", f"decoder.up.{num_blocks - 1 - i}.upsample.")
        n = n.replace("mid_block.resnets.0", "mid.block_1").replace("mid_block.resnets.1", "mid.block_2")
        if "mid_block.attentions.0" in n:
            n = n.replace("mid_block.attentions.0", "mid.attn_1")
            n = (n.replace("group_norm", "norm").replace("to_q", "q").replace("to_k", "k").replace("to_v", "v")
                  .replace("to_out.0", "proj_out"))
            if n.endswith(".weight") and v.dim() == 2:
                v = v[:, :, None, None]
        n = n.replace("conv_shortcut", "nin_shortcut")
        out[n] = v.clone()
    return out


def test_reference_vae_converter_feeds_the_b200_autoencoder():
    """audiodiffusion/utils.py:156-291 (`convert_ldm_vae_checkpoint`, UNCHANGED) turns an ldm-format checkpoint into
    exactly the state dict the B200 `AutoencoderKL` loads.  The converter's key mapping (ldm key -> hf key and shape, read
    off the reference by tests/golden/make_golden.py into vae_ldm_to_hf.json) is applied to an ldm checkpoint and the
    result must load strictly and give back every original tensor."""
    from audio_diffusion_b200.vae import AutoencoderKL                     # what the shim's `diffusers.AutoencoderKL` is
    from oracle.vae_oracle import VAEConfig, init_weights
    w = init_weights(VAEConfig(), seed=3)
    ldm = _hf_to_ldm_vae(w)
    assert any(k.startswith("encoder.down.0.block.0.") for k in ldm) and "decoder.mid.attn_1.q.weight" in ldm
    assert ldm["decoder.mid.attn_1.q.weight"].dim() == 4
    with open(os.path.join(GOLDEN, "vae_ldm_to_hf.json")) as f:
        mapping = json.load(f)["map"]
    assert {old for old, _, _ in mapping} == set(ldm)
    conv = {new: ldm[old].reshape(shape) for old, new, shape in mapping}
    vae = AutoencoderKL(in_channels=1, out_channels=1, down_block_types=("DownEncoderBlock2D",) * 4,
                        up_block_types=("UpDecoderBlock2D",) * 4, block_out_channels=(128, 256, 512, 512),
                        layers_per_block=2, latent_channels=1)
    vae.load_state_dict(conv)                                               # strict: every key must land
    sd = vae.state_dict()
    assert set(sd) == set(w) and len(sd) == 248
    for k in w:
        assert torch.equal(sd[k], w[k]), k


def test_gradient_allreduce_gloo_world2():
    """Data-parallel training's host logic (scripts/train_unet.py:181,259 via accelerate DDP): one all-reduce of the flat
    gradient buffer, mean over ranks — over gloo with world_size 2 (NCCL on the GPU box)."""
    code = f"""
import os, sys
sys.path.insert(0, {ROOT!r})
import torch, torch.distributed as dist
from audio_diffusion_b200.parallel import allreduce_mean_
rank = int(os.environ['RANK'])
dist.init_process_group('gloo', rank=rank, world_size=2)
flat = torch.arange(1000, dtype=torch.float32) * (rank + 1)
allreduce_mean_(flat)
assert torch.equal(flat, torch.arange(1000, dtype=torch.float32) * 1.5), flat[:4]
dist.destroy_process_group()
print('OK', rank)
"""
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29617", WORLD_SIZE="2")
    procs = [subprocess.Popen([sys.executable, "-c", code], env=dict(env, RANK=str(r)), stdout=subprocess.PIPE,
                              stderr=subprocess.PIPE, text=True) for r in range(2)]
    outs = [p.communicate(timeout=300) for p in procs]
    for p, (o, e) in zip(procs, outs):
        assert p.returncode == 0 and "OK" in o, o + e


def test_pipeline_directory_round_trip(tmp_path):
    """`pipeline.save_pretrained(dir)` / `AudioDiffusionPipeline.from_pretrained(dir)` (scripts/train_unet.py:106-111,
    :302-303; audiodiffusion/__init__.py:30-32) in the diffusers directory layout — model_index.json, unet/, vqvae/,
    scheduler/, mel/ — including a latent pipeline's AutoencoderKL and the deprecated attention key names of old hub files.
    Host logic only (no kernels run)."""
    import json

    from safetensors.torch import load_file, save_file

    from audio_diffusion_b200.mel import Mel
    from audio_diffusion_b200.pipeline import AudioDiffusionPipeline
    from audio_diffusion_b200.schedulers import DDIMScheduler
    from audio_diffusion_b200.unet import UNet2DModel
    from audio_diffusion_b200.vae import AutoencoderKL

    unet = UNet2DModel(sample_size=(8, 8), in_channels=1, out_channels=1, layers_per_block=1, block_out_channels=(128, 128),
                       down_block_types=("DownBlock2D", "AttnDownBlock2D"), up_block_types=("AttnUpBlock2D", "UpBlock2D"),
                       seed=1)
    vae = AutoencoderKL(in_channels=1, out_channels=1, down_block_types=("DownEncoderBlock2D",) * 2,
                        up_block_types=("UpDecoderBlock2D",) * 2, block_out_channels=(128, 128), layers_per_block=1,
                        latent_channels=1, seed=2)
    pipe = AudioDiffusionPipeline(vqvae=vae, unet=unet, mel=Mel(x_res=16, y_res=16, hop_length=256), scheduler=DDIMScheduler())
    d = str(tmp_path / "pipe")
    pipe.save_pretrained(d)
    idx = json.load(open(os.path.join(d, "model_index.json")))
    assert idx["unet"][1] == "UNet2DModel" and idx["vqvae"][1] == "AutoencoderKL" and idx["scheduler"][1] == "DDIMScheduler"
    # rewrite the U-Net weights with the deprecated attention names of older hub checkpoints
    f = os.path.join(d, "unet", "diffusion_pytorch_model.safetensors")
    sd = load_file(f)
    ren = {".to_q.": ".query.", ".to_k.": ".key.", ".to_v.": ".value.", ".to_out.0.": ".proj_attn."}
    old = {}
    for k, v in sd.items():
        for a, b in ren.items():
            k = k.replace(a, b)
        old[k] = v
    assert any(".query." in k for k in old)
    save_file(old, f)
    back = AudioDiffusionPipeline.from_pretrained(d)
    assert isinstance(back.scheduler, DDIMScheduler) and back.mel.x_res == 16 and back.mel.hop_length == 256
    for k, v in unet.state_dict().items():
        assert torch.equal(back.unet.state_dict()[k], v), k
    for k, v in vae.state_dict().items():
        assert torch.equal(back.vqvae.state_dict()[k], v), k
    assert back.unet.sample_size in ((8, 8), [8, 8]) and back.vqvae.config["latent_channels"] == 1


class ScriptedMel(FakeMel):
    """FakeMel plus the audio-conditioning surface (`load_audio`, `audio_slice_to_image`) with a fixed image."""

    def load_audio(self, audio_file=None, raw_audio=None):
        self.loaded = True

    def audio_slice_to_image(self, slice):
        from PIL import Image
        rng = np.random.default_rng(5)
        return Image.fromarray(rng.integers(0, 256, (self.y_res, self.x_res), dtype=np.uint8))


def cond_call(sched):
    """Arguments of the audio-conditioned / in-painting call (`raw_audio`, `start_step`, `mask_start_secs`,
    `mask_end_secs`, pipeline_audio_diffusion.py:133-185) the product's pipeline is compared on."""
    kw = dict(batch_size=1, raw_audio=np.zeros(16 * 512 * 2, dtype=np.float32), slice=0, start_step=2, steps=6,
              noise=torch.randn(1, 1, 16, 16, generator=torch.Generator().manual_seed(3)),   # start_step is batch-1 only (:150)
              step_generator=torch.Generator().manual_seed(4), mask_start_secs=0.05, mask_end_secs=0.05, return_dict=False)
    if sched == "ddim":
        kw["eta"] = 0.5
    return kw


@pytest.mark.parametrize("sched", ["ddpm", "ddim"])
def test_mirrored_pipeline_equals_reference_pipeline_on_cpu(sched, monkeypatch):
    """The product's own `AudioDiffusionPipeline.__call__` (audio_diffusion_b200/pipeline.py) against the images the
    reference's unchanged file returned for the audio-conditioned / in-painting path (`cond_<sched>` of
    tests/golden/reference_pipeline_cpu.npz): identical uint8 images, both driving the CPU oracle U-Net.  For DDIM also
    the inversion (`encode`, :207-242) and `slerp` (:244-263) give the reference's numbers."""
    Mirror = _host_u8_pipeline(monkeypatch)
    pipe = Mirror(vqvae=None, unet=OracleUNet(), mel=ScriptedMel(), scheduler=_scheduler(sched))
    pipe.set_progress_bar_config(disable=True)
    images, (sr, audios) = pipe(**cond_call(sched))
    got, gold = np.stack([np.asarray(im) for im in images]), _golden_images(f"cond_{sched}")
    assert sr == 22050 and len(audios) == 1
    assert gold.shape == (1, 16, 16) and np.array_equal(got, gold), np.abs(got.astype(int) - gold.astype(int)).max()
    if sched == "ddim":
        from PIL import Image
        rng = np.random.default_rng(9)
        pil = [Image.fromarray(rng.integers(0, 256, (16, 16), dtype=np.uint8)) for _ in range(2)]
        pipe = Mirror(vqvae=None, unet=OracleUNet(), mel=ScriptedMel(), scheduler=_scheduler("ddim"))
        pipe.set_progress_bar_config(disable=True)
        enc = pipe.encode(pil, steps=5)
        assert enc.shape == (2, 1, 16, 16) and torch.equal(enc, torch.from_numpy(_golden_images("encode_ddim")))
        a = torch.randn(4, 4, generator=torch.Generator().manual_seed(1))
        b = torch.randn(4, 4, generator=torch.Generator().manual_seed(2))
        assert torch.equal(Mirror.slerp(a, b, 0.3), torch.from_numpy(_golden_images("slerp")))


MEL_CASES = [(256, 256, 512), (64, 64, 1024), (96, 32, 256)]     # (x_res, y_res, hop_length)


def test_mel_host_logic_equals_reference_mel():
    """Slicing / padding / resolution bookkeeping of the engine's `Mel` against the reference's own `audiodiffusion/mel.py`
    class (mel.py:80-133) on the same seeded audio: sizes, dtype and the bytes of the padded audio and of every slice,
    as tests/golden/mel_host_logic.json records them."""
    from audio_diffusion_b200.mel import Mel
    with open(os.path.join(GOLDEN, "mel_host_logic.json")) as f:
        cases = iter(json.load(f)["cases"])
    rng = np.random.default_rng(0)
    for (x_res, y_res, hop) in MEL_CASES:
        for n in [10, x_res * hop - 1, x_res * hop, 3 * x_res * hop + 17]:
            c = next(cases)
            assert (c["x_res"], c["y_res"], c["hop_length"], c["n"]) == (x_res, y_res, hop, n)
            b = Mel(x_res=x_res, y_res=y_res, hop_length=hop)
            b.load_audio(raw_audio=rng.standard_normal(n).astype(np.float32))
            assert (b.slice_size, b.n_mels, b.get_sample_rate()) == (c["slice_size"], c["n_mels"], c["sample_rate"])
            assert b.get_number_of_slices() == c["slices"], (x_res, n)
            assert len(b.audio) == c["audio_len"] and str(b.audio.dtype) == c["audio_dtype"]
            assert hashlib.sha256(b.audio.tobytes()).hexdigest() == c["audio_sha256"]
            slices = hashlib.sha256()
            for s in range(b.get_number_of_slices()):
                slices.update(b.get_audio_slice(s).tobytes())
            assert slices.hexdigest() == c["slices_sha256"]
        b.set_resolution(32, 16)
        assert [b.x_res, b.y_res, b.n_mels, b.slice_size] == c["after_set_resolution_32_16"]
    assert next(cases, None) is None


def test_model_mixin_round_trip_and_conditional_unet_surface(tmp_path):
    """SURVEY §8 f3 boundary: a model built the way the reference's audiodiffusion/audio_encoder.py builds its encoder (a
    `diffusers` ModelMixin + ConfigMixin subclass with an argument-free constructor that holds a `diffusers.Mel`) saves and
    loads through the shim's hub layout, and `diffusers.UNet2DConditionModel` resolves to the engine's class with exactly
    the diffusers state-dict keys / shapes of the architecture scripts/train_unet.py:139-159 builds."""
    code = f"""
import sys
sys.path[:0] = [{ROOT!r}, {os.path.join(ROOT, 'audio_diffusion_b200', 'compat')!r}]
import torch
from diffusers import ConfigMixin, Mel, ModelMixin

class Encoder(ModelMixin, ConfigMixin):
    def __init__(self):
        super().__init__()
        self.mel = Mel(x_res=216, y_res=96)
        self.conv = torch.nn.Sequential(torch.nn.Conv2d(1, 8, 3, padding=1), torch.nn.BatchNorm2d(8), torch.nn.ReLU(),
                                        torch.nn.MaxPool2d(4), torch.nn.Dropout(0.2))
        self.embedding = torch.nn.Linear(8 * 24 * 54, 100)

    def forward(self, x):
        return self.embedding(self.conv(x).flatten(1))

torch.manual_seed(0)
enc = Encoder().eval()
y = enc(torch.rand(2, 1, 96, 216))
assert y.shape == (2, 100)
d = {str(tmp_path / 'enc')!r}
enc.save_pretrained(d)
again = Encoder.from_pretrained(d).eval()
assert torch.equal(again(torch.ones(1, 1, 96, 216)), enc(torch.ones(1, 1, 96, 216)))
from diffusers import UNet2DConditionModel
from audio_diffusion_b200.unet_cond import UNet2DConditionModel as engine_class
assert engine_class is UNet2DConditionModel
u = UNet2DConditionModel(sample_size=(32, 32), in_channels=1, out_channels=1, layers_per_block=2,
                         block_out_channels=(128, 256, 512, 512),
                         down_block_types=("CrossAttnDownBlock2D",) * 3 + ("DownBlock2D",),
                         up_block_types=("UpBlock2D",) + ("CrossAttnUpBlock2D",) * 3, cross_attention_dim=100)
from oracle.unet_cond_oracle import CondUNetConfig, param_shapes
sh = param_shapes(CondUNetConfig(sample_size=(32, 32)))
sd = u.state_dict()
assert set(sh) == set(sd) and all(tuple(sd[k].shape) == tuple(sh[k]) for k in sh)
assert sum(v.numel() for v in sd.values()) == 135559809
print('ok')
"""
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr[-2000:]


def test_grad_bucket_bounds_are_parameter_boundaries():
    """Buckets of the (opt-in) overlapped gradient all-reduce: ascending, start at 0, end at the buffer size, every inner
    boundary on a parameter's start offset (b200ad_unet_set_grad_buckets requires it)."""
    from audio_diffusion_b200.parallel import grad_bucket_bounds
    sizes = [1152, 128, 147456, 128, 65536, 512, 589824, 256, 36864, 128]
    offs, tot = [], 0
    for n in sizes:
        offs.append(tot)
        tot += n
    b = grad_bucket_bounds(offs, tot, nbuckets=4)
    assert b[0] == 0 and b[-1] == tot and all(x < y for x, y in zip(b, b[1:]))
    assert all(x in offs for x in b[1:-1])
    assert grad_bucket_bounds([0], 100, nbuckets=4) == [0, 100]          # a single tensor: one bucket


def test_bench_extras_formatting():
    """bench.py's `configs` object (C3 / C4 / B1 / C5 / Mel) is assembled on the host from a flat {name: seconds} dict that
    travelled through a max-over-ranks all-reduce: every sub-object and the rates derived from it."""
    import importlib.util
    import os
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(os.path.dirname(__file__), "..", "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    ex = {"c3_step_s": 0.035, "c3_tail_s": 0.07, "c3_call50_s": 1.82, "mel_encode_s": 0.0013, "mel_decode_s": 0.034,
          "c4_step_s": 0.0081, "c4_tail_s": 0.18, "c4_vae_decode_s": 0.078, "b1_step_s": 0.0046, "b1_host_enqueue_s": 0.0044,
          "b1_launches": 123.0, "b1_graph_step_s": 0.0044, "c5_step_s": 0.051, "c5_step_nosync_s": 0.050, "c5_launches": 830.0}
    out = bench.format_extras(ex, 2, 1439.1, 6572.5)
    assert set(out) == {"C3_ddim50", "C4_latent", "B1_latency", "C5_train", "mel_codec"}
    assert abs(out["C3_ddim50"]["value"] - 128 / (50 * 0.035 + 0.07)) < 1e-9
    assert abs(out["C5_train"]["value"] - 32 / 0.051) < 1e-9 and abs(out["C5_train"]["exposed_allreduce_ms"] - 1.0) < 1e-6
    assert out["B1_latency"]["ms_per_step"] == 4.4 and out["mel_codec"]["decode_frac"] < 1


def test_bench_dump_outputs(tmp_path, monkeypatch):
    """bench.py --dump-outputs: float32 .npy files; a tensor over the size cap keeps the same seeded rows on every call."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    small = torch.randn(3, 1, 4, 4, dtype=torch.float64)
    bench.dump_outputs(str(tmp_path / "a"), {"sample": small})
    got = np.load(tmp_path / "a" / "sample.npy")
    assert got.dtype == np.float32 and np.array_equal(got, small.float().numpy())
    monkeypatch.setattr(bench, "MAX_DUMP_BYTES", 5 * 16 * 4)                 # room for 5 of the 12 samples
    big = torch.randn(12, 1, 4, 4)
    for d in ("b", "c"):
        bench.dump_outputs(str(tmp_path / d), {"sample": big})
    b, c = np.load(tmp_path / "b" / "sample.npy"), np.load(tmp_path / "c" / "sample.npy")
    assert b.shape == (5, 1, 4, 4) and b.nbytes <= bench.MAX_DUMP_BYTES and np.array_equal(b, c)
    assert all(any(np.array_equal(r, s) for s in big.numpy()) for r in b)
