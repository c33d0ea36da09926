"""A training script driven end to end on the engine's import surfaces (`audio_diffusion_b200/compat`: diffusers,
accelerate) through `python -m audio_diffusion_b200.compat.run`: two epochs on a synthetic on-disk dataset,
`save_pretrained`, then a resumed run with `--from_pretrained` and `--start_epoch`.

The script is tests/shims/train_unet.py, written against the same import surfaces as the upstream
scripts/train_unet.py.  With AUDIO_DIFFUSION_SRC naming an unchanged teticio/audio-diffusion checkout, the upstream
script runs instead, byte-identical (train_unet.py:106-111, :216-224, :302-303).

The product's UNet2DModel has no CPU path, so `diffusers.UNet2DModel` is overlaid by a test-only autograd module backed
by the oracle (tests/shims/cpu_unet); everything else — Accelerator, schedulers, EMA, LR schedule, pipeline save / load,
Mel — is the product code the GPU run uses."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("AUDIO_DIFFUSION_SRC")
SCRIPT = (os.path.join(REF, "scripts", "train_unet.py") if REF else
          os.path.join(ROOT, "tests", "shims", "train_unet.py"))


def _run(args, tmp_path, timeout=900):
    env = dict(os.environ, PYTHONPATH=ROOT, B200AD_COMPAT_OVERLAY=os.path.join(ROOT, "tests", "shims", "cpu_unet"),
               CUDA_VISIBLE_DEVICES="", OMP_NUM_THREADS="8")
    r = subprocess.run([sys.executable, "-m", "audio_diffusion_b200.compat.run", SCRIPT] + args, cwd=str(tmp_path), env=env,
                       capture_output=True, text=True, timeout=timeout)
    assert r.returncode == 0, r.stderr[-3000:]
    return r


def test_unchanged_train_script_two_epochs_then_resume(tmp_path):
    import datasets
    from PIL import Image
    rng = np.random.default_rng(0)
    imgs = [Image.fromarray(rng.integers(0, 256, (32, 32), dtype=np.uint8)) for _ in range(4)]
    ds = datasets.Dataset.from_dict({"image": imgs, "audio_file": [f"a{i}.wav" for i in range(4)], "slice": list(range(4))})
    data = tmp_path / "data"
    datasets.DatasetDict({"train": ds}).save_to_disk(str(data))
    out = tmp_path / "model"
    common = ["--dataset_name", str(data), "--output_dir", str(out), "--train_batch_size", "2",
              "--lr_warmup_steps", "2", "--hop_length", "512"]
    _run(common + ["--num_epochs", "2", "--gradient_accumulation_steps", "2"], tmp_path)
    # the directory the script wrote follows the upstream layout (model_index.json with diffusers / audio_diffusion names)
    index = json.load(open(out / "model_index.json"))
    assert index["_class_name"] == "AudioDiffusionPipeline"
    assert index["unet"] == ["diffusers", "UNet2DModel"] and index["scheduler"] == ["diffusers", "DDPMScheduler"]
    assert index["mel"] == ["audio_diffusion", "Mel"]
    assert (out / "unet" / "diffusion_pytorch_model.safetensors").exists() and (out / "mel" / "mel_config.json").exists()
    cfg = json.load(open(out / "unet" / "config.json"))
    assert tuple(cfg["block_out_channels"]) == (128, 128, 256, 256, 512, 512) and cfg["sample_size"] == [32, 32]
    from safetensors.torch import load_file
    w1 = {k: v.clone() for k, v in load_file(str(out / "unet" / "diffusion_pytorch_model.safetensors")).items()}  # file is rewritten below
    logs = list((out / "logs").rglob("events.out.tfevents.*"))
    assert logs, "accelerator.log -> tensorboard event file"
    # resume: --from_pretrained + --start_epoch 2 fast-forwards optimizer / LR schedule / EMA step count, trains epoch 2
    _run(common + ["--num_epochs", "3", "--start_epoch", "2", "--from_pretrained", str(out)], tmp_path)
    w2 = load_file(str(out / "unet" / "diffusion_pytorch_model.safetensors"))
    assert set(w1) == set(w2)
    assert any(not np.array_equal(w1[k].numpy(), w2[k].numpy()) for k in ("conv_in.weight", "conv_out.weight"))
