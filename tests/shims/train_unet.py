"""Test-only training script for tests/test_cpu_train_script.py: DDPM training of the audio-diffusion-256 U-Net
architecture on an on-disk dataset of mel-spectrogram images, written against the import surfaces an upstream
audio-diffusion training script uses (`accelerate`, `diffusers`, `datasets`), so that the engine's versions of them run
end to end under `python -m audio_diffusion_b200.compat.run`.

It covers: Accelerator with gradient accumulation, clipping and a TensorBoard tracker; get_scheduler (cosine with
warm-up); EMAModel; DDPMScheduler.add_noise; AudioDiffusionPipeline.save_pretrained in the upstream directory layout;
and a resumed run (--from_pretrained, --start_epoch) that fast-forwards the LR schedule and the EMA step count over
the epochs already trained."""
import argparse
import math
import os

import numpy as np
import torch
import torch.nn.functional as F
from accelerate import Accelerator
from accelerate.logging import get_logger
from accelerate.utils import ProjectConfiguration
from datasets import load_from_disk
from diffusers import DDPMScheduler, UNet2DModel
from diffusers.optimization import get_scheduler
from diffusers.pipelines.audio_diffusion import Mel
from diffusers.training_utils import EMAModel

from audio_diffusion_b200.pipeline import AudioDiffusionPipeline

ARCH = dict(in_channels=1, out_channels=1, layers_per_block=2, block_out_channels=(128, 128, 256, 256, 512, 512),
            down_block_types=("DownBlock2D",) * 4 + ("AttnDownBlock2D", "DownBlock2D"),
            up_block_types=("UpBlock2D", "AttnUpBlock2D") + ("UpBlock2D",) * 4)


def to_batch(rows):
    """uint8 greyscale images -> float [-1, 1], (B, 1, H, W)."""
    x = np.stack([np.asarray(r["image"], dtype=np.float32) for r in rows]) / 255.0
    return {"input": torch.from_numpy((x - 0.5) / 0.5)[:, None]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--dataset_name", required=True)
    ap.add_argument("--output_dir", required=True)
    ap.add_argument("--train_batch_size", type=int, default=16)
    ap.add_argument("--num_epochs", type=int, default=1)
    ap.add_argument("--start_epoch", type=int, default=0)
    ap.add_argument("--gradient_accumulation_steps", type=int, default=1)
    ap.add_argument("--learning_rate", type=float, default=1e-4)
    ap.add_argument("--lr_warmup_steps", type=int, default=500)
    ap.add_argument("--hop_length", type=int, default=512)
    ap.add_argument("--from_pretrained", default=None)
    args = ap.parse_args()

    acc = Accelerator(gradient_accumulation_steps=args.gradient_accumulation_steps, log_with="tensorboard",
                      project_config=ProjectConfiguration(project_dir=".",
                                                          logging_dir=os.path.join(args.output_dir, "logs")))
    logger = get_logger(__name__)
    dataset = load_from_disk(args.dataset_name)["train"]
    width, height = dataset[0]["image"].size
    loader = torch.utils.data.DataLoader(dataset, batch_size=args.train_batch_size, shuffle=True, collate_fn=to_batch)

    if args.from_pretrained is not None:
        pipe = AudioDiffusionPipeline.from_pretrained(args.from_pretrained)
        model, noise_scheduler, mel = pipe.unet, pipe.scheduler, pipe.mel
    else:
        model = UNet2DModel(sample_size=(height, width), **ARCH)
        noise_scheduler = DDPMScheduler(num_train_timesteps=1000)
        mel = Mel(x_res=width, y_res=height, hop_length=args.hop_length)

    optimizer = torch.optim.AdamW(model.parameters(), lr=args.learning_rate, betas=(0.95, 0.999), weight_decay=1e-6,
                                  eps=1e-8)
    steps_per_epoch = math.ceil(len(loader) / args.gradient_accumulation_steps)
    lr_scheduler = get_scheduler("cosine", optimizer, num_warmup_steps=args.lr_warmup_steps,
                                 num_training_steps=steps_per_epoch * args.num_epochs)
    model, optimizer, loader, lr_scheduler = acc.prepare(model, optimizer, loader, lr_scheduler)
    ema = EMAModel(model.parameters(), inv_gamma=1.0, power=0.75, max_value=0.9999)
    if acc.is_main_process:
        acc.init_trackers("train_unet")

    global_step = 0
    for epoch in range(args.num_epochs):
        if epoch < args.start_epoch:          # trained by the run being resumed: advance the schedules only
            for _ in range(steps_per_epoch):
                lr_scheduler.step()
                ema.optimization_step += 1
            global_step += len(loader)
            continue
        model.train()
        for batch in loader:
            clean = batch["input"]
            noise = torch.randn_like(clean)
            t = torch.randint(0, noise_scheduler.config.num_train_timesteps, (clean.shape[0],), device=clean.device)
            noisy = noise_scheduler.add_noise(clean, noise, t)
            with acc.accumulate(model):
                loss = F.mse_loss(model(noisy, t)["sample"], noise)
                acc.backward(loss)
                if acc.sync_gradients:
                    acc.clip_grad_norm_(model.parameters(), 1.0)
                optimizer.step()
                lr_scheduler.step()
                if acc.sync_gradients:
                    ema.step(model.parameters())
                optimizer.zero_grad()
            global_step += 1
            acc.log({"loss": loss.item(), "lr": lr_scheduler.get_last_lr()[0], "ema_decay": ema.cur_decay_value},
                    step=global_step)
        logger.info("epoch %d done, step %d", epoch, global_step)
        acc.wait_for_everyone()

    if acc.is_main_process:
        unet = acc.unwrap_model(model)
        ema.copy_to(unet.parameters())
        AudioDiffusionPipeline(vqvae=None, unet=unet, mel=mel, scheduler=noise_scheduler).save_pretrained(args.output_dir)
    acc.end_training()


if __name__ == "__main__":
    main()
