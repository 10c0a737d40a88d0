"""Likelihood driver: the negative ELBO in bits/dim of a set of images under a checkpoint (GaussianDiffusion.calc_all_bpd),
alone or sharded over the GPUs of one node.

    torchrun --nproc-per-node 8 -m v_diffusion_b200.bpd --config-path cfg.json --default-config-path defaults.json \
        --ckpt-path ckpt.pt --use-ema --images test_uint8.npy --labels test_labels.npy --batch-size 256 --seed 0 --out bpd.json

--images: uint8 NHWC (N, R, R, C), the layout images_to_uint8 writes; they map to model space as (x / 255 - 0.5) / 0.5 in fp32
(ToTensor, then Normalize(0.5, 0.5)).  --labels: (N,) class ids as the network takes them (1 ... num_classes, 0 = no class),
or (N, num_classes) multi-hot rows for a multitag network.  The images are cut into global batches of --batch-size; batch k
draws its q-sample noise from the stream keyed by seed + k, and rank r runs a contiguous run of batches, so every image's
result is the same at any world size.  The bound uses --sample-timesteps steps (T = 1000 is the usual figure) and follows
the standard definition written out in include/vdt_b200.h; it is not pinned to the reference's own likelihood code.
"""
import argparse
import json
import math
import os
import subprocess

import numpy as np
import torch
import torch.distributed as dist

from .generate import gather_shards, load_reference_checkpoint, shard_bounds


def card():
    """Name, power limit and max SM clock of the current GPU, read alongside the numbers they qualify."""
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm",
                           "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        if q.returncode == 0 and q.stdout.strip():
            return q.stdout.strip().splitlines()[0]
    except (OSError, subprocess.TimeoutExpired):
        pass
    return torch.cuda.get_device_name()


def images_to_model_space(images, device):
    """uint8 NHWC -> fp32 NCHW in [-1, 1]: ToTensor (x / 255) then Normalize(0.5, 0.5)."""
    x = torch.from_numpy(np.ascontiguousarray(images)).to(device).permute(0, 3, 1, 2).to(torch.float32)
    return ((x / 255.0 - 0.5) / 0.5).contiguous()


def main():
    from . import load_config, build_from_config
    ap = argparse.ArgumentParser()
    ap.add_argument("--config-path", required=True)
    ap.add_argument("--default-config-path", default=None, help="defaults merged under --config-path (none when omitted)")
    ap.add_argument("--ckpt-path", required=True, help="reference or TrainingStep checkpoint (.pt)")
    ap.add_argument("--use-ema", action="store_true")
    ap.add_argument("--images", required=True, help=".npy of uint8 NHWC images")
    ap.add_argument("--labels", default=None, help=".npy of class ids (N,) or multi-hot rows (N, num_classes)")
    ap.add_argument("--sample-timesteps", type=int, default=1000, help="T, the number of steps of the bound")
    ap.add_argument("--no-clip-denoised", action="store_true", help="do not clip the x0 predictions to [-1, 1]")
    ap.add_argument("--batch-size", type=int, default=256)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", required=True, help="JSON result (rank 0)")
    args = ap.parse_args()
    if args.batch_size < 1:
        ap.error("--batch-size must be >= 1")

    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    rank = dist.get_rank() if world > 1 else 0

    state_dict, use_cfg = load_reference_checkpoint(args.ckpt_path, args.use_ema)
    if args.default_config_path:
        config = load_config(args.config_path, args.default_config_path)
    else:
        with open(args.config_path) as f:
            config = json.load(f)
    diffusion, model, chw = build_from_config(config, use_cfg, 0.0, args.sample_timesteps)
    model.load_state_dict(state_dict)
    model = model.to(device).eval()

    images = np.load(args.images, mmap_mode="r")
    if images.dtype != np.uint8 or images.ndim != 4 or tuple(images.shape[1:]) != (chw[1], chw[2], chw[0]):
        raise ValueError(f"--images must be uint8 NHWC (N, {chw[1]}, {chw[2]}, {chw[0]}), got {images.dtype} "
                         f"{tuple(images.shape)}")
    labels = None
    if args.labels:
        labels = torch.from_numpy(np.load(args.labels))
        if labels.shape[0] != images.shape[0]:
            raise ValueError(f"--labels has {labels.shape[0]} rows for {images.shape[0]} images")
    elif model.num_classes:
        raise ValueError("a class-conditional network needs --labels (0 ids evaluate it unconditionally)")

    T, N, bs = args.sample_timesteps, images.shape[0], args.batch_size
    nb = (N + bs - 1) // bs
    b_lo, b_hi = shard_bounds(nb, rank, world)
    rows = []
    for k in range(b_lo, b_hi):
        i0, i1 = k * bs, min(N, (k + 1) * bs)
        x0 = images_to_model_space(images[i0:i1], device)
        y = None if labels is None else labels[i0:i1]
        total, terms, prior, _ = diffusion.calc_all_bpd(model, x0, y=y, clip_denoised=not args.no_clip_denoised, device=device,
                                                        seed=args.seed + k)
        row = torch.full((bs, T + 2), float("nan"), dtype=torch.float64)
        row[: i1 - i0, 0], row[: i1 - i0, 1], row[: i1 - i0, 2:] = total, prior, terms
        rows.append(row)
    local = torch.stack(rows) if rows else torch.zeros((0, bs, T + 2), dtype=torch.float64)
    # whole batches travel, so gather_shards' per-rank split (shard_bounds over the batches) matches the one above
    every = gather_shards(local.to(device), nb).cpu().reshape(nb * bs, T + 2)[:N]
    if rank == 0:
        total = every[:, 0]
        result = {"total_bpd_mean": total.mean().item(),
                  "total_bpd_stderr": (total.std().item() / math.sqrt(N)) if N > 1 else float("nan"),
                  "prior_bpd_mean": every[:, 1].mean().item(), "terms_bpd_mean": every[:, 2:].mean(0).tolist(),
                  "sample_timesteps": T, "images": N, "n_gpus": world, "card": card(),
                  "total_bpd": total.tolist()}
        with open(args.out, "w") as f:
            json.dump(result, f)
        print(json.dumps({k: v for k, v in result.items() if k not in ("terms_bpd_mean", "total_bpd")}), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
