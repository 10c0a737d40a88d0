"""Progressive distillation driver (Salimans & Ho, 2022): from a teacher checkpoint sampled with --teacher-steps DDIM steps, each
stage trains a student that samples in half as many (DistillationStep), on one GPU or under torchrun.

    torchrun --nproc-per-node 8 -m v_diffusion_b200.distill --config-path cfg.json --default-config-path defaults.json \
        --ckpt-path ckpt.pt --use-ema --images train_uint8.npy --labels train_labels.npy --teacher-steps 1024 --stages 4 \
        --iters 20000 --batch-size 128 --lr 1e-4 --w-guide 0 --out-dir distill/

--images / --labels: the layout bpd.py reads (uint8 NHWC images; (N,) class ids 1 ... num_classes or (N, num_classes) multi-hot
rows).  --batch-size is per GPU; every rank draws its own batches (seeded by --seed and its rank).

Stage k (1-based) distils the current teacher at 2N steps into a student at N = --teacher-steps / 2^k: the student starts as a
copy of the teacher with fresh AdamW state, the learning rate decays linearly from --lr to 0 over --iters, and the stage writes
<out-dir>/student_N.pt in TrainingStep.checkpoint's layout plus "sample_timesteps": N and "distill_w_guide": w.  The student's
EMA weights (its raw weights with --no-ema) are the next stage's teacher.  A checkpoint loads with
``generate --ckpt-path student_N.pt --use-ema --sample-timesteps N --use-ddim`` (with --w-guide 0 after a guided teacher,
--w-guide > 0: the student learned the guided prediction).
"""
import argparse
import json
import os
import time

import numpy as np
import torch
import torch.distributed as dist

from .bpd import card, images_to_model_space
from .generate import load_reference_checkpoint


@torch.no_grad()
def _broadcast_(tensors):
    """Every rank takes rank 0's values (the EMA shadow lives on the leader only)."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        for t in tensors:
            dist.broadcast(t, src=0)


def main(argv=None):
    from . import load_config, build_from_config
    from .training import DistillationStep
    ap = argparse.ArgumentParser()
    ap.add_argument("--config-path", required=True)
    ap.add_argument("--default-config-path", default=None, help="defaults merged under --config-path (none when omitted)")
    ap.add_argument("--ckpt-path", required=True, help="teacher: reference or TrainingStep checkpoint (.pt)")
    ap.add_argument("--use-ema", action="store_true", help="start from the teacher checkpoint's EMA weights")
    ap.add_argument("--images", required=True, help=".npy of uint8 NHWC training images")
    ap.add_argument("--labels", default=None, help=".npy of class ids (N,) or multi-hot rows (N, num_classes)")
    ap.add_argument("--teacher-steps", type=int, required=True, help="2 N0: the DDIM steps of the first teacher")
    ap.add_argument("--stages", type=int, default=1, help="halvings of the step count")
    ap.add_argument("--iters", type=int, required=True, help="optimizer steps per stage")
    ap.add_argument("--batch-size", type=int, default=128, help="per GPU")
    ap.add_argument("--lr", type=float, default=1e-4, help="initial learning rate of every stage (decays linearly to 0)")
    ap.add_argument("--ema-decay", type=float, default=0.9999)
    ap.add_argument("--no-ema", action="store_true", help="keep no EMA: the raw weights are the next teacher")
    ap.add_argument("--w-guide", type=float, default=0.0, help="> 0: distil the guided teacher into a student sampled without CFG")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out-dir", required=True)
    args = ap.parse_args(argv)
    if args.stages < 1 or args.iters < 1 or args.batch_size < 1:
        ap.error("--stages, --iters and --batch-size must be >= 1")
    if args.teacher_steps < 2 or args.teacher_steps % (1 << args.stages):
        ap.error(f"--teacher-steps must be a multiple of 2^stages = {1 << args.stages}")
    if args.w_guide < 0:
        ap.error("--w-guide must be >= 0")

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
    p_uncond = float(config.get("conditional", {}).get("p_uncond", 0.1))
    images = np.load(args.images, mmap_mode="r")
    labels = torch.from_numpy(np.load(args.labels)) if args.labels else None
    if labels is not None and labels.shape[0] != images.shape[0]:
        raise ValueError(f"--labels has {labels.shape[0]} rows for {images.shape[0]} images")
    if args.w_guide > 0 and labels is None:
        raise ValueError("--w-guide > 0 needs a class-conditional teacher and --labels")
    os.makedirs(args.out_dir, exist_ok=True)

    teacher_sd = state_dict
    gen = torch.Generator().manual_seed(args.seed * 7919 + rank)
    for stage in range(1, args.stages + 1):
        N = args.teacher_steps >> stage
        diffusion, teacher, chw = build_from_config(config, use_cfg, 0.0, N)
        diffusion.p_uncond = p_uncond
        if stage == 1:
            if images.dtype != np.uint8 or images.ndim != 4 or tuple(images.shape[1:]) != (chw[1], chw[2], chw[0]):
                raise ValueError(f"--images must be uint8 NHWC (N, {chw[1]}, {chw[2]}, {chw[0]}), got {images.dtype} "
                                 f"{tuple(images.shape)}")
            if teacher.num_classes and labels is None:
                raise ValueError("a class-conditional network needs --labels")
        teacher.load_state_dict(teacher_sd)
        teacher = teacher.to(device).eval()
        _, student, _ = build_from_config(config, use_cfg, 0.0, N)
        student.load_state_dict(teacher_sd)
        student = student.to(device).train()
        ds = DistillationStep(student, teacher, diffusion, w_guide=args.w_guide, lr=args.lr, use_ema=not args.no_ema,
                              ema_decay=args.ema_decay, distributed=world > 1, rank=rank, world_size=world, device=device)
        losses, t0 = [], time.perf_counter()
        for it in range(args.iters):
            idx = torch.randint(images.shape[0], (args.batch_size,), generator=gen).sort().values.numpy()
            x = images_to_model_space(images[idx], device)
            y = None if labels is None else labels[idx].to(device)
            loss = ds.step(x, y, lr=args.lr * (1.0 - it / args.iters))       # linear decay to 0 (the paper's schedule)
            losses.append(loss)
        losses = torch.stack(losses).cpu().tolist()
        torch.cuda.synchronize()
        seconds = time.perf_counter() - t0
        path = os.path.join(args.out_dir, f"student_{N}.pt")
        ds.save_checkpoint(path, epoch=stage, sample_timesteps=N, distill_w_guide=args.w_guide)
        # the next teacher: the EMA shadow (kept by the leader only, so broadcast) or the raw weights
        src = ds.optimizer.shadow if ds.optimizer.shadow else dict(student.named_parameters())
        nxt = {k: src[k].detach().clone() for k, _ in student.named_parameters()}
        _broadcast_(list(nxt.values()))
        teacher_sd = {k: v.cpu() for k, v in nxt.items()}
        if rank == 0:
            print(json.dumps({"stage": stage, "student_steps": N, "teacher_steps": 2 * N, "iters": args.iters,
                              "loss_first": losses[0], "loss_last": losses[-1], "seconds": seconds,
                              "ckpt": path, "n_gpus": world, "card": card()}), flush=True)
        del ds, student, teacher
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
