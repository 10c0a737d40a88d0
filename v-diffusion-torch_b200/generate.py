"""Sampling driver: the batch loop of the reference's generate.py (generate.py:100-150) sharded over the GPUs
of one node.  Every sample's trajectory is independent (GroupNorm is per sample, attention per image, the CFG
pair lives inside one sample), so rank r simply owns a contiguous slice of the global batch, with its own noise,
labels, weight replica and CUDA graphs; there is no communication inside the loop.  The only collective is the
final gather of the images (as in Trainer.sample_fn, train_utils.py:181-183).

    torchrun --nproc-per-node 8 -m v_diffusion_b200.generate --config-path cfg.json --default-config-path defaults.json \
        --ckpt-path ckpt.pt --use-ddim --sample-timesteps 100 --w-guide 1.0 --total-size 32768 --save-path out.pt
"""
import argparse
import json
import math
import os
import sys
import time

import torch
import torch.distributed as dist


def shard_bounds(total, rank, world):
    """Contiguous, balanced split of `total` samples: the first total % world ranks get one extra."""
    base, extra = divmod(total, world)
    start = rank * base + min(rank, extra)
    return start, start + base + (1 if rank < extra else 0)


def gather_shards(local, total, group=None):
    """all_gather of per-rank shards of (possibly) different length along dim 0 -> (total, ...) on every rank."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return local
    world = dist.get_world_size(group)
    width = math.ceil(total / world)
    pad = torch.zeros((width,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    pad[: local.shape[0]] = local
    parts = [torch.empty_like(pad) for _ in range(world)]
    dist.all_gather(parts, pad, group=group)
    out = []
    for r, part in enumerate(parts):
        s, e = shard_bounds(total, r, world)
        out.append(part[: e - s])
    return torch.cat(out, dim=0)


def sample_sharded(sample_fn, total, batch_size, seed=1234, gather=True, device=None):
    """Runs ``sample_fn(n, generator) -> (n, C, H, W) tensor`` over this rank's slice of ``total`` samples in
    batches of ``batch_size`` and returns the gathered (total, C, H, W) tensor (or the local shard).
    Per-rank generator seeds are ``seed + rank`` (SURVEY §8d cfg 2)."""
    rank = dist.get_rank() if dist.is_available() and dist.is_initialized() else 0
    world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
    start, end = shard_bounds(total, rank, world)
    gen = torch.Generator(device=device if device is not None else "cpu").manual_seed(seed + rank)
    outs = []
    for b0 in range(start, end, batch_size):
        n = min(batch_size, end - b0)
        outs.append(sample_fn(n, gen))
    local = torch.cat(outs, dim=0) if outs else None
    if local is None:
        raise ValueError("a rank received an empty shard: total must be >= world size")
    return gather_shards(local, total) if gather else local


_queue_calls = 0


def sample_balanced(sample_fn, total, batch_size, seed=1234, gather=True, device=None):
    """Dynamic variant of `sample_sharded` for boxes whose GPUs do not run at the same speed (under the 1 kW power cap
    the per-GPU step times of an 8-GPU box spread by 4.5 - 8.7 %, profiles/r2j_bench_8gpu_*_per_rank.json; it only pays
    when that spread exceeds one batch, profiles/r2j_generate_static_vs_dynamic_8gpu.txt): the global batches
    ``0 .. ceil(total / batch_size) - 1`` sit in one queue and every rank claims the next index with an atomic add on
    the process group's store, so a faster GPU simply runs more batches.  Batch k always uses generator seed
    ``seed + k``, which makes the result independent of which rank ran it and of the world size.
    Returns the (total, C, H, W) tensor on every rank (one all_reduce over a zero-initialised buffer: every row is
    written by exactly one rank), or with ``gather=False`` the list of (first_row, tensor) this rank produced."""
    global _queue_calls
    multi = dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
    nb = (total + batch_size - 1) // batch_size
    if multi:
        store = dist.distributed_c10d._get_default_store()
        key = f"vdt_b200_batch_queue_{_queue_calls}"
        _queue_calls += 1
        claim = lambda: store.add(key, 1) - 1
    else:
        counter = iter(range(nb + 1))
        claim = lambda: next(counter)
    mine = []
    while True:
        k = claim()
        if k >= nb:
            break
        b0 = k * batch_size
        gen = torch.Generator(device=device if device is not None else "cpu").manual_seed(seed + k)
        mine.append((b0, sample_fn(min(batch_size, total - b0), gen)))
    if not gather:
        return mine
    if multi:
        # every rank learns the sample shape from whoever ran batch 0 (a slow rank may have claimed nothing)
        shape = [tuple(mine[0][1].shape[1:]) + (str(mine[0][1].dtype),)] if mine and mine[0][0] == 0 else [None]
        owner = [None] * dist.get_world_size()
        dist.all_gather_object(owner, shape[0])
        shape = next(o for o in owner if o is not None)
        dtype = getattr(torch, shape[-1].split(".")[-1])
        dev = device if device is not None else (mine[0][1].device if mine else "cpu")
        full = torch.zeros((total,) + tuple(shape[:-1]), dtype=dtype, device=dev)
    else:
        full = torch.zeros((total,) + tuple(mine[0][1].shape[1:]), dtype=mine[0][1].dtype, device=mine[0][1].device)
    for b0, x in mine:
        full[b0: b0 + x.shape[0]] = x
    if multi:
        dist.all_reduce(full)
    return full


def images_to_uint8(x):
    """generate.py:149 on the device: fp32 NCHW samples -> uint8 NHWC pixels, (x * 127.5 + 127.5).clamp(0, 255)
    truncated to uint8 and permuted (0, 2, 3, 1), in one kernel (vdt_images_to_uint8)."""
    import ctypes as C
    from . import _lib
    if x.device.type != "cuda":
        raise RuntimeError("images_to_uint8 runs on CUDA only; there is no CPU fallback")
    x = x.to(torch.float32).contiguous()
    B, Cc, H, W = x.shape
    out = torch.empty((B, H, W, Cc), dtype=torch.uint8, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().vdt_images_to_uint8(_lib.ptr(x), _lib.ptr(out), B, Cc, H * W, _lib.current_stream_ptr()))
    return out


def load_reference_checkpoint(path, use_ema=False):
    """generate.py:33-44: a reference checkpoint is {"model": sd, "ema": {"shadow": sd-like, ...}, ...}; DDP
    checkpoints carry a "module." prefix; a class-conditional model is recognised by its class_embed.* keys.
    Returns (state_dict, use_cfg)."""
    ckpt = torch.load(path, map_location="cpu")
    state_dict = ckpt["ema"]["shadow"] if use_ema else ckpt["model"]
    state_dict = {(k.split(".", 1)[1] if k.startswith("module.") else k): v for k, v in state_dict.items()}
    use_cfg = "class_embed" in {k.split(".")[0] for k in state_dict}
    return state_dict, use_cfg


def main():
    from . import GaussianDiffusion, UNet, load_config, build_from_config  # noqa: F401
    ap = argparse.ArgumentParser()
    ap.add_argument("--config-path", required=True)
    ap.add_argument("--default-config-path", required=True)
    ap.add_argument("--ckpt-path", default=None, help="reference checkpoint (.pt); random init when omitted")
    ap.add_argument("--use-ema", action="store_true")
    ap.add_argument("--use-ddim", action="store_true")
    ap.add_argument("--solver", choices=["ddim", "dpmpp_2m"], default="ddim",
                    help="ddim: the reference's first-order step; dpmpp_2m: DPM-Solver++(2M) on the same time grid "
                         "(needs --use-ddim; fewer --sample-timesteps for a comparable trajectory)")
    ap.add_argument("--sample-timesteps", type=int, default=1024)      # generate.py:25
    ap.add_argument("--uncond", action="store_true")
    ap.add_argument("--w-guide", type=float, default=0.1)              # generate.py:27
    ap.add_argument("--batch-size", type=int, default=128)
    ap.add_argument("--total-size", type=int, default=50000)
    ap.add_argument("--save-path", default=None, help="torch.save of the uint8 NHWC images (rank 0)")
    ap.add_argument("--seed", type=int, default=1234)
    ap.add_argument("--schedule", choices=["static", "dynamic"], default="static",
                    help="static: rank r owns a contiguous slice (seeds seed + rank); dynamic: a shared batch queue, "
                         "batch k seeded seed + k (same images at any world size; faster GPUs run more batches)")
    ap.add_argument("--warmup-batches", type=int, default=0, help="untimed batches before the reported wall-clock")
    ap.add_argument("--label-path", default=None, help="multitag models: torch-saved (N, num_classes) attribute table")
    args = ap.parse_args()
    if args.solver == "dpmpp_2m" and not args.use_ddim:
        ap.error("--solver dpmpp_2m needs --use-ddim (DPM-Solver++(2M) is not defined for ancestral sampling)")
    solver = None if args.solver == "ddim" else args.solver

    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)

    state_dict, use_cfg = None, True
    if args.ckpt_path:
        state_dict, use_cfg = load_reference_checkpoint(args.ckpt_path, args.use_ema)
    config = load_config(args.config_path, args.default_config_path)
    if not args.ckpt_path:
        use_cfg = bool(config.get("conditional", {}).get("use_cfg", False))
    diffusion, model, chw = build_from_config(config, use_cfg, args.w_guide, args.sample_timesteps, args.uncond)
    if state_dict is not None:
        model.load_state_dict(state_dict)
    model = model.to(device).eval()
    num_classes = model.num_classes

    multitags = bool(model.multitags) and num_classes > 0
    tag_rows = None
    if multitags and not args.uncond:
        # generate.py:119-127 draws rows of the dataset's own attribute table; there is no dataset on this path, so the
        # table comes from a file: a (N, num_classes) 0/1 tensor saved with torch.save
        if not args.label_path:
            raise NotImplementedError("class-conditional multitag sampling needs --label-path (a torch-saved (N, "
                                      f"{num_classes}) multi-hot attribute table) or --uncond")
        tag_rows = torch.load(args.label_path, map_location="cpu").float()
        if tag_rows.ndim != 2 or tag_rows.shape[1] != num_classes:
            raise ValueError(f"--label-path must hold a (N, {num_classes}) tensor, got {tuple(tag_rows.shape)}")

    def sample_fn(n, gen):
        noise = torch.randn((n,) + chw, device=device, generator=gen)
        if multitags:
            if args.uncond:
                label = torch.zeros((n, num_classes), dtype=torch.float32, device=device)            # generate.py:123-124
            else:
                pick = torch.randint(len(tag_rows), (n,), device=device, generator=gen).cpu()       # generate.py:126
                label = tag_rows[pick].to(device)
        elif num_classes:
            label = torch.zeros(n, dtype=torch.int64, device=device) if args.uncond else \
                torch.randint(num_classes, (n,), device=device, generator=gen) + 1       # generate.py:132-134
        else:
            label = None
        # every batch draws its own noise seed from this rank's generator: without it the library's on-device stream
        # would replay the same per-step normals for every batch (ancestral sampling, no injected noise)
        seed = int(torch.randint(0, 2 ** 62, (1,), device=device, generator=gen).item())
        return diffusion.p_sample(model, (n,) + chw, noise=noise, label=label, device=device, seed=seed,
                                  use_ddim=args.use_ddim, solver=solver).to(device)

    run = sample_balanced if args.schedule == "dynamic" else sample_sharded
    calls = [0]

    def counted(n, gen):
        calls[0] += 1
        return sample_fn(n, gen)
    if args.warmup_batches:                                   # graph capture and workspace allocation outside the clock
        for _ in range(args.warmup_batches):
            sample_fn(args.batch_size, torch.Generator(device=device).manual_seed(0))
    torch.cuda.synchronize()
    if dist.is_initialized():
        dist.barrier()
    t0 = time.perf_counter()
    x = run(counted, args.total_size, args.batch_size, seed=args.seed, device=device)
    torch.cuda.synchronize()
    seconds = time.perf_counter() - t0
    per_rank = [calls[0]]
    if dist.is_initialized():
        per_rank = [None] * world
        dist.all_gather_object(per_rank, calls[0])
    if not dist.is_initialized() or dist.get_rank() == 0:
        print(json.dumps({"schedule": args.schedule, "images": args.total_size, "seconds": seconds,
                          "images_per_s": args.total_size / seconds, "n_gpus": world, "batches_per_rank": per_rank}),
              file=sys.stderr, flush=True)
    if (not dist.is_initialized() or dist.get_rank() == 0) and args.save_path:
        torch.save(images_to_uint8(x).cpu(), args.save_path)      # generate.py:149 (the PNG encoding itself is I/O, out of scope)
    if dist.is_initialized():
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
