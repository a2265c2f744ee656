#!/usr/bin/env python
"""Thin equivalent of the upstream README's train.py (README.md:64-74; the script itself is absent upstream).

    python train.py --create_sample_data
    python train.py --data_dir data/sample --epochs 50
"""
import argparse
import os

import torch

from roomslam_b200 import RoomSLAM, data
from roomslam_b200.train_utils import FlatParams, FusedAdamW, seed_everything

# README.md:147-157
BATCH_SIZE, LEARNING_RATE, HIDDEN_SIZE, SEQUENCE_LENGTH, MAX_OBJECTS, NUM_EPOCHS = 32, 1e-3, 128, 500, 10, 100


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--data_dir", default="data/sample")
    ap.add_argument("--epochs", type=int, default=NUM_EPOCHS)
    ap.add_argument("--batch_size", type=int, default=BATCH_SIZE)
    ap.add_argument("--lr", type=float, default=LEARNING_RATE)
    ap.add_argument("--precision", default="fp32", choices=["fp32", "bf16", "auto"])
    ap.add_argument("--create_sample_data", action="store_true")
    ap.add_argument("--checkpoint_dir", default="checkpoints")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--deterministic", action="store_true",
                    help="seed everything and turn on torch.use_deterministic_algorithms: bit-identical reruns")
    args = ap.parse_args()
    if args.create_sample_data:
        data.create_sample_data(args.data_dir, seq_len=SEQUENCE_LENGTH, max_objects=MAX_OBJECTS, seed=args.seed)
        print(f"wrote sample data to {args.data_dir}")
        return
    if args.deterministic:
        seed_everything(args.seed)
    torch.manual_seed(args.seed)
    x, tgt = data.load_dir(args.data_dir, SEQUENCE_LENGTH, MAX_OBJECTS)
    n_val = max(1, len(x) // 10)
    model = RoomSLAM(hidden_size=HIDDEN_SIZE, max_objects=MAX_OBJECTS, precision=args.precision).cuda()
    flat = FlatParams(model)
    opt = FusedAdamW(flat, lr=args.lr, max_grad_norm=1.0)
    os.makedirs(args.checkpoint_dir, exist_ok=True)
    best = float("inf")
    for epoch in range(args.epochs):
        model.train()
        perm = torch.randperm(len(x) - n_val) + n_val
        total, batches = 0.0, 0
        for s in range(0, len(perm), args.batch_size):
            idx = perm[s:s + args.batch_size]
            xb = x[idx].cuda(non_blocking=True)
            tb = {k: v[idx].cuda(non_blocking=True) for k, v in tgt.items()}
            flat.zero_grad()
            loss = model.compute_loss(model(xb), tb)
            loss["total"].backward()
            opt.step()
            total += loss["total"].item()
            batches += 1
        model.eval()
        with torch.no_grad():
            vl = model.compute_loss(model(x[:n_val].cuda()), {k: v[:n_val].cuda() for k, v in tgt.items()})["total"].item()
        print(f"epoch {epoch + 1}/{args.epochs}  train {total / max(batches, 1):.4f}  val {vl:.4f}")
        if vl < best:
            best = vl
            torch.save({"epoch": epoch, "model_state_dict": model.state_dict(), "val_loss": vl,
                        "config": vars(args)}, os.path.join(args.checkpoint_dir, "best_model.pth"))


if __name__ == "__main__":
    main()
