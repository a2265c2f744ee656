#!/usr/bin/env python
"""The shipped benchmark's training driver (src/benchmark/train.py:356-509) on roomslam_b200: raw trace files and
collider files in, BiLSTM + query decoder trained with the Hungarian set loss, evaluated every epoch, checkpoints in the
upstream layout (model_state_dict / optimizer_state_dict / val_loss / metrics / config).

    python train_benchmark.py --data_dir dataset/train --val_dir dataset/val --epochs 200
    python train_benchmark.py --d_model 256 --num_queries 80 --precision bf16     # build_model's defaults, tensor cores

--precision bf16 runs the LSTM recurrence on tensor cores (bf16 operands, fp32 accumulation and cell state); it exists for
--d_model 256 only and is about 6x faster per training step there (DESIGN.md section 7.2).  fp32 is the default and the
exact path.  The precision is recorded in config.json; checkpoints load into either precision.

Everything between the JSON files and the optimizer runs on the GPU: features (rs_trace_features), model, matching,
loss, metrics.  The JSON parsing and the upstream augmentation pipeline (dataloader.py:340-392) are host-side and out of
this library's scope; this driver uses each recorded trace once per epoch, unaugmented."""
import argparse
import glob
import json
import os

import torch

from roomslam_b200 import data, preprocess
from roomslam_b200.evaluation import MetricAccumulator
from roomslam_b200.lstm_model import build_model
from roomslam_b200.set_loss import SetCriterion
from roomslam_b200.train_utils import seed_everything

WEIGHTS = {"class_loss": 2.0, "l1_loss": 5.0, "giou_loss": 2.0}                 # train.py:433-437


def load_split(split_dir: str, max_colliders: int = 50):
    """One sample per ``*_data_*.json`` trace file, all sharing the split's ``colliders.json`` (dataloader.py:97-150)."""
    files = sorted(glob.glob(os.path.join(split_dir, "*_data_*.json")))
    if not files:
        raise ValueError(f"no trace files (*_data_*.json) in {split_dir}")
    tgt = data.load_colliders(os.path.join(split_dir, "colliders.json"), max_colliders)
    return [data.load_trace_points(f) for f in files], tgt


def batches(points, tgt, batch_size, max_len, shuffle, gen=None):
    order = torch.randperm(len(points), generator=gen).tolist() if shuffle else list(range(len(points)))
    for s in range(0, len(order), batch_size):
        idx = order[s:s + batch_size]
        feats = preprocess.trace_features([points[i] for i in idx], max_len=max_len)
        targets = {k: v.unsqueeze(0).expand(len(idx), *v.shape).contiguous().cuda() for k, v in tgt.items()}
        yield feats["traces"], feats["trace_mask"], targets


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--data_dir", default="dataset/train")
    ap.add_argument("--val_dir", default="dataset/val")
    ap.add_argument("--save_dir", default="checkpoints")
    ap.add_argument("--epochs", type=int, default=200)
    ap.add_argument("--batch_size", type=int, default=20)
    ap.add_argument("--lr", type=float, default=2e-4)
    ap.add_argument("--weight_decay", type=float, default=1e-4)
    ap.add_argument("--d_model", type=int, default=128)
    ap.add_argument("--precision", choices=("fp32", "bf16"), default="fp32",
                    help="LSTM recurrence: fp32, or bf16 on tensor cores (d_model 256 only)")
    ap.add_argument("--num_queries", type=int, default=30)
    ap.add_argument("--max_trace_len", type=int, default=3000)
    ap.add_argument("--iou_thresh", type=float, default=0.5)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--deterministic", action="store_true",
                    help="seed everything and turn on torch.use_deterministic_algorithms: bit-identical reruns")
    args = ap.parse_args()
    config = dict(vars(args), model_type="lstm")
    os.makedirs(args.save_dir, exist_ok=True)
    json.dump(config, open(os.path.join(args.save_dir, "config.json"), "w"), indent=2)
    if args.deterministic:
        seed_everything(args.seed)
    torch.manual_seed(args.seed)
    gen = torch.Generator().manual_seed(args.seed)
    train_pts, train_tgt = load_split(args.data_dir)
    val_pts, val_tgt = load_split(args.val_dir)
    model = build_model(num_queries=args.num_queries, d_model=args.d_model, model_type="lstm", precision=args.precision).cuda()
    criterion = SetCriterion(WEIGHTS)
    optimizer = torch.optim.AdamW(model.parameters(), lr=args.lr, weight_decay=args.weight_decay)
    scheduler = torch.optim.lr_scheduler.ReduceLROnPlateau(optimizer, mode="min", factor=0.5, patience=5, threshold=1e-3,
                                                           cooldown=1, min_lr=1e-6)                 # train.py:454-458
    best = float("inf")
    for epoch in range(args.epochs):
        model.train()
        total, n = 0.0, 0
        for x, mask, targets in batches(train_pts, train_tgt, args.batch_size, args.max_trace_len, True, gen):
            optimizer.zero_grad()
            losses = criterion(model(x, mask), targets)
            losses["total_loss"].backward()
            torch.nn.utils.clip_grad_norm_(model.parameters(), 1.0)                                 # train.py:220
            optimizer.step()
            total += float(losses["total_loss"].detach())
            n += 1
        model.eval()
        acc, vtotal, vn = MetricAccumulator("cuda", args.iou_thresh), 0.0, 0
        with torch.no_grad():
            for x, mask, targets in batches(val_pts, val_tgt, args.batch_size, args.max_trace_len, False):
                out = model(x, mask)
                vtotal += float(criterion(out, targets)["total_loss"])
                vn += 1
                acc.update(out, targets)
        val_loss, metrics = vtotal / max(vn, 1), acc.compute()
        scheduler.step(val_loss)
        print(f"Epoch {epoch}: Train {total / max(n, 1):.4f} | Val {val_loss:.4f} | mIoU={metrics['mIoU']:.3f} "
              f"P={metrics['precision']:.3f} R={metrics['recall']:.3f} F1={metrics['f1']:.3f} ClsAcc={metrics['cls_acc']:.3f} | "
              f"LR={optimizer.param_groups[0]['lr']:.6f}")
        if val_loss < best:
            best = val_loss
            torch.save({"epoch": epoch, "model_state_dict": model.state_dict(), "optimizer_state_dict": optimizer.state_dict(),
                        "val_loss": val_loss, "metrics": metrics, "config": config}, os.path.join(args.save_dir, "best_model.pth"))
        if (epoch + 1) % 10 == 0:
            torch.save({"epoch": epoch, "model_state_dict": model.state_dict(), "optimizer_state_dict": optimizer.state_dict(),
                        "train_loss": total / max(n, 1)}, os.path.join(args.save_dir, f"checkpoint_epoch_{epoch}.pth"))
    print("Training completed!")


if __name__ == "__main__":
    main()
