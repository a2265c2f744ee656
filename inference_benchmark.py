#!/usr/bin/env python
"""The shipped benchmark's inference CLI (src/benchmark/inference.py:8-21,199-330) on roomslam_b200: checkpoint + trace
JSON in, collider JSON out (same keys: colliders[] with type / label / confidence / center / size / radius / height, and
metadata).  Features, model, confidence filter and per-class NMS all run on the GPU.

    python inference_benchmark.py --checkpoint checkpoints/best_model.pth --input trace.json --output colliders.json
"""
import argparse
import json

import torch

from roomslam_b200 import preprocess
from roomslam_b200.evaluation import post_process_predictions
from roomslam_b200.lstm_model import build_model


def load_model(checkpoint_path: str, device="cuda", precision: str = "fp32"):
    """inference.py:8-21: the checkpoint's own config picks the architecture (defaults: 50 queries, d_model 256).
    precision "bf16" runs the LSTM recurrence on tensor cores (d_model 256); checkpoints load into either precision."""
    ck = torch.load(checkpoint_path, map_location="cpu", weights_only=False)
    config = ck.get("config", {})
    model = build_model(num_queries=config.get("num_queries", 50), d_model=config.get("d_model", 256),
                        model_type=config.get("model_type", "lstm"), precision=precision)
    model.load_state_dict(ck["model_state_dict"], strict=True)
    return model.to(device).eval(), config


def predict(model, traces_file: str, confidence_threshold: float = 0.7, nms_threshold: float = 0.3, max_len: int = 3000):
    """inference.py:199-274.  The trace file is a list of {timestamp, x, y, z} (or a dict holding it under 'traces' /
    'trajectory')."""
    data = json.load(open(traces_file))
    pts = data if isinstance(data, list) else data.get("traces", data.get("trajectory", []))
    if len(pts) == 0:
        print("Warning: No traces found in file")
        return []
    raw = torch.tensor([[p["x"], p["y"], p["z"], p["timestamp"]] for p in pts], dtype=torch.float32)
    batch = preprocess.trace_features([raw], max_len=max_len, sort=True)          # the reference always sorts by time
    with torch.no_grad():
        out = model(batch["traces"], batch["trace_mask"])
    return post_process_predictions(out["pred_boxes"][0], out["pred_classes"][0], confidence_threshold, nms_threshold)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--checkpoint", required=True, help="Path to model checkpoint")
    ap.add_argument("--input", required=True, help="Input trace file (JSON)")
    ap.add_argument("--output", default=None, help="Output file for predictions")
    ap.add_argument("--threshold", type=float, default=0.7, help="Confidence threshold (default: 0.7)")
    ap.add_argument("--nms", type=float, default=0.3, help="NMS IoU threshold (default: 0.3)")
    ap.add_argument("--precision", choices=("fp32", "bf16"), default="fp32",
                    help="LSTM recurrence: fp32, or bf16 on tensor cores (d_model 256 checkpoints only)")
    args = ap.parse_args()
    print(f"Loading model from {args.checkpoint}")
    model, _ = load_model(args.checkpoint, precision=args.precision)
    print(f"Processing {args.input}")
    preds = predict(model, args.input, args.threshold, args.nms)
    print(f"\nFound {len(preds)} colliders:")
    for i, p in enumerate(preds):
        print(f"  {i + 1}. {p['label']} at ({p['center']['x']:.2f}, {p['center']['y']:.2f}, {p['center']['z']:.2f}) "
              f"- confidence: {p['confidence']:.3f}")
    if args.output:
        json.dump({"colliders": preds, "metadata": {"num_colliders": len(preds), "confidence_threshold": args.threshold,
                                                    "nms_threshold": args.nms}}, open(args.output, "w"), indent=2)
        print(f"\nResults saved to {args.output}")


if __name__ == "__main__":
    main()
