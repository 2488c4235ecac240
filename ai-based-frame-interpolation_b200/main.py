#!/usr/bin/env python
"""CLI with the reference main.py's sub-commands and flags (reference main.py:40-72): train / infer / video / serve /
info. `infer` and `video` drive model.inference.FrameInterpolator, `train` drives model.train.main (the B200
training step)."""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def _scene_threshold(text):
    from model.scene import check_threshold
    try:
        return check_threshold(text)
    except ValueError as e:
        raise argparse.ArgumentTypeError(str(e)) from None


def _crop_size(text):
    from model.train import crop_size
    return crop_size(text)


def _frame_rate(text):
    from model.timing import parse_rate
    try:
        return parse_rate(text)
    except ValueError as e:
        raise argparse.ArgumentTypeError(str(e)) from None


class _TypedFactor(argparse.Action):
    """Stores --factor and notes that it was given; argparse calls it for abbreviations (--fac 3) as well."""

    def __call__(self, parser, namespace, values, option_string=None):
        setattr(namespace, self.dest, values)
        namespace.factor_typed = True


def build_parser():
    p = argparse.ArgumentParser(description="AI-Based Frame Interpolation (B200-native path)")
    sub = p.add_subparsers(dest="command", help="Available commands")
    # flags, defaults and required-ness as reference main.py:40-72; --frame-cache, --color, --crop, --gpus,
    # --scene-threshold and --fps are the only additions
    t = sub.add_parser("train", help="Train the frame interpolation model")
    t.add_argument("--data-dir", required=True, help="Directory containing training data")
    t.add_argument("--epochs", type=int, default=100, help="Number of training epochs")
    t.add_argument("--batch-size", type=int, default=8, help="Training batch size")
    t.add_argument("--lr", type=float, default=0.001, help="Learning rate")
    t.add_argument("--device", default="auto", help="Device to use (cuda/auto)")
    t.add_argument("--frame-cache", action="store_true",
                   help="Decode every frame once into GPU memory and build the batches there (default: off)")
    t.add_argument("--color", action="store_true",
                   help="Train the colour model UNet(6, 3) on BGR frames instead of the grey one (default: off)")
    t.add_argument("--crop", type=_crop_size, default=None, metavar="S",
                   help="Train on random S x S windows (S a multiple of 16) of frames at their native size, mirrored "
                        "and with the input pair swapped at random, instead of resizing to 256x256 (default: off)")
    i = sub.add_parser("infer", help="Run inference on two frames")
    i.add_argument("--frame1", required=True, help="Path to first frame")
    i.add_argument("--frame2", required=True, help="Path to second frame")
    i.add_argument("--output", required=True, help="Output path for interpolated frame")
    i.add_argument("--model", default="best_model.pth", help="Path to trained model")
    i.add_argument("--device", default="auto", help="Device to use (cuda/auto)")
    v = sub.add_parser("video", help="Interpolate frames in a video")
    v.add_argument("--input", required=True, help="Input video path")
    v.add_argument("--output", required=True, help="Output video path")
    v.add_argument("--factor", type=int, default=2, action=_TypedFactor, help="Interpolation factor")
    v.add_argument("--model", default="best_model.pth", help="Path to trained model")
    v.add_argument("--device", default="auto", help="Device to use (cuda/auto)")
    v.add_argument("--gpus", type=int, default=None,
                   help="Shard the frame pairs over this many GPUs of the box (default: $FI_GPUS, else 1)")
    v.add_argument("--scene-threshold", type=_scene_threshold, default=None, metavar="T",
                   help="Detect scene cuts (score in (0, 100], try 10) and repeat the frame before a cut instead of "
                        "blending two shots (default: off)")
    v.add_argument("--fps", type=_frame_rate, default=None, metavar="RATE",
                   help="Convert to this output frame rate, e.g. 60, 59.94 or 60000/1001 (instead of --factor)")
    s = sub.add_parser("serve", help="Start the web API server")
    s.add_argument("--host", default="0.0.0.0", help="Host to bind to")
    s.add_argument("--port", type=int, default=8000, help="Port to bind to")
    s.add_argument("--reload", action="store_true", help="Enable auto-reload for development")
    info = sub.add_parser("info", help="Show model information")
    info.add_argument("--model", default="best_model.pth", help="Path to model file")
    return p


def main(argv=None):
    parser = build_parser()
    args = parser.parse_args(argv)
    if args.command == "video" and args.fps is not None and getattr(args, "factor_typed", False):
        parser.error("video: --fps and --factor exclude each other (--fps sets the output rate)")
    if not args.command:
        build_parser().print_help()
        return 0
    device = getattr(args, "device", "auto")  # `serve` / `info` have no --device (the reference crashes here)
    device = "cuda" if device == "auto" else device
    try:
        if args.command == "train":
            from model.train import main as train_main
            # reference main.py:92 forwards only --data-dir / --epochs, so its training always runs train.py's own
            # defaults (Adam lr 1e-4, batch 8) whatever --lr / --batch-size say; here flags the user typed ARE forwarded
            # and untouched ones keep train.py's defaults
            fwd = ["--data-dir", args.data_dir, "--epochs", str(args.epochs), "--device", args.device]
            typed = {a.split("=")[0] for a in (sys.argv[1:] if argv is None else argv)}
            if "--lr" in typed:
                fwd += ["--lr", str(args.lr)]
            if "--batch-size" in typed:
                fwd += ["--batch-size", str(args.batch_size)]
            if args.frame_cache:
                fwd.append("--frame-cache")
            if args.color:
                fwd.append("--color")
            if args.crop is not None:
                fwd += ["--crop", str(args.crop)]
            train_main(fwd)
            return 0
        if args.command == "infer":
            import cv2
            from model.inference import FrameInterpolator
            interpolator = FrameInterpolator(args.model, device)
            frame1, frame2 = cv2.imread(args.frame1), cv2.imread(args.frame2)
            if frame1 is None or frame2 is None:
                print("Error: Could not read input frames")
                return 1
            print("Generating intermediate frame...")
            cv2.imwrite(args.output, interpolator.interpolate_frames(frame1, frame2))
            print(f"Interpolated frame saved to: {args.output}")
        elif args.command == "video":
            from model.inference import FrameInterpolator
            interpolator = FrameInterpolator(args.model, device, gpus=args.gpus, scene_threshold=args.scene_threshold)
            if args.fps is None:
                print(f"Interpolating video: {args.input}\nOutput: {args.output}\nFactor: {args.factor}x")
                n = interpolator.interpolate_video(args.input, args.output, args.factor)
            else:
                print(f"Interpolating video: {args.input}\nOutput: {args.output}\nFrame rate: {args.fps} fps")
                n = interpolator.interpolate_video(args.input, args.output, fps=args.fps)
            print(f"Video interpolation completed! ({n} frames written)")
            if args.scene_threshold is not None:
                print(f"Scene cuts found: {len(interpolator.last_scene_cuts)} (threshold {args.scene_threshold:g})")
        elif args.command == "serve":
            import uvicorn
            print(f"Starting API server on {args.host}:{args.port}")
            uvicorn.run("api.app:app", host=args.host, port=args.port, reload=args.reload)
        elif args.command == "info":
            # reference main.py:139-158: checkpoint summary, then the architecture's parameter counts
            if not os.path.exists(args.model):
                print(f"Model file not found: {args.model}")
                return 0
            import torch
            checkpoint = torch.load(args.model, map_location="cpu")
            meta = checkpoint if isinstance(checkpoint, dict) and "model_state_dict" in checkpoint else {}

            def fmt(v):  # the reference crashes formatting 'Unknown' with :.6f; print it as is
                return f"{v:.6f}" if isinstance(v, (int, float)) else str(v)

            print(f"Model: {args.model}")
            print(f"Epoch: {meta.get('epoch', 'Unknown')}")
            print(f"Training Loss: {fmt(meta.get('train_loss', 'Unknown'))}")
            print(f"Validation Loss: {fmt(meta.get('val_loss', 'Unknown'))}")
            from model.unet import architecture_name, model_from_state_dict
            model, _ = model_from_state_dict(meta.get("model_state_dict", checkpoint))
            total = sum(p.numel() for p in model.parameters())
            trainable = sum(p.numel() for p in model.parameters() if p.requires_grad)
            print(f"Architecture: {architecture_name(model)}")
            print(f"Total Parameters: {total:,}")
            print(f"Trainable Parameters: {trainable:,}")
    except ImportError as e:
        print(f"Import error: {e}")
        return 1
    except Exception as e:
        print(f"Error: {e}")
        return 1
    return 0


if __name__ == "__main__":
    sys.exit(main())
