#!/usr/bin/env python3
"""Command-line separation of one audio file -- the reference's inference/separate.py on the B200 path.

    python -m mss_tf_locoformer_b200.separate --input song.wav --checkpoint model.pt [--config cfg.yaml]
        [--output_dir ./separated] [--device cuda] [--sample_rate 44100] [--seed 42]
        [--segment 6.0] [--batch 8] [--precision bf16|fp32|tf32] [--overlap 0.5] [--stereo]

Same flags, same checkpoint / YAML handling, same mono down-mix, same stereo duplication and peak normalisation
of the outputs as /root/reference/inference/separate.py:28-193 (`load_model` :79-116, `separate_audio` :119-169) and
utils/audio.py:14-66, by default.  Things that differ on purpose:

* `--segment S` (default 6 s) runs the track as overlapping S-second segments cross-faded at 50 % overlap
  (segments.separate_track) instead of the reference's single whole-track forward, which needs memory quadratic in the
  track length (MEMORY_ANALYSIS.md:7-11).  `--segment 0` restores the reference behaviour (one forward over the track).
  Under `torchrun --nproc-per-node N` the segments are sharded over the N GPUs and rank 0 writes the files.
* `--overlap F` (default 0.5, in (0, 1)): consecutive segments overlap by the fraction F of the segment (hop =
  max(1, round(L * (1 - F)))).  The number of forwards grows as 1 / (1 - F): 0.75 runs twice as many as 0.5.
* `--stereo` separates every channel of the input on its own (the model is mono) and writes [C, T] stems, peak-normalised
  over all channels of a stem so the balance between them is kept.  Without it the input is down-mixed to mono and each
  stem duplicated to two channels, as the reference does; a mono input gives the same output either way.
  `--segment 0` ignores `--overlap` and `--stereo`: one forward over the down-mixed track, as the reference.
* audio I/O uses scipy.io.wavfile (WAV only): torchaudio's codecs are not installed in this image.  Resampling uses
  scipy.signal.resample_poly, not torchaudio's windowed-sinc kernel.
"""
import argparse
import os
from math import gcd
from pathlib import Path
from typing import Dict, Tuple

import numpy as np
import torch

from .models import TFLocoformerMSS
from .segments import separate_track


def parse_args(argv=None):
    p = argparse.ArgumentParser(description="Separate music sources using TF-Locoformer (B200-native path)")
    p.add_argument("--input", type=str, required=True, help="Input audio file path (WAV)")
    p.add_argument("--output_dir", type=str, default="./separated", help="Output directory for separated sources")
    p.add_argument("--checkpoint", type=str, required=True, help="Path to model checkpoint")
    p.add_argument("--config", type=str, default=None, help="Path to model config file (optional)")
    p.add_argument("--device", type=str, default="cuda", help="Device to use (a CUDA device: there is no CPU path)")
    p.add_argument("--sample_rate", type=int, default=44100, help="Sample rate for processing")
    p.add_argument("--seed", type=int, default=42, help="Random seed")
    p.add_argument("--segment", type=float, default=6.0, help="Segment length in seconds (0 = whole track in one forward)")
    p.add_argument("--batch", type=int, default=8, help="Segments per forward")
    p.add_argument("--precision", type=str, default="bf16", choices=["bf16", "fp32", "tf32"])
    p.add_argument("--overlap", type=_overlap, default=0.5, help="Fraction of a segment shared with the next, in (0, 1)")
    p.add_argument("--stereo", action="store_true", help="Separate every input channel and write multichannel stems")
    return p.parse_args(argv)


def _overlap(text: str) -> float:
    value = float(text)
    if not 0.0 < value < 1.0:
        raise argparse.ArgumentTypeError(f"overlap must be in (0, 1) (got {text})")
    return value


# ---- utils/audio.py:14-66 ------------------------------------------------------------------------------------------
def load_audio(path: str, sample_rate: int = 44100, mono: bool = False) -> Tuple[torch.Tensor, int]:
    """-> audio [C, T] float32 in [-1, 1], sample rate (resampled to `sample_rate` if the file differs)."""
    from scipy.io import wavfile
    sr, data = wavfile.read(path)
    if data.dtype == np.int16:
        x = data.astype(np.float32) / 32768.0
    elif data.dtype == np.int32:
        x = data.astype(np.float32) / 2147483648.0
    elif data.dtype == np.uint8:
        x = (data.astype(np.float32) - 128.0) / 128.0
    else:
        x = data.astype(np.float32)
    if x.ndim == 1:
        x = x[:, None]
    if sr != sample_rate:
        from scipy.signal import resample_poly
        g = gcd(int(sr), int(sample_rate))
        x = resample_poly(x, sample_rate // g, sr // g, axis=0).astype(np.float32)
    audio = torch.from_numpy(np.ascontiguousarray(x.T))
    if mono and audio.shape[0] > 1:
        audio = audio.mean(dim=0, keepdim=True)
    return audio, sample_rate


def save_audio(audio: torch.Tensor, path: str, sample_rate: int = 44100, normalize: bool = True) -> None:
    """audio [C, T] -> 32-bit float WAV; `normalize` divides by the peak as the reference does (utils/audio.py:58-62)."""
    from scipy.io import wavfile
    if normalize:
        max_val = audio.abs().max()
        if max_val > 0:
            audio = audio / max_val
    wavfile.write(path, sample_rate, np.ascontiguousarray(audio.cpu().to(torch.float32).numpy().T))


# ---- inference/separate.py:79-116 ----------------------------------------------------------------------------------
def load_model(checkpoint_path: str, config_path=None, device: str = "cuda") -> TFLocoformerMSS:
    print(f"Loading checkpoint from {checkpoint_path}")
    checkpoint = torch.load(checkpoint_path, map_location="cpu")
    if config_path is not None:
        import yaml
        with open(config_path, "r") as f:
            config = yaml.safe_load(f)
        model_config = dict(config.get("model", {}))
    else:
        model_config = {}
    model = TFLocoformerMSS(**model_config)
    state = checkpoint["model_state_dict"] if "model_state_dict" in checkpoint else checkpoint
    model.load_state_dict(state)
    model = model.to(device)
    model.eval()
    print("Model loaded successfully")
    return model


def downmix(audio: torch.Tensor) -> torch.Tensor:
    """[C, T] -> [T]: stereo is averaged to mono as the reference does (inference/separate.py:135-139)."""
    return audio.mean(dim=0) if audio.shape[0] > 1 else audio[0]


def to_stereo(source_audio: torch.Tensor) -> torch.Tensor:
    """[T] or [1, T] -> [2, T] by duplicating the channel (inference/separate.py:158-162)."""
    if source_audio.ndim == 1:
        return source_audio.unsqueeze(0).repeat(2, 1)
    if source_audio.shape[0] == 1:
        return source_audio.repeat(2, 1)
    return source_audio


def separate_audio(model, audio_path: str, output_dir: str, device: str = "cuda", sample_rate: int = 44100,
                   segment: float = 6.0, batch: int = 8, rank: int = 0, overlap: float = 0.5,
                   stereo: bool = False) -> Dict[str, str]:
    """inference/separate.py:119-169 with segment-wise inference; returns {source: written path} (rank 0 writes).
    ``stereo``: separate each channel of a multichannel input and write [C, T] stems (``segment`` > 0 only)."""
    print(f"\nProcessing: {audio_path}")
    audio, sr = load_audio(audio_path, sample_rate=sample_rate, mono=False)
    print(f"Loaded audio: {audio.shape}, sample rate: {sr}")
    channels = stereo and segment > 0 and audio.shape[0] > 1
    track = audio.to(device) if channels else downmix(audio).to(device)     # [C, T] or [T]
    print("Separating sources...")
    with torch.no_grad():
        seg_len = int(round(segment * sample_rate)) // 2 * 2
        if segment > 0 and track.shape[-1] > seg_len:
            separated = separate_track(model, track, seg_len=seg_len, batch=batch, overlap=overlap)
        elif channels:
            separated = model(track, return_time_domain=True)
        else:
            separated = {k: v[0] for k, v in model(track[None], return_time_domain=True).items()}
    written = {}
    if rank == 0:
        os.makedirs(output_dir, exist_ok=True)
        input_name = Path(audio_path).stem
        for source_name, source_audio in separated.items():
            output_path = os.path.join(output_dir, f"{input_name}_{source_name}.wav")
            save_audio(to_stereo(source_audio.cpu()), output_path, sample_rate=sample_rate, normalize=True)
            print(f"Saved {source_name}: {output_path}")
            written[source_name] = output_path
        print(f"\nSeparation complete! Results saved to {output_dir}")
    return written


def main(argv=None):
    args = parse_args(argv)
    torch.manual_seed(args.seed)
    np.random.seed(args.seed)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    device = args.device
    if world > 1:
        import torch.distributed as dist
        local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(local)
        device = f"cuda:{local}"
        dist.init_process_group("nccl", device_id=torch.device(device))
    try:
        model = load_model(args.checkpoint, config_path=args.config, device=device)
        model.precision = args.precision
        separate_audio(model, args.input, args.output_dir, device=device, sample_rate=args.sample_rate,
                       segment=args.segment, batch=args.batch, rank=rank, overlap=args.overlap, stereo=args.stereo)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
