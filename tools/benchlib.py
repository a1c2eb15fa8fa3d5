"""Measurement helpers shared by the tools/*_bench.py scripts (imported from the script's directory)."""
import statistics
import subprocess

import torch

HBM_BYTES_PER_S = 7.7e12                      # B200 HBM3e bandwidth of one GPU, NVIDIA's HGX B200 data sheet


def power_limit():
    """The current card's power limit as nvidia-smi prints it, or "unknown"."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader",
                              f"--id={torch.cuda.current_device()}"], capture_output=True, text=True, timeout=30)
        return out.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def event_ms(fn, reps=1):
    """Milliseconds per call of fn, `reps` calls between one CUDA-event pair on a synchronised device."""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def spread(xs, digits=3):
    return {"median": round(statistics.median(xs), digits), "min": round(min(xs), digits),
            "max": round(max(xs), digits)}
