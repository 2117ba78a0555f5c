"""Time `PGHIStream` on a B200.

    python tools/bench_pghi_stream.py [--out results/bench_pghi_stream.json]

* Real-time use: B = 1, 1024/256, float32, one frame per push over 10 s of frames at 22.05 kHz, with a device
  synchronise after every push as a consumer that plays the samples would.  Median and p99 host time per push, and the
  device time per push (CUDA events around the whole run, divided by the pushes).
* Throughput: the cfg2 shape (B = 512 ten-second clips, 1024/256, float32) pushed 32 frames at a time, against offline
  `pghi` followed by the ISTFT (`torch.istft` of its output is not used: the library's ISTFT plan is), both in the
  same run after warm-up.
The card's name and power limit are read in the same run."""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from bench_pghi import card, harmonic  # noqa: E402
from spectrogram_inversion_b200 import PGHIStream, pghi  # noqa: E402
from spectrogram_inversion_b200.engine import StftPlan  # noqa: E402
from spectrogram_inversion_b200.stft_args import args_helper  # noqa: E402


def stream_all(mag, k, w, hop):
    st = PGHIStream(hop_length=hop, window=w)
    for t in range(0, mag.shape[-1], k):
        st.push(mag[..., t:t + k])
    return st.flush()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    sr, n_fft, hop = 22050, 1024, 256
    w = torch.hann_window(n_fft, device="cuda")
    res = {"card": card()}

    # real time: one frame per push, synchronised
    x1 = harmonic(1, 10 * sr, sr, seed=1).float()
    mag1 = torch.stft(x1, n_fft, hop, window=w, return_complex=True).abs()[0].contiguous()
    T1 = mag1.shape[-1]
    stream_all(mag1[:, :64], 1, w, hop)                          # warm-up: plans, modules
    torch.cuda.synchronize()
    st = PGHIStream(hop_length=hop, window=w)
    host = []
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for t in range(T1):
        t0 = time.perf_counter()
        st.push(mag1[:, t:t + 1])
        torch.cuda.synchronize()
        host.append(time.perf_counter() - t0)
    b.record()
    b.synchronize()
    st.flush()
    host.sort()
    res["realtime"] = {"frames": T1, "host_ms_median": 1e3 * host[len(host) // 2],
                       "host_ms_p99": 1e3 * host[int(0.99 * (len(host) - 1))],
                       "device_ms_per_push": a.elapsed_time(b) / T1, "hop_ms_at_22050": 1e3 * hop / sr}

    # throughput at the cfg2 shape: stream (32 frames per push) against offline pghi + ISTFT
    B = 512
    x = harmonic(B, 10 * sr, sr, seed=2).float()
    mag = torch.stft(x, n_fft, hop, window=w, return_complex=True).abs().contiguous()
    del x
    T = mag.shape[-1]
    plan = StftPlan(args_helper(mag, window=w, hop_length=hop), T, B, torch.float32, mag.device)

    def offline():
        return plan.istft(plan.pack(pghi(mag, window=w, hop_length=hop)))

    def streamed():
        return stream_all(mag, 32, w, hop)

    times = {"offline_ms": [], "stream_ms": []}
    offline(), streamed()
    for _ in range(3):                                           # alternate the two
        for key, fn in (("offline_ms", offline), ("stream_ms", streamed)):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            times[key].append(e0.elapsed_time(e1))
    res["cfg2"] = {"B": B, "T": T, "frames_per_push": 32, **{k: sorted(v)[1] for k, v in times.items()},
                   "all": times}
    print(json.dumps(res, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
