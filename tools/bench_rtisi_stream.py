"""Streaming RTISI-LA (RTISIStream) at the cfg3 shape: n_fft 1024 / hop 256, look_ahead 3, 25 inner iterations,
938 frames = 10 s at 24 kHz, for B in {1, 16, 256} and chunks of {1, 4, 16, 64} frames.

    python tools/bench_rtisi_stream.py [--out result.json]

Per (B, chunk), after a warm-up stream of the same shapes:
  gpu_us     GPU time per push: CUDA events recorded around each push of a stream run without host synchronisation
             (the first push, which has no look-ahead to wait for, and the flush are left out);
  host_us    enqueue-to-completion per push: host clock around push() + synchronise;
  rtf        real-time factor per stream: audio of one chunk (chunk * hop / 24000 s) over gpu_us;
  stream_ms  the whole 938 frames pushed chunk by chunk and flushed, events around all of it;
  whole_ms   RTISI_LA on all 938 frames at once, same B.
The card's name and power limit are read in the same run (nvidia-smi query only)."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import spectrogram_inversion_b200 as S  # noqa: E402

N_FFT, HOP, LA, ITERS, SR, T = 1024, 256, 3, 25, 24000, 938


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as ex:            # the name from torch at least
        return f"{torch.cuda.get_device_name(0)} (power limit not read: {ex})"


def stream_events(mag, chunk, kw):
    """Push all frames without synchronising; per-push event pairs and the total."""
    s = S.RTISIStream(look_ahead=LA, max_iter=ITERS, **kw)
    ev = []
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for t in range(0, T, chunk):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        s.push(mag[..., t:t + chunk])
        b.record()
        ev.append((a, b))
    s.flush()
    t1.record()
    torch.cuda.synchronize()
    per = [a.elapsed_time(b) * 1e3 for a, b in ev[1:]]
    return statistics.median(per), t0.elapsed_time(t1)


def stream_host(mag, chunk, kw, n_push=60):
    s = S.RTISIStream(look_ahead=LA, max_iter=ITERS, **kw)
    per = []
    for i, t in enumerate(range(0, min(T, n_push * chunk), chunk)):
        torch.cuda.synchronize()
        h = time.perf_counter()
        s.push(mag[..., t:t + chunk])
        torch.cuda.synchronize()
        if i:
            per.append((time.perf_counter() - h) * 1e6)
    s.flush()
    return statistics.median(per)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--batches", default="1,16,256")
    ap.add_argument("--chunks", default="1,4,16,64")
    o = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_rtisi_stream: needs a CUDA device")
    dev = torch.device("cuda")
    info = card()
    print(f"card: {info}")
    w = torch.hann_window(N_FFT, device=dev)
    kw = dict(window=w, hop_length=HOP)
    rows = []
    for B in [int(v) for v in o.batches.split(",")]:
        g = torch.Generator(device=dev).manual_seed(B)
        x = torch.randn(B, (T - 1) * HOP, device=dev, generator=g)
        mag = torch.stft(x, N_FFT, HOP, window=w, return_complex=True).abs().contiguous()
        assert mag.shape[-1] == T
        for _ in range(2):
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            S.RTISI_LA(mag, look_ahead=LA, max_iter=ITERS, alpha=0.99, verbose=0, **kw)
            b.record()
            torch.cuda.synchronize()
            whole = a.elapsed_time(b)
        for chunk in [int(v) for v in o.chunks.split(",")]:
            s = S.RTISIStream(look_ahead=LA, max_iter=ITERS, **kw)       # warm-up: every shape of the timed run
            for t in range(0, min(T, 4 * chunk), chunk):
                s.push(mag[..., t:t + chunk])
            s.flush()
            gpu_us, total = stream_events(mag, chunk, kw)
            host_us = stream_host(mag, chunk, kw)
            r = dict(B=B, chunk=chunk, gpu_us=round(gpu_us, 1), host_us=round(host_us, 1),
                     rtf=round(chunk * HOP / SR / (gpu_us * 1e-6), 2), stream_ms=round(total, 2), whole_ms=round(whole, 2))
            rows.append(r)
            print(f"B={B:4d} chunk={chunk:3d}: {gpu_us:9.1f} us GPU / push, {host_us:9.1f} us host enqueue-to-completion, "
                  f"RTF {r['rtf']:8.2f} per stream, stream {total:9.2f} ms vs whole call {whole:8.2f} ms", flush=True)
    if o.out:
        os.makedirs(os.path.dirname(os.path.abspath(o.out)), exist_ok=True)
        with open(o.out, "w") as f:
            json.dump(dict(card=info, shape=dict(n_fft=N_FFT, hop=HOP, look_ahead=LA, max_iter=ITERS, frames=T), rows=rows),
                      f, indent=1)


if __name__ == "__main__":
    main()
