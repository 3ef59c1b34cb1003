"""Throughput of restoring clips of DIFFERENT lengths, three arms in one run on one GPU (prints one JSON line).

--workload gsr (default), the VoiceFixer path:
  (a) one VoiceFixer.restore call per clip, the way a user without restore_many works: every new frame count builds a new
      plan, and those builds are inside the timed pass (one pass, no warm-up);
  (b) VoiceFixer.restore_many(max_batch=32): sorted, grouped, one vf_restore_varlen call per group (warm-up passes first);
  (c) 32 x 10 s equal clips through restore_varlen and through restore, alternating, to price the per-clip masking.

--workload ssr, the SSR_UNet / GSR-UNet path (unet_v2 + ISTFT), the same three arms:
  (a) one SSR_UNet.restore call per clip, plan builds included;
  (b) SSR_UNet.restore_many (one vf_ssr_restore_varlen call per group), after warm-up, checked bit for bit against (a);
  (c) 16 x 10 s equal clips through ssr_restore_varlen and through SSR_UNet.restore, alternating.
  An SSR plan holds ~2.2 GB per clip and 1024 padded frames, and restore_many keeps one plan per group, so the default set
  is smaller (32 clips, groups of 8): all of (b)'s plans stay cached (the line reports evictions during the timed passes).

The clip set is seeded: --clips lengths uniform in [--min-s, --max-s] seconds, speech-like synthetic audio (bench.py's
synth_batch) and bench.py's seeded synthetic weights.  The line also carries the padded / useful frame ratio of (b), the
card name and its power limit (read in the same run), and whether (a) and (b) agree bit for bit.

    python tools/bench_varlen.py [--workload gsr|ssr] [--clips N] [--max-batch B] [--steps 5] [--warmup 2] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SR = 44100
HOP = 441


def power_limit_w(index):
    try:
        out = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=20)
        return float(out.stdout.strip().splitlines()[0])
    except Exception:
        return None


def padded_frame_ratio(lengths, max_batch):
    from voicefixer_main_b200.model import group_sizes
    frames = sorted(1 + n // HOP for n in lengths)
    padded, pos = 0, 0
    for g in group_sizes(len(frames), max_batch):
        grp = frames[pos:pos + g]
        pos += g
        padded += g * (-(-max(grp) // 64) * 64)
    return padded / sum(frames)


def timed(fn, steps):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / steps, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", choices=("gsr", "ssr"), default="gsr")
    ap.add_argument("--clips", type=int, default=None, help="default 256 (gsr) / 32 (ssr)")
    ap.add_argument("--min-s", type=float, default=1.0)
    ap.add_argument("--max-s", type=float, default=15.0)
    ap.add_argument("--seed", type=int, default=2024)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--max-batch", type=int, default=None, help="default 32 (gsr) / 8 (ssr)")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    ssr = a.workload == "ssr"
    if a.clips is None:
        a.clips = 32 if ssr else 256
    if a.max_batch is None:
        a.max_batch = 8 if ssr else 32
    res = bench_ssr(a) if ssr else bench_gsr(a)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


def clip_set(a, dev):
    from bench import synth_batch
    rng = np.random.default_rng(a.seed)
    lengths = [int(x) for x in rng.integers(int(a.min_s * SR), int(a.max_s * SR) + 1, size=a.clips)]
    audio = synth_batch(a.clips, max(lengths), a.seed)
    clips = [audio[i, :n].contiguous().to(dev) for i, n in enumerate(lengths)]
    return lengths, clips, sum(lengths) / SR


def bench_gsr(a):
    from bench import synth_batch
    from voicefixer_main_b200 import VoiceFixer
    from voicefixer_main_b200.weights import make_state

    dev = torch.device("cuda:0")
    lengths, clips, audio_s = clip_set(a, dev)

    m = VoiceFixer().load_state_dict(make_state(1234)).eval().to(dev)
    eng = m._engine()

    # (a) one restore per clip, plan builds included
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out_a = [m.restore(c[None])[0] for c in clips]
    torch.cuda.synchronize()
    t_a = time.perf_counter() - t0
    plans_a = eng.plan_cache_info()

    # (b) restore_many: the first pass builds the plans (reported), then warm-up and timed passes
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out_b = m.restore_many(clips, max_batch=a.max_batch)
    torch.cuda.synchronize()
    t_b_first = time.perf_counter() - t0
    for _ in range(a.warmup):
        m.restore_many(clips, max_batch=a.max_batch)
    t_b, out_b2 = timed(lambda: m.restore_many(clips, max_batch=a.max_batch), a.steps)
    same = all(torch.equal(x, y) for x, y in zip(out_a, out_b)) and all(torch.equal(x, y) for x, y in zip(out_b, out_b2))
    n_diff = sum(not torch.equal(x, y) for x, y in zip(out_a, out_b))

    # (c) 32 x 10 s equal clips: restore_varlen vs restore, alternating
    x = synth_batch(32, 10 * SR, 1).to(dev)
    lens = [10 * SR] * 32
    for _ in range(a.warmup + 2):                  # +2: eager run and graph capture of both plans
        m.restore(x)
        eng.restore_varlen(x, lens)
    tv, tr = [], []
    for _ in range(a.steps):
        tr.append(timed(lambda: m.restore(x), 1)[0])
        tv.append(timed(lambda: eng.restore_varlen(x, lens), 1)[0])
    same_c = torch.equal(m.restore(x), eng.restore_varlen(x, lens))
    eng.check_errors()

    res = {
        "metric": "varlen_restore",
        "device": torch.cuda.get_device_name(dev),
        "power_limit_w": power_limit_w(dev.index or 0),
        "clips": a.clips, "lengths_s": [a.min_s, a.max_s], "seed": a.seed, "audio_s": round(audio_s, 2),
        "weights": "seeded synthetic (bench.py make_state(1234))",
        "a_per_clip_restore": {"warmup": "none: one pass, plan builds included", "s": round(t_a, 3),
                               "audio_s_per_s": round(audio_s / t_a, 1), "clips_per_s": round(a.clips / t_a, 1),
                               "distinct_frame_counts": len(set(1 + n // HOP for n in lengths)), "plan_cache": plans_a},
        "b_restore_many": {"max_batch": a.max_batch, "first_pass_s": round(t_b_first, 3),
                           "warmup": f"first pass + {a.warmup} passes", "steps": a.steps, "s": round(t_b, 4),
                           "audio_s_per_s": round(audio_s / t_b, 1), "clips_per_s": round(a.clips / t_b, 1),
                           "padded_over_useful_frames": round(padded_frame_ratio(lengths, a.max_batch), 4)},
        "c_equal_32x10s": {"warmup": a.warmup + 2, "steps": a.steps,
                           "restore_ms": round(1e3 * float(np.median(tr)), 2), "restore_varlen_ms": round(1e3 * float(np.median(tv)), 2),
                           "varlen_over_restore": round(float(np.median(tv)) / float(np.median(tr)), 4), "bit_identical": bool(same_c)},
        "a_vs_b_bit_identical": bool(same), "a_vs_b_clips_differing": n_diff,
    }
    return res


def bench_ssr(a):
    from bench import synth_batch
    from voicefixer_main_b200 import SSR_UNet
    from voicefixer_main_b200.weights import make_ssr_state

    dev = torch.device("cuda:0")
    lengths, clips, audio_s = clip_set(a, dev)
    m = SSR_UNet().load_state_dict(make_ssr_state(1234)).eval().to(dev)
    eng = m._engine()

    # (a) one SSR_UNet.restore per clip, plan builds included
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out_a = [m.restore(c[None])[0] for c in clips]
    torch.cuda.synchronize()
    t_a = time.perf_counter() - t0
    plans_a = eng.plan_cache_info()

    # (b) restore_many: the first pass builds the plans (reported), then warm-up and timed passes
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out_b = m.restore_many(clips, max_batch=a.max_batch)
    torch.cuda.synchronize()
    t_b_first = time.perf_counter() - t0
    for _ in range(a.warmup):
        m.restore_many(clips, max_batch=a.max_batch)
    before = eng.plan_cache_info()
    t_b, out_b2 = timed(lambda: m.restore_many(clips, max_batch=a.max_batch), a.steps)
    plans_b = eng.plan_cache_info()
    same = all(torch.equal(x, y) for x, y in zip(out_a, out_b)) and all(torch.equal(x, y) for x, y in zip(out_b, out_b2))
    n_diff = sum(not torch.equal(x, y) for x, y in zip(out_a, out_b))
    del out_a, out_b, out_b2

    # (c) 16 x 10 s equal clips: ssr_restore_varlen vs restore, alternating
    nc = 16
    x = synth_batch(nc, 10 * SR, 1).to(dev)
    lens = [10 * SR] * nc
    for _ in range(a.warmup + 2):                  # +2: eager run and graph capture of both plans
        m.restore(x)
        eng.ssr_restore_varlen(x, lens)
    tv, tr = [], []
    for _ in range(a.steps):
        tr.append(timed(lambda: m.restore(x), 1)[0])
        tv.append(timed(lambda: eng.ssr_restore_varlen(x, lens), 1)[0])
    same_c = torch.equal(m.restore(x), eng.ssr_restore_varlen(x, lens))
    eng.check_errors()

    return {
        "metric": "ssr_varlen_restore",
        "device": torch.cuda.get_device_name(dev),
        "power_limit_w": power_limit_w(dev.index or 0),
        "clips": a.clips, "lengths_s": [a.min_s, a.max_s], "seed": a.seed, "audio_s": round(audio_s, 2),
        "weights": "seeded synthetic (make_ssr_state(1234))",
        "a_per_clip_restore": {"warmup": "none: one pass, plan builds included", "s": round(t_a, 3),
                               "audio_s_per_s": round(audio_s / t_a, 1), "clips_per_s": round(a.clips / t_a, 1),
                               "distinct_frame_counts": len(set(1 + n // HOP for n in lengths)), "plan_cache": plans_a},
        "b_restore_many": {"max_batch": a.max_batch, "first_pass_s": round(t_b_first, 3),
                           "warmup": f"first pass + {a.warmup} passes", "steps": a.steps, "s": round(t_b, 4),
                           "audio_s_per_s": round(audio_s / t_b, 1), "clips_per_s": round(a.clips / t_b, 1),
                           "padded_over_useful_frames": round(padded_frame_ratio(lengths, a.max_batch), 4),
                           "plan_cache": plans_b, "evicted_during_timed_passes": plans_b["evicted"] - before["evicted"]},
        f"c_equal_{nc}x10s": {"warmup": a.warmup + 2, "steps": a.steps,
                              "restore_ms": round(1e3 * float(np.median(tr)), 2),
                              "ssr_restore_varlen_ms": round(1e3 * float(np.median(tv)), 2),
                              "varlen_over_restore": round(float(np.median(tv)) / float(np.median(tr)), 4),
                              "bit_identical": bool(same_c)},
        "a_vs_b_bit_identical": bool(same), "a_vs_b_clips_differing": n_diff,
    }


if __name__ == "__main__":
    main()
