"""Time the closed-loop codec over a GOP at 1920x1024: a synthetic GOP of 12 (`synth.make_gop`: an I-frame and 11 P-frames),
coded by `gop.compress_gop` into version-2 containers and, separately, version-3 containers (row streams).
Per version, in the same run and alternating within each repetition: `compress_gop`, `decompress_gop` (the latents of all
11 frames entropy-decoded as one batch, then the synthesis frame by frame) and a frame-by-frame loop of `decompress` (each
frame's latents decoded on their own, as `decompress_gop` did before the batch), and `decompress_latents_many` of the 11
containers alone (the batched entropy decode without the synthesis).  Host clock around each call with a device
synchronise after it, median of `reps` after a warm-up; the per-GOP feature caches are off on both ends, so every frame
computes what a GOP's first P-frame computes.  Every round trip is checked bit for bit against compress_gop's frames.
It also prints what the closed loop costs on the same frames, over the 11 P-frames: coded bpp / PSNR (`gop.validate_codec`:
rates from the containers' bytes, PSNR of the frames a second module decodes) beside the estimated bpp / PSNR that
`gop.validate` reports for them (the likelihoods and reconstruction of the open-loop `forward`: `code_gop` -> `gop_stats`,
validate's P-frame sums).  The GPU's name and power limit are read in the same run.
python tools/codec_gop_bench.py [reps] [--amp]  ->  one JSON line."""
import argparse
import json
import sys
import time

import torch

sys.path.insert(0, ".")
from oracle.stats import build_oracle
from tdvc_b200 import gop, synth
from tdvc_b200.model import VideoCompressor
from tools.decode_bench import gpu_info

H, W, GOP = 1024, 1920, 12


def _module(orc, dev):
    m = VideoCompressor().eval()
    m.load_state_dict(orc.state_dict())
    m.cache_features = False
    return m.to(dev)


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return 1e3 * (time.perf_counter() - t0), out


def decompress_frame_by_frame(net, i_frame, containers):
    refs = gop.RefBuffer(gop.pad(i_frame, 64))
    recons = []
    for data in containers:
        window, keys = refs.window()
        recon = net.decompress(data, window, ref_keys=keys)
        refs.push(recon)
        recons.append(gop.crop(recon, (H, W)))
    return recons


def med(v):
    return round(sorted(v)[len(v) // 2], 3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("reps", nargs="?", type=int, default=3)
    ap.add_argument("--amp", action="store_true", help="code with enable_amp=True (\"mixed\" precision containers)")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    orc = build_oracle()
    enc, dec = _module(orc, dev), _module(orc, dev)
    frames = synth.make_gop(H, W, gop=GOP, seed=0).to(dev)
    i_frame, p_frames = frames[:1], frames[1:]
    res = {"gpu": gpu_info(), "frame": f"{W}x{H}", "gop": GOP, "p_frames": GOP - 1, "enable_amp": args.amp, "reps": args.reps}
    for key, rows in (("v2", False), ("v3", True)):
        c_ms, b_ms, f_ms, l_ms = [], [], [], []
        for rep in range(args.reps + 1):   # rep 0: warm-up (packs the weights, builds the tables and the plans)
            t, (containers, recons) = timed(lambda: gop.compress_gop(enc, i_frame, p_frames, args.amp, row_streams=rows))
            t_b, got = timed(lambda: gop.decompress_gop(dec, i_frame, containers, (H, W)))
            t_f, one = timed(lambda: decompress_frame_by_frame(dec, i_frame, containers))
            t_l, _ = timed(lambda: dec.decompress_latents_many(containers))
            for i in range(GOP - 1):
                assert torch.equal(got[i], recons[i]), (key, "decompress_gop", i)
                assert torch.equal(one[i], recons[i]), (key, "decompress", i)
            if rep:
                c_ms.append(t)
                b_ms.append(t_b)
                f_ms.append(t_f)
                l_ms.append(t_l)
        res[key] = {"container_bytes": sum(len(d) for d in containers), "bytes_per_frame": [len(d) for d in containers],
                    "compress_gop_ms": med(c_ms), "decompress_gop_ms": med(b_ms), "decompress_frame_by_frame_ms": med(f_ms),
                    "decompress_latents_many_ms": med(l_ms),
                    "decode_speedup": round(med(f_ms) / med(b_ms), 3), "bit_exact": True,
                    "compress_gop_ms_all": [round(v, 3) for v in c_ms], "decompress_gop_ms_all": [round(v, 3) for v in b_ms],
                    "decompress_frame_by_frame_ms_all": [round(v, 3) for v in f_ms],
                    "decompress_latents_many_ms_all": [round(v, 3) for v in l_ms]}
    # the closed loop's cost on the same frames: one GOP whose I-frame is the raw frame 0 (no I-frame coder here), P-frames only
    dataset = [(p_frames.cpu(), i_frame[0].cpu(), 0.0, 0.0, None, frames.cpu())]
    with torch.no_grad():
        est = gop.summarise(gop.gop_stats(gop.code_gop(enc, i_frame, p_frames, enable_amp=args.amp, with_msssim=True)))
    res["estimated"] = {k: round(est[k], 6) for k in ("bpp", "bpp_mv", "bpp_res", "psnr", "msssim")}
    for key, rows in (("v2", False), ("v3", True)):
        p = gop.validate_codec(dataset, enc, decoder=dec, enable_amp=args.amp, row_streams=rows)["p"]
        res[f"coded_{key}"] = {k: round(p[k], 6) for k in ("bpp", "bpp_mv", "bpp_res", "bpp_container", "psnr", "msssim")}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
