"""Time the device decoder of the y latent (`tdvc_ar_decode`) against the encoder (`tdvc_ar_code`) on a 1920x1024 P-frame
(64x120 latent, 7,680 dependent decode steps per coder), both coders.  The encoder's cluster size is 16 CTAs per image by
default; 8, or 0 (16 where that launches, else 8), time the other variants, and the decoder reproduces whichever ran.
CUDA events around each launch after warm-up; the GPU's name and power limit are read in the same run.
TDVC_B200_AR_DEBUG=1 adds the encoder's per-phase times on stderr.
--container: also time `VideoCompressor.decompress_latents` end to end (host clock around the call, which returns only
once both coders' latents are on the device) on the version-2 container of the frame `forward(is_compress=True)` coded,
decoded by a second module loaded from the same weights; the per-coder `tdvc_ar_decode` times of the same run stand beside
it, so the overlap of the two coders' chains can be read off.
--codec: also time the closed-loop codec end to end: `VideoCompressor.compress` (features to container bytes, host rANS
included) and `VideoCompressor.decompress` of its container by a second module (container to reconstruction), each with a
host clock around the call and a device synchronise after it, median of `reps` after a warm-up.  The per-GOP feature caches
are off, so every frame computes everything a GOP's first P-frame computes; the round trip is checked bit for bit.
--row-streams: also time the row-stream decoder `tdvc_ar_decode_rows` per coder (one rANS string per latent row, decoded
wavefront by wavefront) in the same loop as `tdvc_ar_code` and `tdvc_ar_decode`; with --codec also
`compress(row_streams=True)` and `decompress` of its version-3 container, and both containers' sizes.
python tools/decode_bench.py [reps] [--encoder-cluster {0,8,16}] [--container] [--codec] [--row-streams]  ->  one JSON
line."""
import argparse
import json
import subprocess
import sys
import time

import torch

sys.path.insert(0, ".")
from oracle.stats import build_oracle
from tdvc_b200 import coding, synth
from tdvc_b200.model import VideoCompressor


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else torch.cuda.get_device_name(0)


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("reps", nargs="?", type=int, default=5)
    ap.add_argument("--encoder-cluster", type=int, choices=(0, 8, 16), default=16)
    ap.add_argument("--container", action="store_true", help="also time decompress_latents on the frame's container")
    ap.add_argument("--codec", action="store_true", help="also time compress and decompress end to end")
    ap.add_argument("--row-streams", action="store_true", help="also time the row-stream decoder (container version 3)")
    args = ap.parse_args()
    reps, cl = args.reps, args.encoder_cluster
    dev = torch.device("cuda:0")
    orc = build_oracle()
    net = VideoCompressor().eval()
    net.load_state_dict(orc.state_dict())
    net = net.to(dev)
    x, refs = synth.make_frame_pair(1024, 1920, seed=0)
    gt = {}
    with torch.no_grad():
        net(x.to(dev), refs.to(dev), False, is_compress=True, taps=gt)
    blob = coding.pack_frame(net.last_coded, frame={"size": (1024, 1920), "N": 1, "precision": "exact"})
    W = net._weights(dev)
    plan = net._plan(1, 1024, 1920, dev)
    hy, wy = 64, 120
    res = {"gpu": gpu_info(), "frame": "1920x1024", "latent": [hy, wy], "encoder_cluster": cl}
    if args.container:
        # before the loop below recodes the plan's latents: the container holds forward()'s strings (automatic cluster)
        dec = VideoCompressor().eval()
        dec.load_state_dict(orc.state_dict())
        dec = dec.to(dev)
        ms = []
        for rep in range(reps + 1):   # rep 0: warm-up (packs the weights, builds the tables and the decoder's plan)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = dec.decompress_latents(blob)
            ms.append(1e3 * (time.perf_counter() - t0))
            for nm in ("mv", "res"):
                assert torch.equal(out[nm]["y_hat"], gt[f"{nm}.ac.y_hat"]), nm
                assert torch.equal(out[nm]["z_hat"], gt[f"{nm}.z_hat"].permute(0, 2, 3, 1)), nm
        ms = ms[1:]
        res["container"] = {"bytes": len(blob), "clusters": [net.last_coded[nm]["cluster"] for nm in ("mv", "res")],
                            "decompress_latents_ms": round(sorted(ms)[len(ms) // 2], 3),
                            "decompress_latents_ms_all": [round(t, 3) for t in ms]}
    for cn in ("mv", "rs"):
        tabs = W["_tables"][cn]
        params = plan.buf(f"{cn}.params", 1, hy, wy, 256)
        enc_ms, dec_ms, row_ms = [], [], []
        for rep in range(reps + 1):   # rep 0: warm-up
            t_enc, h = timed(lambda: coding.launch_coding(plan, W, cn, tabs, cluster=cl))
            hold = dict(h)   # the pinned host symbols stay valid until the next launch_coding
            enc = coding.finish_coding(h, keep=True)
            res["encoder_cluster_used"] = enc["cluster"]
            t_dec, h = timed(lambda: coding.launch_decoding(W, cn, tabs, enc["strings"][0], params, enc["cluster"]))
            dec = coding.finish_decoding(h)
            assert torch.equal(dec["y_hat"], enc["y_hat"]) and torch.equal(dec["y_symbols"], enc["y_symbols"])
            if args.row_streams:
                rows = coding.finish_coding(hold, rows=True)["strings"][0]
                t_row, h = timed(lambda: coding.launch_decoding(W, cn, tabs, rows, params, enc["cluster"], rows=True))
                dec = coding.finish_decoding(h)
                assert torch.equal(dec["y_hat"], enc["y_hat"]) and torch.equal(dec["y_symbols"], enc["y_symbols"])
            if rep:
                enc_ms.append(t_enc)
                dec_ms.append(t_dec)
                if args.row_streams:
                    row_ms.append(t_row)
        dec_med = sorted(dec_ms)[len(dec_ms) // 2]
        res[cn] = {"ar_code_ms": round(sorted(enc_ms)[len(enc_ms) // 2], 3), "ar_decode_ms": round(dec_med, 3),
                   "ar_decode_us_per_step": round(1e3 * dec_med / (hy * wy), 3),
                   "ar_decode_ms_all": [round(t, 3) for t in dec_ms]}
        if args.row_streams:
            res[cn].update({"ar_decode_rows_ms": round(sorted(row_ms)[len(row_ms) // 2], 3),
                            "ar_decode_rows_ms_all": [round(t, 3) for t in row_ms]})
    if args.codec:
        enc, dec = (_module(orc, dev, cache=False) for _ in range(2))
        xd, rd = x.to(dev), refs.to(dev)
        for key, rows in (("codec", False), ("codec_rows", True)) if args.row_streams else (("codec", False),):
            c_ms, d_ms = [], []
            for rep in range(reps + 1):   # rep 0: warm-up (packs the weights, builds the tables and both plans)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                recon, data = enc.compress(xd, rd, row_streams=rows)
                torch.cuda.synchronize()
                t1 = time.perf_counter()
                got = dec.decompress(data, rd)
                torch.cuda.synchronize()
                t2 = time.perf_counter()
                assert torch.equal(got, recon)
                c_ms.append(1e3 * (t1 - t0))
                d_ms.append(1e3 * (t2 - t1))
            c_ms, d_ms = c_ms[1:], d_ms[1:]
            res[key] = {"bytes": len(data), "compress_ms": round(sorted(c_ms)[len(c_ms) // 2], 3),
                        "decompress_ms": round(sorted(d_ms)[len(d_ms) // 2], 3),
                        "compress_ms_all": [round(t, 3) for t in c_ms], "decompress_ms_all": [round(t, 3) for t in d_ms]}
    print(json.dumps(res))


def _module(orc, dev, cache=True):
    m = VideoCompressor().eval()
    m.load_state_dict(orc.state_dict())
    m.cache_features = cache
    return m.to(dev)


if __name__ == "__main__":
    main()
