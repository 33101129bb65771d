"""Time the device decoder of the y latent (`tdvc_ar_decode`) against the encoder (`tdvc_ar_code`) on a 1920x1024 P-frame
(64x120 latent, 7,680 dependent decode steps per coder), both coders.  The encoder's cluster size is 16 CTAs per image by
default; 8, or 0 (16 where that launches, else 8), time the other variants, and the decoder reproduces whichever ran.
CUDA events around each launch after warm-up; the GPU's name and power limit are read in the same run.
TDVC_B200_AR_DEBUG=1 adds the encoder's per-phase times on stderr.
python tools/decode_bench.py [reps] [--encoder-cluster {0,8,16}]  ->  one JSON line."""
import argparse
import json
import subprocess
import sys

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
    args = ap.parse_args()
    reps, cl = args.reps, args.encoder_cluster
    dev = torch.device("cuda:0")
    orc = build_oracle()
    net = VideoCompressor().eval()
    net.load_state_dict(orc.state_dict())
    net = net.to(dev)
    x, refs = synth.make_frame_pair(1024, 1920, seed=0)
    with torch.no_grad():
        net(x.to(dev), refs.to(dev), False, is_compress=True)
    W = net._weights(dev)
    plan = net._plan(1, 1024, 1920, dev)
    hy, wy = 64, 120
    res = {"gpu": gpu_info(), "frame": "1920x1024", "latent": [hy, wy], "encoder_cluster": cl}
    for cn in ("mv", "rs"):
        tabs = W["_tables"][cn]
        params = plan.buf(f"{cn}.params", 1, hy, wy, 256)
        enc_ms, dec_ms = [], []
        for rep in range(reps + 1):   # rep 0: warm-up
            t_enc, h = timed(lambda: coding.launch_coding(plan, W, cn, tabs, cluster=cl))
            enc = coding.finish_coding(h, keep=True)
            res["encoder_cluster_used"] = enc["cluster"]
            t_dec, h = timed(lambda: coding.launch_decoding(W, cn, tabs, enc["strings"][0], params, enc["cluster"]))
            dec = coding.finish_decoding(h)
            assert torch.equal(dec["y_hat"], enc["y_hat"]) and torch.equal(dec["y_symbols"], enc["y_symbols"])
            if rep:
                enc_ms.append(t_enc)
                dec_ms.append(t_dec)
        dec_med = sorted(dec_ms)[len(dec_ms) // 2]
        res[cn] = {"ar_code_ms": round(sorted(enc_ms)[len(enc_ms) // 2], 3), "ar_decode_ms": round(dec_med, 3),
                   "ar_decode_us_per_step": round(1e3 * dec_med / (hy * wy), 3),
                   "ar_decode_ms_all": [round(t, 3) for t in dec_ms]}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
