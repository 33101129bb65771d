"""ORACLE tool: 1920x1024 fixtures (BASELINE configs 2 and 5) from the reference's OWN unmodified model code
(oracle/ref_import.py), run once in the build container where /root/reference exists (~25 min on 8 threads).

    python -m oracle.make_golden_fullres [pair] [chain]

Two fixtures, both with the conditioned weights (seed 1111) the small fixtures use (stored as samples, see below):

  tests/golden/p1024x1920_s0.npz      one P-frame with four DISTINCT raw reference frames (synth.make_frame_pair,
        seed 0): full reconstruction (uint16, x 65535), both bpp, every quantised symbol of both coders (int8), the
        FeatureFix match indices, and - for BASELINE config 5 (multi-frame fusion + in-loop filter at full size) -
        stride-32 samples and 64x64-tile means of prediction1 / prediction (mcfilter output) / recon_feat.
  tests/golden/chain1024x1920_s100.npz  six chained P-frames of the GOP bench.py codes first (synth.make_gop seed 100,
        reference window with warm-up duplication, reference tools/predict.py:51-68): per frame the symbols, indices, bpp,
        MSE against the source frame, a stride-4 sample of the reconstruction (uint16) and its 64x64-tile means.

Reconstruction and bpp come from the REFERENCE code; symbols / indices / stage tensors from the restatement
oracle/model.py run on the same inputs, which is asserted bit-exact with the reference on recon and bpp for every frame.

Every quantised symbol of the pair and of chain frame 1 is stored, and every z symbol of every frame, so that the tests see
each flipped symbol.  The rest is not stored whole (each file stays below 1 MB): shrink_pair / shrink_chain keep fixed samples
of it - every n-th element of a flattened array (`sample`), every n-th pixel position with its three channels
(`pixel_sample`) - and the tests take the same samples of the CUDA path's tensors.
"""
import os
import sys
import time
import warnings

import numpy as np
import torch

warnings.filterwarnings("ignore")

H, W = 1024, 1920
OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
STAGES = ("prediction1", "prediction", "recon_feat")
Y_STEP_CHAIN = 31              # symbols of chain frames 2.. (an odd step walks across channels, rows and columns)
PIX_STEP, S4_PIX_STEP = 97, 23  # pixel positions of the full reconstruction / of its stride-4 grid (chain)
S32_STEP, TILE_STEP = 8, 3      # stride-32 stage samples / 64x64-tile means


def sample(a, step):
    """Every `step`-th element of the flattened array (numpy or torch)."""
    return a.reshape(-1)[::step]


def pixel_sample(img, step):
    """(1, 3, H, W) -> (3, n): every `step`-th pixel position (row-major), all three channels."""
    return img.reshape(3, -1)[:, ::step]


def shrink_pair(d):
    """Full-size arrays of the pair fixture -> what tests/golden/p1024x1920_s0.npz stores."""
    out = {k: d[k] for k in ("h", "w", "seed", "state_checksum", "input_checksum", "bpp_res", "bpp_mv", "mse", "ind")}
    for c in ("mv", "res"):
        for k in (c + "_y_hat", c + "_z_hat_minus_med"):
            out[k] = d[k]
    out["recon_q16"] = pixel_sample(d["recon_q16"], PIX_STEP)
    for k in STAGES:
        out["s32_" + k] = sample(d["s32_" + k], S32_STEP)
        out["tile_" + k] = sample(d["tile_" + k], TILE_STEP)
        out["stat_" + k] = d["stat_" + k]
    return out


def shrink_chain(d):
    """Full-size arrays of the chain fixture (the frames coded so far) -> what tests/golden/chain1024x1920_s100.npz stores."""
    out = {k: d[k] for k in ("h", "w", "seed", "n_p", "state_checksum", "input_checksum")}
    t = 1
    while f"f{t}_mse" in d:
        p = f"f{t}_"
        for k in ("bpp_res", "bpp_mv", "mse", "ind", "recon_tile", "mv_z_hat_minus_med", "res_z_hat_minus_med"):
            out[p + k] = d[p + k]
        for c in ("mv", "res"):
            out[p + c + "_y_hat"] = d[p + c + "_y_hat"] if t == 1 else sample(d[p + c + "_y_hat"], Y_STEP_CHAIN)
        out[p + "recon_s4_q16"] = pixel_sample(d[p + "recon_s4_q16"], S4_PIX_STEP)
        t += 1
    return out


def _q16(x):
    return torch.round(x.clamp(0, 1) * 65535.0).to(torch.int32).numpy().astype(np.uint16)


def _tile_mean(x, t=64):
    return torch.nn.functional.avg_pool2d(x.double(), t).numpy()


def _symbols(d, taps, orc, prefix=""):
    for c in ("mv", "res"):
        yh = taps[f"{c}.y_hat"]
        med = getattr(orc, f"{c}Coder").entropy_bottleneck.quantiles[:, 0, 1].detach().view(1, -1, 1, 1)
        zq = torch.round(taps[f"{c}.z_hat"] - med)
        for nme, v in ((f"{c}_y_hat", yh), (f"{c}_z_hat_minus_med", zq)):
            assert v.abs().max() <= 32767
            dt = np.int8 if v.abs().max() <= 127 else np.int16
            d[prefix + nme] = v.numpy().astype(dt)
    d[prefix + "ind"] = taps["loopfilter.ind"].numpy().astype(np.int32)


def _run_both(ref, orc, x, refs):
    taps = {}
    with torch.no_grad():
        t0 = time.time()
        r = ref(x, refs, False)
        t1 = time.time()
        o = orc(x, refs, False, taps=taps)
        t2 = time.time()
    assert torch.equal(r[0], o[0]) and torch.equal(r[1], o[1]) and torch.equal(r[2], o[2]), \
        "oracle/model.py is not bit-exact with the reference code at 1920x1024"
    print(f"  reference {t1 - t0:.0f} s, restatement {t2 - t1:.0f} s, bpp_res {r[1].item():.5f} bpp_mv {r[2].item():.5f}", flush=True)
    return r, taps


def make_pair(ref, orc, csum):
    from tdvc_b200 import synth
    x, refs = synth.make_frame_pair(H, W, seed=0)
    (recon, bres, bmv), taps = _run_both(ref, orc, x, refs)
    d = dict(h=H, w=W, seed=0, state_checksum=csum, input_checksum=float(x.double().sum() + refs.double().sum()),
             recon_q16=_q16(recon), bpp_res=bres.numpy(), bpp_mv=bmv.numpy(),
             mse=float(((recon.double() - x.double()) ** 2).mean()))
    _symbols(d, taps, orc)
    for k in STAGES:
        v = taps[k]
        d["s32_" + k] = v[:, :, ::32, ::32].contiguous().numpy()
        d["tile_" + k] = _tile_mean(v).astype(np.float32)
        d["stat_" + k] = np.array([v.double().mean().item(), v.double().abs().mean().item(), v.abs().max().item()])
    np.savez_compressed(os.path.join(OUT, "p1024x1920_s0.npz"), **shrink_pair(d))
    print("pair written", flush=True)


def make_chain(ref, orc, csum, n_p=6, seed=100):
    from tdvc_b200 import gop as G
    from tdvc_b200 import synth
    frames = synth.make_gop(H, W, gop=n_p + 1, seed=seed)
    d = dict(h=H, w=W, seed=seed, n_p=n_p, state_checksum=csum, input_checksum=float(frames.double().sum()))
    refs = [frames[0:1]]
    for t in range(1, n_p + 1):
        x = frames[t:t + 1]
        print(f"chain frame {t}", flush=True)
        (recon, bres, bmv), taps = _run_both(ref, orc, x, G.reference_window(refs))
        refs.append(recon)
        if len(refs) > 4:
            refs = [refs[0]] + refs[-3:]
        p = f"f{t}_"
        d[p + "bpp_res"], d[p + "bpp_mv"] = bres.numpy(), bmv.numpy()
        d[p + "mse"] = float(((recon.double() - x.double()) ** 2).mean())
        d[p + "recon_s4_q16"] = _q16(recon[:, :, ::4, ::4].contiguous())
        d[p + "recon_tile"] = _tile_mean(recon).astype(np.float32)
        _symbols(d, taps, orc, p)
        del taps
        np.savez_compressed(os.path.join(OUT, f"chain1024x1920_s{seed}.npz"), **shrink_chain(d))   # rewritten after every frame
    print("chain written", flush=True)


def main(which):
    from oracle import ref_import
    from oracle.stats import build_oracle
    from tdvc_b200 import synth
    torch.set_num_threads(os.cpu_count() or 1)
    orc = build_oracle()
    ref = ref_import.reference_video_compressor().eval()
    ref.load_state_dict(orc.state_dict(), strict=True)
    csum = synth.state_checksum(orc.state_dict())
    os.makedirs(OUT, exist_ok=True)
    if not which or "pair" in which:
        make_pair(ref, orc, csum)
    if not which or "chain" in which:
        make_chain(ref, orc, csum)


if __name__ == "__main__":
    main(sys.argv[1:])
