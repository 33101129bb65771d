"""Developer tool (GPU): the CUDA path against the two 1920x1024 fixtures, printed instead of asserted.  Reconstructions,
stage tensors and the symbols of chain frames 2.. are compared on the samples the fixtures store (oracle/make_golden_fullres.py)."""
import math
import sys
import warnings

import numpy as np
import torch

warnings.filterwarnings("ignore")
sys.path.insert(0, ".")
sys.path.insert(0, "tests")

from oracle import make_golden_fullres as GF  # noqa: E402


def flips(g, taps, net, p=""):
    out = {}
    for c, cn in (("mv", "mvCoder"), ("res", "resCoder")):
        yh = taps[f"{c}.y_hat"].cpu()
        y = taps[f"{c}.y"].cpu()
        want = g[p + f"{c}_y_hat"]
        if want.shape != tuple(yh.shape):     # a sampled latent: flips among the stored symbols only
            yh, y = GF.sample(yh, GF.Y_STEP_CHAIN), GF.sample(y, GF.Y_STEP_CHAIN)
        bad = torch.from_numpy(yh.numpy().astype(np.int16) != want.astype(np.int16))
        tie = ((y - torch.floor(y)) - 0.5).abs()
        out[c] = (int(bad.sum()), bad.numel(), float(tie[bad].max()) if bad.any() else 0.0, bad)
        med = getattr(net, cn).entropy_bottleneck.quantiles[:, 0, 1].detach().view(1, -1, 1, 1).cpu()
        zq = torch.round(taps[f"{c}.z_hat"].cpu() - med).numpy().astype(np.int16)
        out[c + ".z"] = int((zq != g[p + f"{c}_z_hat_minus_med"].astype(np.int16)).sum())
    return out


def main():
    from conftest import load_golden
    from oracle.stats import build_oracle
    from tdvc_b200 import gop as G
    from tdvc_b200 import synth
    from tdvc_b200.model import VideoCompressor
    dev = torch.device("cuda:0")
    orc = build_oracle()
    net = VideoCompressor().eval()
    net.load_state_dict(orc.state_dict(), strict=True)
    net = net.to(dev)
    g = load_golden("p1024x1920_s0")
    x, refs = synth.make_frame_pair(1024, 1920, seed=0)
    print("input checksum rel diff", abs(float(x.double().sum() + refs.double().sum()) - float(g["input_checksum"])) / float(g["input_checksum"]))
    for precision in ("exact", "mixed"):
        net.precision = precision
        taps = {}
        with torch.no_grad():
            recon, bres, bmv = net(x.to(dev), refs.to(dev), False, taps=taps)
        f = flips(g, taps, net)
        print(precision, "flips mv", f["mv"][:3], "res", f["res"][:3], "z", f["mv.z"], f["res.z"])
        bad_mv = f["mv"][3].any(1, keepdim=True).float()
        for r in (0, 2, 4, 8, 12):
            m = torch.nn.functional.max_pool2d(bad_mv, 2 * r + 1, 1, r) > 0
            inside = (f["res"][3] & m).sum().item()
            print(f"   res flips within {r} latents of an mv flip: {inside} of {f['res'][0]}")
        outside = f["res"][3] & ~(torch.nn.functional.max_pool2d(bad_mv, 17, 1, 8) > 0)
        y = taps["res.y"].cpu()
        tie = ((y - torch.floor(y)) - 0.5).abs()
        print("   max tie distance of res flips outside r=8:", float(tie[outside].max()) if outside.any() else 0.0)
        print("   ind equal", bool((taps["loopfilter.ind"].cpu().numpy().astype(np.int32) == g["ind"]).all()),
              "bpp rel", abs(bres.item() - float(g["bpp_res"][0])) / float(g["bpp_res"][0]), abs(bmv.item() - float(g["bpp_mv"][0])) / float(g["bpp_mv"][0]))
        want = torch.from_numpy(g["recon_q16"].astype(np.float32) / 65535.0)
        err = (GF.pixel_sample(recon.cpu(), GF.PIX_STEP) - want).abs().max(0).values
        allbad = (f["mv"][3] | f["res"][3]).any(1, keepdim=True).float()
        for r in (0, 4, 8, 12, 16):
            m = torch.nn.functional.interpolate(torch.nn.functional.max_pool2d(allbad, 2 * r + 1, 1, r), scale_factor=16, mode="nearest")[0, 0] > 0
            m = GF.sample(m, GF.PIX_STEP)
            print(f"   recon max err outside r={r} latents of any flip: {(err[~m].max().item() if (~m).any() else 0.0):.3e} (masked {m.float().mean().item():.4f}); overall {err.max().item():.3e}")
        mse = ((recon.cpu().double() - x.double()) ** 2).mean().item()
        print("   dPSNR", 10 * math.log10(1 / mse) - 10 * math.log10(1 / float(g["mse"])))
        for k in ("prediction1", "prediction", "recon_feat"):
            v = taps[k].cpu()
            scale = float(g["stat_" + k][2])
            d = (GF.sample(v[:, :, ::32, ::32], GF.S32_STEP) - torch.from_numpy(g["s32_" + k])).abs()
            tm = GF.sample(torch.nn.functional.avg_pool2d(v.double(), 64).float(), GF.TILE_STEP)
            print(f"   {k}: scale {scale:.3f} sample max err {d.max().item():.3e} frac>1e-4*scale {(d > 1e-4 * scale).float().mean().item():.2e}; "
                  f"tile-mean max err {(tm - torch.from_numpy(g['tile_' + k])).abs().max().item():.3e}")
    del taps
    # ---- chain
    g = load_golden("chain1024x1920_s100")
    n_p = int(g["n_p"])
    frames = synth.make_gop(1024, 1920, gop=n_p + 1, seed=int(g["seed"])).to(dev)
    for precision in ("exact", "mixed"):
        net.precision = precision
        refs = [frames[0:1]]
        for t in range(1, n_p + 1):
            taps = {}
            x = frames[t:t + 1]
            with torch.no_grad():
                recon, bres, bmv = net(x, G.reference_window(refs), False, taps=taps)
            refs.append(recon)
            if len(refs) > 4:
                refs = [refs[0]] + refs[-3:]
            p = f"f{t}_"
            f = flips(g, taps, net, p)
            mse = ((recon.double() - x.double()) ** 2).mean().item()
            want = torch.from_numpy(g[p + "recon_s4_q16"].astype(np.float32) / 65535.0)
            d = (GF.pixel_sample(recon[:, :, ::4, ::4].cpu(), GF.S4_PIX_STEP) - want).abs()
            tm = torch.nn.functional.avg_pool2d(recon.double(), 64).float().cpu()
            print(f"{precision} chain frame {t}: flips mv {f['mv'][:3]} res {f['res'][:3]} z {f['mv.z']} {f['res.z']} | "
                  f"ind eq {bool((taps['loopfilter.ind'].cpu().numpy().astype(np.int32) == g[p + 'ind']).all())} | bpp rel "
                  f"{abs(bres.item() - float(g[p + 'bpp_res'][0])) / float(g[p + 'bpp_res'][0]):.2e} {abs(bmv.item() - float(g[p + 'bpp_mv'][0])) / float(g[p + 'bpp_mv'][0]):.2e} | "
                  f"dPSNR {10 * math.log10(1 / mse) - 10 * math.log10(1 / float(g[p + 'mse'])):+.5f} | recon s4 max {d.max().item():.2e} "
                  f"frac>1e-3 {(d > 1e-3).float().mean().item():.2e} | tile mean max {(tm - torch.from_numpy(g[p + 'recon_tile'])).abs().max().item():.2e}")
            del taps


if __name__ == "__main__":
    main()
