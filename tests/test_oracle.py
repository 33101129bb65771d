"""CPU tests of the oracle itself (-m "not gpu"): the restatement is pinned against
 (a) the reference's own unmodified code imported from TDVC_REFERENCE_ROOT (skipped where that tree is absent),
 (b) the committed golden fixtures made from (a) by oracle/make_golden.py, and the reference's state_dict layout and loader
     sample lists (tests/golden/reference_lists.json),
 (c) the reference's DCNv2 known-answer test (reference main/utils/dcnv2/testcuda.py:36-71).
"""
import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import dcn_naive, ref_import
from tdvc_b200 import synth

needs_ref = pytest.mark.skipif(not ref_import.available(),
                               reason="needs a checkout of the reference TDVC source tree at TDVC_REFERENCE_ROOT")


def test_state_dict_keys_and_checksum():
    """On a freshly built oracle: any forward of the session's shared one (other test modules run it) has zeroed the masked
    taps of its context models, since MaskedConv2d masks its weight in place as compressai's does."""
    from oracle.stats import build_oracle
    sd = build_oracle().state_dict()
    g = load_golden("p64x64_s1")
    assert abs(synth.state_checksum(sd) - float(g["state_checksum"])) < 1e-6 * float(g["state_checksum"])
    for must in ("mvCoder.g_a.0.gdn.gamma", "mvCoder.entropy_bottleneck._matrix0",
                 "resCoder.context_prediction.mask", "motion_est.spynet.basic_module.5.basic_module.4.conv.weight",
                 "motion_est.attn.conv1.conv.weight", "mcnet.dconv.conv_offset_mask.weight", "mcnet.feat_down.weight",
                 "loopfilter.conv_13.bias", "mcfilter.layer1.temporal_conv3d.weight", "motion_est.spynet.mean"):
        assert must in sd, must


def _reference_lists():
    import json
    import os
    from conftest import ROOT
    return json.load(open(os.path.join(ROOT, "tests", "golden", "reference_lists.json")))


def test_strict_state_dict_roundtrip_with_reference(oracle_model):
    """The reference's state_dict keys in order with their shapes (tests/golden/reference_lists.json): a checkpoint of either
    loads strictly into the other."""
    want = [(k, tuple(s)) for k, s in _reference_lists()["state_dict"]]
    assert [(k, tuple(v.shape)) for k, v in oracle_model.state_dict().items()] == want


@needs_ref
def test_restatement_bit_exact_vs_reference_code(oracle_model):
    ref = ref_import.reference_video_compressor().eval()
    ref.load_state_dict(oracle_model.state_dict(), strict=True)
    x, refs = synth.make_frame_pair(64, 128, seed=5)
    with torch.no_grad():
        a = oracle_model(x, refs, False)
        b = ref(x, refs, False)
    for p, q in zip(a, b):
        assert torch.equal(p, q)


@pytest.mark.parametrize("name", ["p64x64_s1", "p128x192_s2"])
def test_oracle_matches_golden(oracle_model, name):
    g = load_golden(name)
    x, refs = synth.make_frame_pair(int(g["h"]), int(g["w"]), seed=int(g["seed"]))
    assert abs(float(x.double().sum() + refs.double().sum()) - float(g["input_checksum"])) < 1e-3
    taps = {}
    with torch.no_grad():
        recon, bres, bmv = oracle_model(x, refs, False, taps=taps)
    # different host CPUs / thread counts reorder fp32 sums: not bit-exact across machines
    assert np.abs(recon.numpy() - g["recon"]).max() < 1e-4
    assert abs(bres.item() - float(g["bpp_res"][0])) < 1e-4 * float(g["bpp_res"][0])
    assert abs(bmv.item() - float(g["bpp_mv"][0])) < 1e-4 * float(g["bpp_mv"][0])
    for c in ("mv", "res"):
        same = (taps[f"{c}.y_hat"].numpy().astype(np.int16) == g[f"{c}_y_hat"]).mean()
        assert same >= 0.999, (c, same)
    assert (taps["loopfilter.ind"].numpy().astype(np.int32) == g["ind"]).all()


def test_dcn_zero_offset_known_answer():
    """reference testcuda.py:36-71: zero offsets, mask = sigmoid(0), identity-centre weights => 2*out == in."""
    torch.manual_seed(0)
    N, C, H, W, dg = 2, 8, 7, 9, 2
    x = torch.randn(N, C, H, W)
    wgt = torch.zeros(C, C, 3, 3)
    for c in range(C):
        wgt[c, c, 1, 1] = 1.0
    off = torch.zeros(N, dg * 18, H, W)
    msk = torch.sigmoid(torch.zeros(N, dg * 9, H, W))
    for fn in (dcn_naive.dcn_v2_forward_naive, dcn_naive.dcn_v2_forward_vectorised, dcn_naive.dcn_v2_forward):
        out = fn(x, wgt, torch.zeros(C), off, msk, dg)
        assert (2 * out - x).abs().max() < 1e-10 + 1e-7, fn.__name__


def test_dcn_three_restatements_agree():
    torch.manual_seed(1)
    N, C, O, H, W, dg = 1, 16, 8, 6, 7, 8
    x = torch.randn(N, C, H, W)
    wgt = torch.randn(O, C, 3, 3) * 0.1
    b = torch.randn(O)
    off = torch.randn(N, dg * 18, H, W) * 3.0
    msk = torch.rand(N, dg * 9, H, W)
    a = dcn_naive.dcn_v2_forward_naive(x, wgt, b, off, msk, dg)
    v = dcn_naive.dcn_v2_forward_vectorised(x, wgt, b, off, msk, dg)
    t = dcn_naive.dcn_v2_forward(x, wgt, b, off, msk, dg)
    assert (a - v).abs().max() < 2e-5 and (a - t).abs().max() < 2e-5


def test_compressai_port_basics():
    from oracle.compressai_port import GDN, EntropyBottleneck, GaussianConditional, MaskedConv2d
    torch.manual_seed(0)
    g = GDN(8)
    x = torch.randn(1, 8, 4, 4)
    beta = g.beta_reparam(g.beta)
    gamma = g.gamma_reparam(g.gamma)
    want = x / torch.sqrt(beta.view(1, 8, 1, 1) + torch.einsum("ij,njhw->nihw", gamma, x * x))
    assert (g(x) - want).abs().max() < 1e-6
    assert torch.allclose(beta, torch.ones(8), atol=1e-6) and torch.allclose(gamma, 0.1 * torch.eye(8), atol=1e-6)
    eb = EntropyBottleneck(4).eval()
    z = torch.randn(1, 4, 3, 3) * 3
    zh, lik = eb(z)
    assert torch.equal(zh, torch.round(z)) and (lik >= 1e-9).all() and (lik <= 1).all()
    # likelihoods over all integers sum to ~1 per channel
    grid = torch.arange(-60, 61).float().view(1, 1, -1, 1).expand(1, 4, -1, 1).contiguous()
    _, l2 = eb(grid)
    assert (l2.sum(dim=2) - 1).abs().max() < 2e-2  # init_scale 10: heavy tails beyond +-60
    gc = GaussianConditional(None).eval()
    y = torch.tensor([[[[0.4, 2.6, -1.5]]]])
    out, lk = gc(y, torch.tensor([[[[0.01, 1.0, 2.0]]]]), means=torch.tensor([[[[0.0, 0.2, 0.0]]]]))
    assert torch.allclose(out, torch.tensor([[[[0.0, 2.2, -2.0]]]]))  # round(-1.5) = -2 (half to even)
    assert lk[0, 0, 0, 0] > 0.99999  # sigma floored at 0.11
    m = MaskedConv2d(2, 4, 5, padding=2)
    assert int(m.mask[0, 0].sum()) == 12


# ------------------------------------------------------------------------------------------------ MS-SSIM
def _msssim_cases():
    import json
    import os
    from conftest import ROOT
    return json.load(open(os.path.join(ROOT, "tests", "golden", "msssim.json")))


def test_msssim_oracle_vs_golden():
    """oracle/ms_ssim.py against values of the reference's own ms_ssim (fixture made by oracle/make_golden.py)."""
    from oracle import ms_ssim as O
    from oracle.make_golden import msssim_inputs
    for c in _msssim_cases():
        x, y = msssim_inputs(c["seed"], tuple(c["shape"]), c["noise"])
        per = O.ms_ssim(x, y, data_range=1.0, size_average=False)
        assert torch.allclose(per, torch.tensor(c["per_image"]), atol=2e-5, rtol=0)
        assert abs(float(O.ms_ssim(x, y, data_range=1.0)) - c["mean"]) < 2e-5


@needs_ref
def test_msssim_oracle_vs_reference_function():
    """... and against the reference function imported verbatim, on fresh inputs (odd sizes exercise the padded pooling)."""
    import importlib
    from oracle import ms_ssim as O
    ref_import.load_reference_pnet()
    R = importlib.import_module("main.model.ms_ssim_torch")
    torch.manual_seed(3)
    for shape in ((1, 3, 163, 177), (2, 3, 192, 224)):
        x = torch.rand(shape)
        y = (x + 0.08 * torch.randn(shape)).clamp(0, 1)
        assert torch.allclose(O.ms_ssim(x, y, data_range=1.0, size_average=False),
                              R.ms_ssim(x, y, data_range=1.0, size_average=False), atol=2e-5, rtol=0)
    x = torch.rand(1, 3, 176, 176)
    assert abs(float(R.ms_ssim(x, x, data_range=1.0)) - 1.0) < 1e-6 and abs(float(O.ms_ssim(x, x, data_range=1.0)) - 1.0) < 1e-6


def _sample_list_trees(root):
    """Empty-file trees laid out as the reference's datasets: vimeo_septuplet (<dir>/<clip>/im1..im7.png, directory names
    chosen so that natural and plain sorting differ) and an evaluation tree (ori_img/<seq>/imNNN.png +
    compress_img_bpg/<seq>/<qp>/imNNN_<qp>.{png,txt}).  Returns (vimeo root, evaluation root, GOP size)."""
    import os
    vimeo = root / "vimeo"
    for d, clip in (("00010", "0002"), ("00002", "0010"), ("00002", "0009")):
        os.makedirs(vimeo / d / clip)
        for i in range(1, 8):
            open(vimeo / d / clip / f"im{i}.png", "wb").close()
    ev, gop, qp = root / "eval", 3, 27
    for seq, nfr in (("Seq10_416x240_50", 7), ("Seq2_416x240_30", 6), ("BQSquare_416x240_60", 9)):
        os.makedirs(ev / "ori_img" / seq)
        os.makedirs(ev / "compress_img_bpg" / seq / str(qp))
        for i in range(nfr):
            open(ev / "ori_img" / seq / f"im{i + 1:03d}.png", "wb").close()
        for g in range(nfr // gop):
            stem = ev / "compress_img_bpg" / seq / str(qp) / f"im{g * gop + 1:03d}_{qp}"
            open(str(stem) + ".png", "wb").close()
            open(str(stem) + ".txt", "w").write(f"{0.25 * (g + 1)}\n")
    return vimeo, ev, gop


def _sample_lists(root):
    """tdvc_b200.data's sample lists for the trees of _sample_list_trees, paths relative to `root`."""
    import os
    from tdvc_b200 import data as D
    vimeo, ev, gop = _sample_list_trees(root)

    def rel(x):
        return [rel(v) for v in x] if isinstance(x, (list, tuple)) else os.path.relpath(x, root) if isinstance(x, str) else x

    got_in, got_ref = D.VimeoDataset.get_vimeo(str(vimeo))
    out = {"vimeo": {"input": rel(got_in), "ref": rel(got_ref)}}
    for name, lmbda, hevc_class in (("uvg", 2048, None), ("hevc", 64, "D")):
        ds = D.GopDataset(str(ev), lmbda, gop, testfull=True, hevc_class=hevc_class)
        out[name] = {"ref": rel(ds.ref), "refbpp": list(ds.refbpp), "input": rel(ds.input), "len": len(ds)}
    return out


def test_dataset_sample_lists_match_reference_code(tmp_path):
    """tdvc_b200.data lists the same samples as the reference's own loaders (reference main/dataloader/dataset.py:
    `DataSet.get_vimeo` :210-247, `UVGDataSet.__init__` :16-60, `HEVCDataSet.__init__` :100-166) return for the same trees,
    recorded in tests/golden/reference_lists.json."""
    want = _reference_lists()
    got = _sample_lists(tmp_path)
    assert len(got["vimeo"]["input"]) == 21 and got["uvg"]["len"] == 7 and got["hevc"]["len"] == 3
    for k in ("vimeo", "uvg", "hevc"):
        assert got[k] == want[k], k
