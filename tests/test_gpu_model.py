"""End-to-end parity of the CUDA path (through SAMRoad -> ctypes -> C ABI) against the fp32 oracle
on seeded synthetic weights and inputs.  Tolerance (BASELINE.json north_star): mask-logit and
topology-logit max-abs <= 1e-3 with the reference's default-scale weights; the achieved numbers
are written to gpurun_out/parity_report.json.

The oracle runs in fp32 on the GPU (TF32 disabled) so that ViT-B@512 finishes in seconds; it is the
same code the CPU suite pins against the reference's golden fixtures."""
import json
import os

import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import samroad_oracle as O  # noqa: E402
from sam_road_b200 import synth  # noqa: E402
from sam_road_b200 import SAMRoad  # noqa: E402

DEV = "cuda:0"
TOL_LOGIT = 1e-3
# image embeddings (neck output, |feat| <= ~6): every configuration measured 3.0-3.7e-3 on a B200
# (profiles/r02_parity_report_v6.json)
TOL_FEAT = 1e-2
_REPORT = {}


@pytest.fixture(scope="module", autouse=True)
def _fp32_oracle_math(report_dir):
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    yield
    path = os.path.join(report_dir, "parity_report.json")
    old = {}
    if os.path.exists(path):
        try:
            old = json.load(open(path))
        except Exception:
            old = {}
    old.update(_REPORT)
    json.dump(old, open(path, "w"), indent=1, sort_keys=True)


def _config(patch, version="vit_b", topo="normal", lora=0, samdec=False):
    return dict(SAM_VERSION=version, PATCH_SIZE=patch, USE_SAM_DECODER=samdec,
                ENCODER_LORA=lora > 0, LORA_RANK=lora, TOPONET_VERSION=topo, NO_SAM=False)


def _build(cfg, seed=0, gain=1.0):
    spec = O.ModelSpec.from_config(cfg)
    sd = synth.make_state_dict(cfg, seed=seed, logit_gain=gain)
    net = SAMRoad(cfg)
    net.load_state_dict(sd, strict=True)
    net.eval().to(DEV)
    sd_dev = {k: v.to(DEV) for k, v in sd.items()}
    return spec, sd_dev, net


def _maxabs(a, b):
    return (a.float() - b.float()).abs().max().item()


@pytest.mark.parametrize("name,patch,version,B,lora", [
    ("vitb_256", 256, "vit_b", 3, 0),
    ("vitb_512", 512, "vit_b", 2, 0),
    ("vitb_256_lora4", 256, "vit_b", 1, 4),
    ("vith_256", 256, "vit_h", 1, 0),
    ("vitb_256_samdec", 256, "vit_b", 3, 0),       # USE_SAM_DECODER: True (archived configs)
    ("vitb_512_samdec", 512, "vit_b", 2, 0),
    ("vitl_256", 256, "vit_l", 2, 0),              # config/toponet_vitl_256.yaml
    ("vitb_1024", 1024, "vit_b", 1, 0),            # config/toponet_vitb_1024.yaml (64x64 token grid)
    ("vitb_1024_samdec", 1024, "vit_b", 1, 0),     # config/archived/finetune_enc_dec_1024.yaml (T = 4096)
])
def test_encode_and_topo_parity(name, patch, version, B, lora):
    cfg = _config(patch, version, lora=lora, samdec=name.endswith("samdec"))
    spec, sd, net = _build(cfg)
    rgb_u8 = synth.make_tiles(B, patch, seed=3).to(DEV)
    rgb = rgb_u8.float()
    with torch.no_grad():
        o_scores, o_feat, o_logits = O.infer_masks_and_img_features(sd, spec, rgb, return_logits=True)
    pts, prs, val = [t.to(DEV) for t in synth.make_topo_inputs(B, patch, 48, seed=4)]
    with torch.no_grad():
        o_ts, o_tl = O.infer_toponet(sd, spec, o_feat, pts, prs, val, return_logits=True)

    scores, feat = net.infer_masks_and_img_features(rgb)
    assert scores.shape == o_scores.shape and feat.shape == o_feat.shape
    assert scores.dtype == torch.float32 and feat.dtype == torch.float32
    scores_u8, feat_u8 = net.infer_masks_and_img_features(rgb_u8)     # uint8 input extension
    assert torch.equal(scores, scores_u8) and torch.equal(feat, feat_u8)

    logits, scores2, t_logits, t_scores = net(rgb, pts, prs, val)
    assert torch.equal(scores2, scores)
    t_scores2 = net.infer_toponet(feat, pts, prs, val)
    assert torch.equal(t_scores2, t_scores)
    # TopoNet alone on the oracle's own embeddings (isolates TopoNet error from encoder error)
    t_scores_iso = net.infer_toponet(o_feat, pts, prs, val)
    vmask = val.unsqueeze(-1)
    rep = {
        "feat_maxabs": _maxabs(feat, o_feat), "feat_absmax": o_feat.abs().max().item(),
        "mask_logit_maxabs": _maxabs(logits, o_logits),
        "mask_logit_range": [o_logits.min().item(), o_logits.max().item()],
        "mask_score_maxabs": _maxabs(scores, o_scores),
        "topo_logit_maxabs_valid": ((t_logits - o_tl).abs() * vmask).max().item(),
        "topo_logit_maxabs_all": _maxabs(t_logits, o_tl),
        "topo_logit_range": [o_tl.min().item(), o_tl.max().item()],
        "topo_score_maxabs_valid": ((t_scores - o_ts).abs() * vmask).max().item(),
        "topo_score_iso_maxabs_valid": ((t_scores_iso - o_ts).abs() * vmask).max().item(),
        "tolerance_logit": TOL_LOGIT, "tolerance_feat": TOL_FEAT,
    }
    _REPORT[name] = rep
    print(name, json.dumps(rep))
    assert torch.isfinite(logits).all() and torch.isfinite(t_logits).all() and torch.isfinite(feat).all()
    assert rep["feat_maxabs"] <= TOL_FEAT, rep
    assert rep["mask_logit_maxabs"] <= TOL_LOGIT, rep
    # consumers read valid slots only (inferencer.py:213, model.py:536,587); masked slots are the
    # exact bias, rows with no valid pair (flipped to all-valid, model.py:128-130) are sanity-bounded
    assert rep["topo_logit_maxabs_valid"] <= TOL_LOGIT, rep
    assert rep["topo_logit_maxabs_all"] <= 3 * TOL_LOGIT, rep
    assert rep["mask_score_maxabs"] <= TOL_LOGIT and rep["topo_score_maxabs_valid"] <= TOL_LOGIT


def test_benched_configuration_b64_composition():
    """The configuration bench.py times: ViT-B @512, B = 64 tiles in ONE call -- 2-CTA GEMMs, TMA
    reduce-add shortcut epilogues, snake traversal, persistent attention CTAs running dozens of units.
    (a) 4 of the 64 tiles against the oracle at the 1e-3 tolerance; (b) the same 4 tiles from a B = 4
    call with every GEMM on the 1-CTA kernels and ascending traversal (debug mode 1|16), which must agree
    with the B = 64 result to rounding (different tile shapes / epilogues round differently; how the
    variants relate bit-wise is recorded in the report); (c) a tile's result must not depend on where it
    sits in the batch: permuting the batch permutes the output bit for bit."""
    from sam_road_b200 import _lib
    lib = _lib.load()
    cfg = _config(512)
    spec, sd, net = _build(cfg, seed=0)
    B = 64
    rgb = synth.make_tiles(B, 512, seed=21).to(DEV)
    pts, prs, val = [t.to(DEV) for t in synth.make_topo_inputs(B, 512, 256, seed=22, ragged=False)]
    sel = [0, 21, 42, 63]
    runs = {}
    try:
        for tag, mode, idx in (("b64", 0, None), ("b64_smem_shortcut", 4, None), ("b64_1cta", 1 | 16, None),
                               ("b64_no_snake", 16, None), ("b4_1cta", 1 | 16, sel), ("b4", 0, sel)):
            lib.samroad_debug_disable_2cta_gemm(mode)
            a = (rgb, pts, prs, val) if idx is None else (rgb[idx], pts[idx], prs[idx], val[idx])
            logits, _, tl, _ = net(*a)
            feat = net.infer_masks_and_img_features(a[0])[1]
            runs[tag] = (logits, tl, feat) if idx is not None else (logits[sel], tl[sel], feat[sel])
            if tag == "b64":
                logits64 = logits
    finally:
        lib.samroad_debug_disable_2cta_gemm(0)
    with torch.no_grad():    # O.forward, with the image embeddings kept
        _, o_feat, o_logits = O.infer_masks_and_img_features(sd, spec, rgb[sel].float(), return_logits=True)
        _, o_tl = O.infer_toponet(sd, spec, o_feat, pts[sel], prs[sel], val[sel], return_logits=True)
    v = val[sel].unsqueeze(-1)
    eq = lambda a, b: bool(all(torch.equal(x, y) for x, y in zip(runs[a], runs[b])))   # noqa: E731
    rep = {
        "mask_logit_maxabs_b64_vs_oracle": _maxabs(runs["b64"][0], o_logits),
        "topo_logit_maxabs_valid_b64_vs_oracle": ((runs["b64"][1] - o_tl).abs() * v).max().item(),
        "mask_logit_maxabs_b4_1cta_vs_oracle": _maxabs(runs["b4_1cta"][0], o_logits),
        "mask_logit_maxabs_b64_vs_b4_1cta": _maxabs(runs["b64"][0], runs["b4_1cta"][0]),
        "feat_maxabs_b64_vs_b4_1cta": _maxabs(runs["b64"][2], runs["b4_1cta"][2]),
        "feat_maxabs_b64_vs_oracle": _maxabs(runs["b64"][2], o_feat),
        "bit_equal": {"b64_1cta==b4_1cta": eq("b64_1cta", "b4_1cta"), "b64==b64_no_snake": eq("b64", "b64_no_snake"),
                      "b64_smem_shortcut==b64_1cta": eq("b64_smem_shortcut", "b64_1cta"),
                      "b64==b64_smem_shortcut": eq("b64", "b64_smem_shortcut"), "b4==b4_1cta": eq("b4", "b4_1cta")},
    }
    _REPORT["vitb_512_b64_composition"] = rep
    print(json.dumps(rep))
    assert torch.isfinite(logits64).all() and torch.isfinite(runs["b64"][1]).all()
    assert rep["mask_logit_maxabs_b64_vs_oracle"] <= TOL_LOGIT, rep
    assert rep["topo_logit_maxabs_valid_b64_vs_oracle"] <= TOL_LOGIT, rep
    assert rep["mask_logit_maxabs_b4_1cta_vs_oracle"] <= TOL_LOGIT, rep
    assert rep["feat_maxabs_b64_vs_oracle"] <= TOL_FEAT, rep
    assert rep["mask_logit_maxabs_b64_vs_b4_1cta"] <= TOL_LOGIT and rep["feat_maxabs_b64_vs_b4_1cta"] <= 5e-3, rep
    assert rep["bit_equal"]["b64==b64_no_snake"], rep          # traversal order must not change any bit
    # every tile of the batch is computed independently of its neighbours
    perm = torch.randperm(B, generator=torch.Generator().manual_seed(0)).to(DEV)
    logits_p = net(rgb[perm], pts[perm], prs[perm], val[perm])[0]
    assert torch.equal(logits_p, logits64[perm])


@pytest.mark.parametrize("patch", [256, 512])
def test_b64_run_to_run_determinism(patch):
    """Identical calls return identical bits at the benched batch size (64 tiles, ~20 work units per
    persistent CTA in every kernel)."""
    cfg = _config(patch)
    spec, sd, net = _build(cfg, seed=0, gain=6.0)
    rgb = synth.make_tiles(64, patch, seed=3).to(DEV)
    pts, prs, val = [t.to(DEV) for t in synth.make_topo_inputs(64, patch, 128, seed=4)]
    first = net(rgb, pts, prs, val)
    for _ in range(5):
        again = net(rgb, pts, prs, val)
        for a, b in zip(first, again):
            assert torch.equal(a, b), int((a != b).sum())


def test_parity_with_wide_logits():
    """Same check with the last decoder layer / output_proj scaled so logits span several units
    (random init only gives +-0.5): relative tolerance 2e-3 of the logit range."""
    cfg = _config(256)
    spec, sd, net = _build(cfg, seed=1, gain=12.0)
    rgb = synth.make_tiles(2, 256, seed=5).to(DEV).float()
    pts, prs, val = [t.to(DEV) for t in synth.make_topo_inputs(2, 256, 64, seed=6)]
    with torch.no_grad():
        o = O.forward(sd, spec, rgb, pts, prs, val)
    r = net(rgb, pts, prs, val)
    span_m = (o[0].max() - o[0].min()).item()
    span_t = (o[2].max() - o[2].min()).item()
    em, et = _maxabs(r[0], o[0]), _maxabs(r[2], o[2])
    _REPORT["vitb_256_gain12"] = {"mask_logit_maxabs": em, "mask_logit_span": span_m,
                                  "topo_logit_maxabs": et, "topo_logit_span": span_t}
    print(_REPORT["vitb_256_gain12"])
    assert em <= 2e-3 * span_m and et <= 2e-3 * span_t


@pytest.mark.parametrize("topo", ["no_offset", "no_transformer", "no_tgt_features"])
def test_toponet_versions(topo):
    cfg = _config(256, topo=topo)
    spec, sd, net = _build(cfg, seed=2)
    feat = torch.randn(2, 256, 16, 16, device=DEV)
    pts, prs, val = [t.to(DEV) for t in synth.make_topo_inputs(2, 256, 30, seed=8)]
    with torch.no_grad():
        o_ts, o_tl = O.infer_toponet(sd, spec, feat, pts, prs, val, return_logits=True)
    ts = net.infer_toponet(feat, pts, prs, val)
    assert _maxabs(ts, o_ts) <= TOL_LOGIT


def test_toponet_dense_c4():
    """BASELINE config 4 (toponet_vitb_512_cityscale_8x8): dense TopoNet path -- 1024 keypoints per 512
    tile, every one of them a query with 16 neighbour slots (16 384 sequences of 16 per tile), ragged
    validity as inferencer.py:156-176 builds it.  Fused tcgen05 kernel against the oracle."""
    cfg = _config(512)
    spec, sd, net = _build(cfg, seed=5)
    g = torch.Generator().manual_seed(12)
    feat = torch.randn(2, 256, 32, 32, generator=g).to(DEV)
    pts, prs, val = [t.to(DEV) for t in synth.make_topo_inputs(2, 512, 1024, seed=13)]
    assert prs.shape == (2, 1024, 16, 2)
    with torch.no_grad():
        o_ts, o_tl = O.infer_toponet(sd, spec, feat, pts, prs, val, return_logits=True)
    ts = net.infer_toponet(feat, pts, prs, val)
    v = val.unsqueeze(-1)
    err_valid = ((ts - o_ts).abs() * v).max().item()
    _REPORT["toponet_dense_c4"] = {"topo_score_maxabs_valid": err_valid, "sequences": int(2 * 1024),
                                   "valid_fraction": float(val.float().mean().item())}
    assert err_valid <= TOL_LOGIT
    assert _maxabs(ts, o_ts) <= 3 * TOL_LOGIT


def test_toponet_edge_cases():
    """float32 / int32 inputs, all-invalid rows (flipped to valid, model.py:128-130), border points
    x = P (legal: the rtree box query is inclusive, SURVEY.md §8a P8), empty batch."""
    cfg = _config(256)
    spec, sd, net = _build(cfg, seed=3)
    feat = torch.randn(2, 256, 16, 16, device=DEV)
    pts, prs, val = synth.make_topo_inputs(2, 256, 20, seed=9)
    pts[0, 0] = torch.tensor([256, 256])
    pts[1, 1] = torch.tensor([0, 256])
    val[0, 3] = False
    val[1, :] = False
    pts, prs, val = pts.to(DEV), prs.to(DEV), val.to(DEV)
    with torch.no_grad():
        o_ts = O.infer_toponet(sd, spec, feat, pts, prs, val)
        o_tsf = O.infer_toponet(sd, spec, feat, pts.float() + 0.25, prs, val)
    assert _maxabs(net.infer_toponet(feat, pts, prs, val), o_ts) <= TOL_LOGIT
    assert _maxabs(net.infer_toponet(feat, pts.int(), prs.int(), val), o_ts) <= TOL_LOGIT
    assert _maxabs(net.infer_toponet(feat, pts.float() + 0.25, prs, val), o_tsf) <= TOL_LOGIT
    empty = net.infer_toponet(feat, pts[:, :0], prs[:, :0], val[:, :0])
    assert empty.shape == (2, 0, 16, 1)
    s0, f0 = net.infer_masks_and_img_features(torch.zeros((0, 256, 256, 3), device=DEV))
    assert s0.shape == (0, 256, 256, 2) and f0.shape == (0, 256, 16, 16)


def test_non_contiguous_and_errors():
    cfg = _config(256)
    spec, sd, net = _build(cfg, seed=4)
    base = synth.make_tiles(2, 256, seed=10).to(DEV).float()
    view = base.permute(0, 3, 1, 2).contiguous().permute(0, 2, 3, 1)    # non-contiguous NHWC view
    a = net.infer_masks_and_img_features(base)
    b = net.infer_masks_and_img_features(view)
    assert torch.equal(a[0], b[0])
    with pytest.raises(ValueError):
        net.infer_masks_and_img_features(torch.zeros(1, 128, 128, 3, device=DEV))
    with pytest.raises(RuntimeError):
        net.infer_masks_and_img_features(torch.zeros(1, 256, 256, 3))    # CPU tensor: no fallback
