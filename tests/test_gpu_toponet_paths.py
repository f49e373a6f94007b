"""TopoNet paths the model-level tests do not reach, each against the fp32 oracle (TF32 off).

`samroad_toponet` runs the fused tcgen05 kernel only for n_pairs == 16; every other n_pairs (1..15)
goes through the unfused chain: pair features, fp16 QKV GEMM, `topo_attention_kernel` (several
samples per block), two in-place residual `gemm_ln` calls per layer and `topo_output`.  The reference
configs always use 16 neighbour slots, so these tests build their pair queries with other widths.
They also feed validity masks with holes (the kNN builder only ever makes prefix masks) to both
paths, pin the fused kernel against the unfused chain on truncated inputs, and run token counts that
do not fill the 128-token tiles.  Logits are compared as well as scores; masked slots must report
output_proj.bias exactly (eval-mode nested-tensor fast path, SURVEY.md §8a P4).  Achieved numbers
are written to toponet_paths_report.json in the test report directory (`report_dir` fixture)."""
import json
import os

import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import samroad_oracle as O  # noqa: E402
from sam_road_b200 import synth  # noqa: E402
from sam_road_b200 import SAMRoad  # noqa: E402

DEV = "cuda:0"
P = 256                  # tile size of every net here: 16 x 16 embedding grid
TOL_VALID = 1e-3         # logit / score max-abs on valid slots (same bound as the fused path)
TOL_ALL = 3e-3           # logit max-abs on every slot (rows with no valid pair are flipped to all-valid)
_REPORT = {}
_NETS = {}


@pytest.fixture(scope="module", autouse=True)
def _fp32_oracle_math(report_dir):
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    yield
    _NETS.clear()
    path = os.path.join(report_dir, "toponet_paths_report.json")
    old = {}
    if os.path.exists(path):
        try:
            old = json.load(open(path))
        except Exception:
            old = {}
    old.update(_REPORT)
    json.dump(old, open(path, "w"), indent=1, sort_keys=True)


def _net(topo="normal", gain=1.0, seed=0):
    """(spec, device state_dict, SAMRoad) for ViT-B @256 with this TopoNet version; cached per module."""
    key = (topo, gain, seed)
    if key not in _NETS:
        cfg = dict(SAM_VERSION="vit_b", PATCH_SIZE=P, USE_SAM_DECODER=False, ENCODER_LORA=False,
                   TOPONET_VERSION=topo, NO_SAM=False)
        sd = synth.make_state_dict(cfg, seed=seed, logit_gain=gain)
        net = SAMRoad(cfg)
        net.load_state_dict(sd, strict=True)
        net.eval().to(DEV)
        _NETS[key] = (O.ModelSpec.from_config(cfg), {k: v.to(DEV) for k, v in sd.items()}, net)
    return _NETS[key]


def _feat(B, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(B, 256, P // 16, P // 16, generator=g).to(DEV)


def _inputs(B, n_points, Np, seed, ragged=True):
    return [t.to(DEV) for t in synth.make_topo_inputs(B, P, n_points, seed=seed, max_nbr=Np, ragged=ragged)]


def _run(model, feat, pts, prs, val):
    """(cuda logits, cuda scores, oracle logits, oracle scores), all [B, Ns, Np]."""
    spec, sd, net = model
    with torch.no_grad():
        o_s, o_l = O.infer_toponet(sd, spec, feat, pts, prs, val, return_logits=True)
    l, s = net._topo(feat, pts, prs, val, want_logits=True)
    return l[..., 0], s[..., 0], o_l[..., 0], o_s[..., 0]


def _compare(model, l, s, o_l, o_s, val):
    """Error summary of one call.  `val` is the caller's mask (any dtype); the kernels flip rows with
    no valid slot to all-valid, every other masked slot must hold output_proj.bias bit for bit."""
    bias = model[1]["topo_net.output_proj.bias"]
    v = val != 0
    keep = v | ~v.any(dim=-1, keepdim=True)
    dl, ds = (l - o_l).abs(), (s - o_s).abs()
    zero = torch.zeros((), device=l.device)
    return {
        "logit_maxabs_valid": torch.where(v, dl, zero).max().item() if v.numel() else 0.0,
        "logit_maxabs_all": dl.max().item() if dl.numel() else 0.0,
        "score_maxabs_valid": torch.where(v, ds, zero).max().item() if v.numel() else 0.0,
        "logit_range": [o_l.min().item(), o_l.max().item()] if o_l.numel() else [0.0, 0.0],
        "masked_slots": int((~keep).sum().item()),
        "masked_not_bias": int((l[~keep] != bias).sum().item()),
        "flipped_rows": int((~v.any(dim=-1)).sum().item()),
        "tokens": int(l.numel()),
        "finite": bool(torch.isfinite(l).all().item() and torch.isfinite(s).all().item()),
    }


def _assert_parity(rep, tol_valid=TOL_VALID, tol_all=TOL_ALL):
    assert rep["finite"], rep
    assert rep["masked_not_bias"] == 0, rep
    assert rep["logit_maxabs_valid"] <= tol_valid, rep
    assert rep["score_maxabs_valid"] <= tol_valid, rep
    assert rep["logit_maxabs_all"] <= tol_all, rep


# no_offset: the pair features lose the offset term, the logits span about +-1.8 instead of +-1.2 and
# the fp16 operand error grows with them.  Measured on a B200 (1000 W): valid-slot logit max-abs up to
# 1.18e-3 on the unfused path (Np = 8) and 1.22e-3 on the fused kernel (Np = 16, same test), scores
# <= 3.0e-4; with the normal version both paths stay below 6.2e-4.
TOL_VALID_LOGIT = {"no_offset": 2e-3}


@pytest.mark.parametrize("topo", ["normal", "no_offset", "no_tgt_features"])
@pytest.mark.parametrize("Np", [1, 2, 3, 5, 8, 12, 15, 16])
def test_unfused_path_parity(Np, topo):
    """n_pairs < 16: the unfused chain, on kNN queries with Np neighbour slots (prefix masks, ragged
    batch: padded rows have no valid pair).  Np = 16 runs the fused kernel on the same kind of input,
    for comparison."""
    model = _net(topo)
    feat = _feat(3, seed=100 + Np)
    pts, prs, val = _inputs(3, 40, Np, seed=30 + Np)
    assert prs.shape == (3, 40, Np, 2)
    l, s, o_l, o_s = _run(model, feat, pts, prs, val)
    rep = _compare(model, l, s, o_l, o_s, val)
    _REPORT[f"{'fused' if Np == 16 else 'unfused'}_{topo}_np{Np}"] = rep
    tol = TOL_VALID_LOGIT.get(topo, TOL_VALID)
    assert rep["score_maxabs_valid"] <= TOL_VALID, rep
    _assert_parity(rep, tol_valid=tol, tol_all=max(tol, TOL_ALL))


@pytest.mark.parametrize("Np", [1, 7])
def test_unfused_input_types(Np):
    """int32 pairs and points, float32 points off the pixel grid, points on the tile border (x = P)."""
    model = _net()
    feat = _feat(2, seed=7)
    pts, prs, val = _inputs(2, 30, Np, seed=40 + Np)
    pts[0, 0] = torch.tensor([P, P], device=DEV)
    pts[1, 1] = torch.tensor([0, P], device=DEV)
    pts[1, 2] = torch.tensor([P, 3], device=DEV)
    g = torch.Generator().manual_seed(Np)
    ptsf = (pts.float() + (torch.rand(pts.shape, generator=g) - 0.5).to(DEV)).clamp(0, P)
    ptsf[0, 3] = torch.tensor([P, P - 0.25], device=DEV)
    reps = {}
    l64, s64, o_l, o_s = _run(model, feat, pts, prs, val)
    reps["int64"] = _compare(model, l64, s64, o_l, o_s, val)
    l32, s32, _, _ = _run(model, feat, pts.int(), prs.int(), val)
    reps["int32"] = _compare(model, l32, s32, o_l, o_s, val)
    lf, sf, o_lf, o_sf = _run(model, feat, ptsf, prs, val)
    reps["float32_points"] = _compare(model, lf, sf, o_lf, o_sf, val)
    _REPORT[f"unfused_input_types_np{Np}"] = reps
    for rep in reps.values():
        _assert_parity(rep)
    # the index / coordinate dtype only changes how values are loaded, not what is computed
    assert torch.equal(l32, l64) and torch.equal(s32, s64)


def _holey_mask(kind, shape, seed):
    """Validity masks the kNN builder never makes.  Returns (mask, dtype-converted mask or None)."""
    g = torch.Generator().manual_seed(seed)
    R, Np = shape[0] * shape[1], shape[2]
    j = torch.arange(Np).expand(R, Np)
    if kind == "bernoulli":
        m = torch.rand(R, Np, generator=g) < 0.5
    elif kind == "last_only":
        m = j == Np - 1
    elif kind == "middle_one":
        pos = torch.randint(1, Np - 1, (R, 1), generator=g)
        m = j == pos
    elif kind == "alternating":
        m = (j + torch.arange(R).unsqueeze(1)) % 2 == 0
    elif kind == "all_invalid_rows":
        m = torch.rand(R, Np, generator=g) < 0.6
        m[::3] = False
    elif kind == "uint8_values":
        vals = torch.tensor([0, 0, 0, 1, 2, 7, 128, 255], dtype=torch.uint8)
        m = vals[torch.randint(0, len(vals), (R, Np), generator=g)]
    else:
        raise ValueError(kind)
    return m.view(shape).to(DEV)


MASK_KINDS = ["bernoulli", "last_only", "middle_one", "alternating", "all_invalid_rows", "uint8_values"]


@pytest.mark.parametrize("kind", MASK_KINDS)
@pytest.mark.parametrize("Np", [16, 7], ids=["fused_np16", "unfused_np7"])
def test_masks_with_holes(Np, kind):
    """Key-padding masks with holes, a lone last or middle slot, alternating slots, all-invalid rows and
    uint8 masks holding values other than 0/1, on the fused (Np = 16) and the unfused (Np = 7) path."""
    model = _net()
    feat = _feat(2, seed=11)
    pts, prs, _ = _inputs(2, 48, Np, seed=50 + Np, ragged=False)
    val = _holey_mask(kind, prs.shape[:3], seed=60 + Np)
    l, s, o_l, o_s = _run(model, feat, pts, prs, val)
    rep = _compare(model, l, s, o_l, o_s, val)
    rep["valid_fraction"] = float((val != 0).float().mean().item())
    _REPORT[f"mask_{kind}_np{Np}"] = rep
    _assert_parity(rep)
    if kind in ("last_only", "middle_one", "alternating"):
        assert rep["masked_slots"] > 0 and rep["flipped_rows"] == 0
    if kind == "all_invalid_rows":
        assert rep["flipped_rows"] > 0
    if kind == "uint8_values":     # any nonzero byte means valid: same bits as the bool mask
        assert val.dtype == torch.uint8 and int(val.max()) > 1
        lb, sb, _, _ = _run(model, feat, pts, prs, val != 0)
        assert torch.equal(lb, l) and torch.equal(sb, s)


@pytest.mark.parametrize("k", [4, 9, 15])
def test_fused_matches_unfused(k):
    """CUDA against CUDA: an Np = 16 input whose slots >= k are invalid (fused kernel) and its
    truncation to k slots (unfused chain) compute the same sequences, so their valid slots agree and
    the fused slots >= k report the bias exactly.  Rows with no valid slot among the first k are left
    out: the all-invalid flip makes them 16-slot sequences on one side and k-slot ones on the other."""
    model = _net()
    bias = model[1]["topo_net.output_proj.bias"]
    feat = _feat(2, seed=13)
    pts, prs, _ = _inputs(2, 64, 16, seed=70)
    g = torch.Generator().manual_seed(k)
    val = torch.rand(prs.shape[:3], generator=g) < 0.7
    val[:, ::9] = False                            # some rows with no valid slot at all
    val[..., k:] = False
    val = val.to(DEV)
    prs_k, val_k = prs[:, :, :k].contiguous(), val[:, :, :k].contiguous()
    lf, sf, o_lf, o_sf = _run(model, feat, pts, prs, val)
    lu, su, o_lu, o_su = _run(model, feat, pts, prs_k, val_k)
    rep_f = _compare(model, lf, sf, o_lf, o_sf, val)
    rep_u = _compare(model, lu, su, o_lu, o_su, val_k)
    rows = val_k.any(dim=-1, keepdim=True)
    both = rows & val_k
    d = torch.where(both, (lf[..., :k] - lu).abs(), torch.zeros((), device=DEV))
    rep = {"fused_vs_oracle": rep_f, "unfused_vs_oracle": rep_u,
           "fused_vs_unfused_logit_maxabs_valid": d.max().item(),
           "fused_vs_unfused_score_maxabs_valid":
               torch.where(both, (sf[..., :k] - su).abs(), torch.zeros((), device=DEV)).max().item(),
           "rows_compared": int(rows.sum().item()), "rows_left_out": int((~rows).sum().item())}
    _REPORT[f"fused_vs_unfused_k{k}"] = rep
    assert rep["rows_compared"] > 0 and rep["rows_left_out"] > 0
    assert rep["fused_vs_unfused_logit_maxabs_valid"] <= TOL_VALID, rep
    assert rep["fused_vs_unfused_score_maxabs_valid"] <= TOL_VALID, rep
    tail = lf[..., k:][rows.expand(-1, -1, 16 - k)]
    assert tail.numel() > 0 and bool((tail == bias).all()), rep
    for side, lg in (("fused", lf[..., :k]), ("unfused", lu)):
        masked = lg[rows.expand_as(val_k) & ~val_k]
        assert masked.numel() > 0 and bool((masked == bias).all()), (side, rep)
    _assert_parity(rep_f)
    _assert_parity(rep_u)


TOKEN_CASES = [(2, 37, 5), (2, 37, 16), (1, 1, 1), (3, 1, 3), (3, 1, 16), (4, 1021, 8)]


@pytest.mark.parametrize("B,Ns,Np", TOKEN_CASES, ids=[f"b{b}_ns{n}_np{p}" for b, n, p in TOKEN_CASES])
def test_token_counts_off_tile_grid(B, Ns, Np):
    """Token counts B*Ns*Np that leave the last 128-token tile partly empty: 370 and 1184 tokens, one
    sample per tile (a single token at B = Ns = Np = 1), and one 32 672-token call (255 full GEMM
    tiles and a partial one, 1021 attention blocks of four samples)."""
    case = f"b{B}_ns{Ns}_np{Np}"
    model = _net()
    feat = _feat(B, seed=17)
    if Ns == 1:    # one query per tile, pointing into a 40-point set (N != Ns)
        pts, prs, val = _inputs(B, 40, Np, seed=80 + Np, ragged=False)
        prs, val = prs[:, 5:6].contiguous(), val[:, 5:6].contiguous()
        assert bool(val.any())
    else:
        pts, prs, val = _inputs(B, Ns, Np, seed=90 + Np, ragged=Ns > 1000)
    assert prs.shape == (B, Ns, Np, 2)
    l, s, o_l, o_s = _run(model, feat, pts, prs, val)
    rep = _compare(model, l, s, o_l, o_s, val)
    _REPORT[f"tokens_{case}"] = rep
    assert rep["tokens"] == B * Ns * Np
    _assert_parity(rep)


@pytest.mark.parametrize("Np", [5, 12])
def test_unfused_wide_logits(Np):
    """output_proj scaled by 12 so the logits span several units: relative tolerance 2e-3 of the
    oracle's logit span (as test_gpu_model.test_parity_with_wide_logits), holes in the mask."""
    model = _net(gain=12.0, seed=1)
    feat = _feat(2, seed=19)
    pts, prs, val = _inputs(2, 48, Np, seed=110 + Np)
    val = val & _holey_mask("bernoulli", val.shape, seed=Np)
    l, s, o_l, o_s = _run(model, feat, pts, prs, val)
    rep = _compare(model, l, s, o_l, o_s, val)
    span = rep["logit_range"][1] - rep["logit_range"][0]
    rep["logit_span"] = span
    _REPORT[f"unfused_gain12_np{Np}"] = rep
    assert span > 2.0, rep
    assert rep["finite"] and rep["masked_not_bias"] == 0, rep
    assert rep["logit_maxabs_all"] <= 2e-3 * span, rep
