"""-m gpu: the feature-gradient kernels of the backward (K5b: dFeat = Gs . other + the per-row diagonal term
in fp32, F.normalize backward, 1/len, bias column sums; autograd of multimodal.py:736,743,755) at a long
contraction, where `cvcl_feat_grad_norm_bwd_ws` splits the contraction over the SMs (fp32 atomics +
warp-per-row finishing pass) instead of the single cluster-epilogue kernel.  Both paths are checked
against a plain torch fp32 restatement of the same op and against each other."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu


def _inputs(M, E, Kc, diag_off, seed):
    g = torch.Generator().manual_seed(seed)
    dev = torch.device("cuda:0")
    Gs = (torch.randn(M, Kc, generator=g) * 2e-3).to(torch.bfloat16)
    other = torch.nn.functional.normalize(torch.randn(Kc, E, generator=g), dim=1).to(torch.bfloat16)
    feat = torch.nn.functional.normalize(torch.randn(M, E, generator=g), dim=1).to(torch.bfloat16)
    inv = (0.5 + torch.rand(M, generator=g)).float()
    lens = torch.randint(3, 26, (M,), generator=g, dtype=torch.int64)
    return [t.to(dev) for t in (Gs, other, feat, inv, lens)]


def _reference(Gs, other, feat, inv, lens, diag_off, diag_coef, normalize, use_len):
    M = Gs.shape[0]
    g = Gs.float() @ other.float() + diag_coef[:, None] * other[diag_off:diag_off + M].float()
    if normalize:
        dot = (feat.float() * g).sum(1, keepdim=True)
        g = (g - feat.float() * dot) * inv[:, None]
    if use_len:
        g = g / lens[:, None].float()
    return g, g.sum(0)


def _run(transposed, Gs, other, feat, inv, lens, diag_off, diag_coef, normalize, out_kind, scratch):
    from multimodal_baby_b200 import _cabi
    from multimodal_baby_b200.ops import _p, _stream
    M, Kc = Gs.shape
    E = other.shape[1]
    dev = Gs.device
    A = Gs.t().contiguous() if transposed else Gs
    ldg = A.shape[1]
    out32 = torch.empty((M, E), device=dev) if out_kind == "f32" else None
    out16 = torch.empty((M, E), dtype=torch.bfloat16, device=dev) if out_kind == "bf16" else None
    db = torch.zeros((E,), device=dev)
    acc = torch.empty((M, E), device=dev) if scratch else None
    _cabi.call("cvcl_feat_grad_norm_bwd_ws", _p(A), ldg, int(transposed), _p(other), E, M, E, Kc, _p(feat), E, _p(inv),
               int(normalize), _p(lens) if out_kind == "f32" else None, _p(other), E, Kc, diag_off, _p(diag_coef),
               _p(out32), E, _p(out16), E, _p(db), _p(acc), _stream())
    torch.cuda.synchronize()
    return (out32 if out32 is not None else out16.float()), db


@pytest.mark.parametrize("transposed", [False, True])
@pytest.mark.parametrize("out_kind", ["bf16", "f32"])
@pytest.mark.parametrize("Kc", [4096, 1600])
def test_featgrad_splitk_per_row_diag_matches_reference_and_fused_kernel(transposed, out_kind, Kc):
    M, E, diag_off = 512, 512, 256
    Gs, other, feat, inv, lens = _inputs(M, E, Kc, diag_off, 5 + Kc)
    # one coefficient per row (G_ii - bf16(Gs_ii)), of either sign and up to the -2w of an unconfident pair
    w = math.exp(2.659) * 0.5 / Kc
    diag_coef = (torch.rand(M, generator=torch.Generator().manual_seed(Kc)) * 2.5 - 2.0).to(Gs.device) * w
    ref, ref_db = _reference(Gs, other, feat, inv, lens, diag_off, diag_coef, True, out_kind == "f32")
    # split-K path: bf16 output needs the scratch, fp32 output accumulates in place
    got, db = _run(transposed, Gs, other, feat, inv, lens, diag_off, diag_coef, True, out_kind, out_kind == "bf16")
    tol = 6e-3 if out_kind == "bf16" else 2e-4            # bf16 output rounding / fp32 accumulation order
    scale = ref.abs().max()
    assert float((got - ref).abs().max() / scale) <= tol
    assert float((db - ref_db).abs().max() / ref_db.abs().max().clamp_min(1e-20)) <= 2e-2
    if out_kind == "bf16":
        # the single-kernel path (no scratch, bf16 out): same numbers up to bf16 rounding of the output
        fused, db_f = _run(transposed, Gs, other, feat, inv, lens, diag_off, diag_coef, True, out_kind, False)
        assert float((got - fused).abs().max() / scale) <= 8e-3
        assert float((db - db_f).abs().max() / ref_db.abs().max().clamp_min(1e-20)) <= 2e-2


def test_featgrad_splitk_per_row_diag_without_normalize_and_ragged_rows():
    """M not a multiple of 128, no normalisation, rows whose positives fall outside the diag matrix."""
    M, E, Kc, diag_off = 200, 512, 2048, 1900
    Gs, other, feat, inv, lens = _inputs(M, E, Kc, diag_off, 77)
    from multimodal_baby_b200 import _cabi
    from multimodal_baby_b200.ops import _p, _stream
    out = torch.empty((M, E), device=Gs.device)
    coef = -0.5 + 0.01 * torch.arange(M, dtype=torch.float32, device=Gs.device)
    _cabi.call("cvcl_feat_grad_norm_bwd_ws", _p(Gs), Kc, 0, _p(other), E, M, E, Kc, None, 0, None, 0, None,
               _p(other), E, Kc, diag_off, _p(coef), _p(out), E, None, 0, None, None, _stream())
    torch.cuda.synchronize()
    ref = Gs.float() @ other.float()
    n_in = Kc - diag_off                                  # rows m with m + diag_off < Kc get the diagonal term
    ref[:n_in] += coef[:n_in, None] * other[diag_off:].float()
    assert float((out - ref).abs().max() / ref.abs().max()) <= 2e-4
