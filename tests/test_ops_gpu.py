"""GPU parity of the operator kernels, called through the C ABI (ctypes), against
 (1) the CPU oracle, (2) the golden fixtures made by the reference's own code, and
 (3) what the reference's CUDA kernels, compiled unmodified for sm_100a, computed on the same inputs
     (tests/golden/reference_kernels.npz, made by tests/golden/make_golden_kernels.py).
Integer / index results (NMS keep lists) are bit-exact; fp32 results use the tolerance written
next to each assert."""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import ops as O
from oracle.highway_lstm import highway_lstm_forward as oracle_lstm

pytestmark = pytest.mark.gpu
REF_KERNELS_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_kernels.npz")


def rand_boxes(rng, n, lo=1.0, hi=190.0, size=592):
    x1 = rng.uniform(0, 400, n); y1 = rng.uniform(0, 400, n)
    w = rng.uniform(lo, hi, n); h = rng.uniform(lo, hi, n)
    return np.stack([x1, y1, np.minimum(x1 + w, size - 1), np.minimum(y1 + h, size - 1)], 1).astype(np.float32)


def rois_for(rng, n, batch):
    return np.concatenate([rng.randint(0, batch, (n, 1)).astype(np.float32), rand_boxes(rng, n)], 1)


# ------------------------------------------------------------------------------- RoIAlign
@pytest.mark.parametrize("B,C,N", [(1, 32, 17), (6, 512, 120), (2, 70, 33)])
def test_roi_align_forward_vs_oracle(cuda, B, C, N):
    from lib.fpn.roi_align.functions.roi_align import RoIAlignFunction
    rng = np.random.RandomState(B * 100 + N)
    feat = rng.randn(B, C, 37, 37).astype(np.float32)
    rois = rois_for(rng, N, B)
    rois[0, 1:] = [0, 0, 591, 591]           # whole image (large window -> gather path)
    rois[1, 1:] = [-40, -40, 100, 100]       # partly outside -> extrapolation
    rois[2, 1:] = [300, 300, 300, 300]       # degenerate
    out = RoIAlignFunction(7, 7, 1 / 16)(torch.from_numpy(feat).to(cuda), torch.from_numpy(rois).to(cuda))
    ref = O.roi_align_forward(feat, O.normalize_rois(rois, 37, 37, 1 / 16), 7, 7)
    # same fp32 operation order incl. fused multiply-adds -> expected bit-equal; allow 1e-6
    np.testing.assert_allclose(out.cpu().numpy(), ref, rtol=1e-6, atol=1e-6)


def test_roi_align_edge_cases(cuda):
    from lib.fpn.roi_align.functions.roi_align import RoIAlignFunction
    rng = np.random.RandomState(3)
    feat = torch.from_numpy(rng.randn(2, 8, 37, 37).astype(np.float32)).to(cuda)
    empty = RoIAlignFunction(7, 7, 1 / 16)(feat, torch.zeros(0, 5, device=cuda))
    assert tuple(empty.shape) == (0, 8, 7, 7)
    rois = np.array([[7, 10, 10, 50, 50], [-1, 10, 10, 50, 50]], np.float32)  # bad batch index -> zeros
    out = RoIAlignFunction(7, 7, 1 / 16)(feat, torch.from_numpy(rois).to(cuda))
    assert float(out.abs().max()) == 0.0
    # other crop sizes incl. 1x1 (centre sample) and a large crop that takes the generic kernel
    for ph, pw in [(1, 1), (3, 5), (14, 14), (40, 40)]:
        r = rois_for(rng, 9, 2)
        o = RoIAlignFunction(ph, pw, 1 / 16)(feat, torch.from_numpy(r).to(cuda)).cpu().numpy()
        e = O.roi_align_forward(feat.cpu().numpy(), O.normalize_rois(r, 37, 37, 1 / 16), ph, pw)
        np.testing.assert_allclose(o, e, rtol=1e-6, atol=1e-6)


def test_roi_align_nhwc_matches_nchw(cuda):
    from lib.fpn.roi_align.functions.roi_align import RoIAlignFunction, roi_align_nhwc
    rng = np.random.RandomState(5)
    feat = torch.from_numpy(rng.randn(3, 512, 37, 37).astype(np.float32)).to(cuda)
    rois = torch.from_numpy(rois_for(rng, 77, 3)).to(cuda)
    a = RoIAlignFunction(7, 7, 1 / 16)(feat, rois)                         # [N,C,7,7]
    b = roi_align_nhwc(feat.permute(0, 2, 3, 1).contiguous(), rois, 7, 7, 1 / 16)  # [N,49,C]
    assert torch.equal(a.permute(0, 2, 3, 1).reshape(77, 49, 512), b)


@pytest.mark.parametrize("C,ph,pw", [(512, 7, 7), (136, 7, 7), (256, 3, 5), (64, 7, 14), (128, 1, 1), (70, 7, 7)])
def test_roi_align_nhwc_edge_cases(cuda, C, ph, pw):
    """The NHWC kernels (16-byte vector path, and the scalar one for C % 4 != 0) are bit-equal to the NCHW kernel (itself
    bit-equal to the reference's) on whole-image, partly / fully outside, degenerate, DESCENDING and bad-batch rois."""
    from lib.fpn.roi_align.functions.roi_align import RoIAlignFunction, roi_align_nhwc
    rng = np.random.RandomState(C + ph)
    feat = torch.from_numpy(rng.randn(3, C, 37, 37).astype(np.float32)).to(cuda)
    r = rois_for(rng, 64, 3)
    r[0, 1:] = [0, 0, 591, 591]
    r[1, 1:] = [-40, -40, 100, 100]
    r[2, 1:] = [300, 300, 300, 300]
    r[3, 1:] = [400, 380, 200, 120]          # x2 < x1, y2 < y1: sample rows run downwards
    r[4, 1:] = [-500, -500, -300, -300]      # entirely outside
    r[5, 1:] = [100, -90, 180, 700]          # rows outside at both ends, >1 px apart in between
    r[6, 0] = 9                              # bad batch index
    r[7, 1:] = [64, 64, 160, 160]            # samples on exact pixel centres (lo == hi)
    r[8, 1:] = [10, 500, 300, 591]
    rois = torch.from_numpy(r).to(cuda)
    a = RoIAlignFunction(ph, pw, 1 / 16)(feat, rois)
    b = roi_align_nhwc(feat.permute(0, 2, 3, 1).contiguous(), rois, ph, pw, 1 / 16)
    assert torch.equal(a.permute(0, 2, 3, 1).reshape(64, ph * pw, C), b)


def test_roi_align_backward_vs_oracle(cuda):
    from lib.fpn.roi_align.functions.roi_align import RoIAlignFunction
    rng = np.random.RandomState(9)
    B, C, N = 2, 16, 25
    feat = torch.from_numpy(rng.randn(B, C, 37, 37).astype(np.float32)).to(cuda).requires_grad_(True)
    rois = rois_for(rng, N, B)
    rois[0, 1:] = [0, 0, 591, 591]            # whole image
    rois[1, 1:] = [-40, -40, 100, 100]        # partly outside
    rois[2, 1:] = [300, 300, 300, 300]        # degenerate: all 49 bins on one point
    rois[3, 1:] = [400, 380, 200, 120]        # descending
    rois[4, 1:] = [64, 64, 160, 160]          # samples on pixel centres (lo == hi)
    rois[5, 1:] = [100, -90, 180, 700]        # rows outside at both ends
    g = rng.randn(N, C, 7, 7).astype(np.float32)
    out = RoIAlignFunction(7, 7, 1 / 16)(feat, torch.from_numpy(rois).to(cuda))
    out.backward(torch.from_numpy(g).to(cuda))
    ref = O.roi_align_backward(g, O.normalize_rois(rois, 37, 37, 1 / 16), B, C, 37, 37)
    # atomics accumulate in arbitrary order -> fp32 tolerance
    np.testing.assert_allclose(feat.grad.cpu().numpy(), ref, rtol=1e-5, atol=1e-5)
    # linearity: <RoIAlign(f), g> == <f, RoIAlign^T(g)>
    lhs = float((out.detach().double() * torch.from_numpy(g).to(cuda).double()).sum())
    rhs = float((feat.detach().double() * feat.grad.double()).sum())
    assert abs(lhs - rhs) <= 1e-4 * max(1.0, abs(lhs))


def golden_sample(n, k, seed):
    """Seeded flat indices at which an output too large to store whole is kept in REF_KERNELS_GOLDEN."""
    return np.random.RandomState(seed).randint(0, n, k)


def roi_align_launch(lib, feat, rois, grad_out):
    """Forward and backward of a library's ROIAlignForwardLaucher / ROIAlignBackwardLaucher (7x7, 1/16, 37x37 maps)
    on device arrays; returns (pooled [N,C,7,7], feature gradient [B,C,37,37]) as numpy."""
    import motifs_cabi as C
    from lib.fpn.roi_align.functions.roi_align import normalize_rois
    B, Cn, N = feat.shape[0], feat.shape[1], rois.shape[0]
    rn = normalize_rois(rois, 37, 37, 1 / 16)
    out = torch.zeros(N, Cn, 7, 7, device=feat.device)
    gf = torch.zeros(B, Cn, 37, 37, device=feat.device)
    st = C.cur_stream()
    assert lib.ROIAlignForwardLaucher(C.ptr(feat), C.ptr(rn), N, B, 37, 37, 7, 7, Cn, 0.0, C.ptr(out), st) == 1
    assert lib.ROIAlignBackwardLaucher(C.ptr(grad_out), C.ptr(rn), N, B, 37, 37, 7, 7, Cn, C.ptr(gf), st) == 1
    torch.cuda.synchronize()
    return out.cpu().numpy(), gf.cpu().numpy()


def roi_align_reference_case(cuda):
    rng = np.random.RandomState(11)
    B, Cn, N = 6, 512, 300
    feat = torch.from_numpy(rng.randn(B, Cn, 37, 37).astype(np.float32)).to(cuda)
    rois = torch.from_numpy(rois_for(rng, N, B)).to(cuda)
    g = torch.from_numpy(rng.randn(N, Cn, 7, 7).astype(np.float32)).to(cuda)
    return feat, rois, g


def test_roi_align_vs_reference_kernel(cuda):
    """Same inputs as the reference's ROIAlignForward/Backward (compiled unmodified) were given in
    tests/golden/make_golden_kernels.py. The forward is bit-exact: the SHA-256 of the whole output and a seeded sample
    are held. The backward (atomics) is held to 1e-4 on a seeded sample and on the sum of every (image, channel) plane."""
    import hashlib
    import motifs_cabi as C
    gold = np.load(REF_KERNELS_GOLDEN)
    fwd, bwd = roi_align_launch(C.load(), *roi_align_reference_case(cuda))
    i = golden_sample(fwd.size, gold["roi_fwd_sample"].size, 1)
    d = np.abs(fwd.reshape(-1)[i] - gold["roi_fwd_sample"]).max()
    assert np.array_equal(fwd.reshape(-1)[i], gold["roi_fwd_sample"]), d
    assert hashlib.sha256(fwd.tobytes()).hexdigest() == str(gold["roi_fwd_sha256"])      # bit-exact, whole output
    j = golden_sample(bwd.size, gold["roi_bwd_sample"].size, 2)
    np.testing.assert_allclose(bwd.reshape(-1)[j], gold["roi_bwd_sample"], rtol=1e-4, atol=1e-4)
    planes = bwd.reshape(bwd.shape[0] * bwd.shape[1], -1).astype(np.float64)
    assert np.all(np.abs(planes.sum(1) - gold["roi_bwd_plane_sums"])
                  <= 1e-4 * (planes.shape[1] + gold["roi_bwd_plane_abs_sums"]))


# ------------------------------------------------------------------------------- NMS
def nms_case(rng, n):
    b = rand_boxes(rng, n, lo=16, hi=300)
    s = rng.permutation(n).astype(np.float32) / n     # distinct scores: no ties
    return s, b


@pytest.mark.parametrize("n,thr", [(1, 0.7), (63, 0.5), (64, 0.7), (65, 0.3), (1000, 0.3), (6000, 0.7)])
def test_apply_nms_bit_exact_vs_oracle(cuda, n, thr):
    from lib.fpn.nms.functions.nms import apply_nms
    rng = np.random.RandomState(n)
    s, b = nms_case(rng, n)
    got = apply_nms(torch.from_numpy(s).to(cuda), torch.from_numpy(b).to(cuda), pre_nms_topn=6000,
                    post_nms_topn=1000, nms_thresh=thr)
    exp = O.apply_nms(s, b, pre_nms_topn=6000, post_nms_topn=1000, nms_thresh=thr)
    assert got.dtype == torch.int64
    assert np.array_equal(got.cpu().numpy(), exp)


def test_apply_nms_multi_image_and_topn(cuda):
    from lib.fpn.nms.functions.nms import apply_nms
    rng = np.random.RandomState(77)
    per = [500, 1, 0, 321]
    s = np.concatenate([nms_case(rng, n)[0] for n in per]) if per else None
    b = np.concatenate([nms_case(rng, n)[1] for n in per])
    got, im_per = apply_nms(torch.from_numpy(s).to(cuda), torch.from_numpy(b).to(cuda), pre_nms_topn=300,
                            post_nms_topn=50, boxes_per_im=per, nms_thresh=0.6)
    exp, exp_per = O.apply_nms(s, b, pre_nms_topn=300, post_nms_topn=50, boxes_per_im=per, nms_thresh=0.6)
    assert im_per == exp_per
    assert np.array_equal(got.cpu().numpy(), exp)


def nms_reference_cases():
    """(n, threshold, score-sorted boxes) of the comparison with the reference's ApplyNMSGPU."""
    rng = np.random.RandomState(5)
    cases = []
    for n, thr in [(6000, 0.7), (777, 0.3)]:
        s, b = nms_case(rng, n)
        cases.append((n, thr, b[np.argsort(-s, kind="stable")]))
    return cases


def nms_launch(lib, boxes, thr, cuda):
    """Keep list of a library's ApplyNMSGPU (kernel + host loop) on score-sorted boxes."""
    import motifs_cabi as C
    n = boxes.shape[0]
    bs = torch.from_numpy(boxes).to(cuda).contiguous()
    keep = (ctypes.c_int * n)()
    k = lib.ApplyNMSGPU(keep, C.ptr(bs), n, thr, 0)
    return np.array(keep[:k])


def test_nms_drop_in_symbol_vs_reference_kernel(cuda):
    """ApplyNMSGPU (host keep list) of this library vs the oracle and vs the keep lists of the reference's compiled
    kernel + host loop on the same boxes (tests/golden/make_golden_kernels.py)."""
    import motifs_cabi as C
    gold = np.load(REF_KERNELS_GOLDEN)
    for n, thr, boxes in nms_reference_cases():
        mine = nms_launch(C.load(), boxes, thr, cuda)
        assert np.array_equal(mine, O.nms_keep(boxes, thr))
        assert np.array_equal(mine, gold["nms_keep_%d" % n])


# ------------------------------------------------------------------------------- boxes
def test_box_kernels_vs_golden(cuda, golden):
    from lib.fpn.box_utils import bbox_overlaps, bbox_preds
    from lib.fpn.box_intersections_cpu import bbox as bbox_mod
    from lib.draw_rectangles.draw_rectangles import draw_union_boxes, draw_union_boxes_cuda
    a, b = golden["iou_a"], golden["iou_b"]
    assert np.array_equal(bbox_mod.bbox_overlaps(a, b), golden["iou_f64"])          # float64 bit-exact
    assert np.array_equal(bbox_mod.bbox_intersections(a, b), golden["inter_f64"])
    got = bbox_overlaps(torch.from_numpy(a).to(cuda), torch.from_numpy(b).to(cuda)).cpu().numpy()
    assert np.array_equal(got, golden["iou_f32"])                                    # fp32 bit-exact
    assert np.array_equal(draw_union_boxes(golden["draw_pairs"], 27), golden["draw_27"])
    assert np.array_equal(draw_union_boxes(golden["draw_pairs"][:50], 13), golden["draw_13"])
    shifted = draw_union_boxes_cuda(torch.from_numpy(golden["draw_pairs"]).to(cuda), 27, offset=0.5).cpu().numpy()
    assert np.array_equal(shifted, golden["draw_27"] - np.float32(0.5))
    bp = bbox_preds(torch.from_numpy(golden["bp_boxes"]).to(cuda), torch.from_numpy(golden["bp_deltas"]).to(cuda))
    np.testing.assert_allclose(bp.cpu().numpy(), golden["bp_out"], rtol=1e-6, atol=1e-4)  # expf ulp


def test_union_rois(cuda):
    import motifs_cabi as C
    rng = np.random.RandomState(2)
    rois = np.concatenate([np.zeros((40, 1), np.float32), rand_boxes(rng, 40)], 1)
    pairs = rng.randint(0, 40, (100, 2)).astype(np.int64)
    r = torch.from_numpy(rois).to(cuda); p = torch.from_numpy(pairs).to(cuda)
    u = torch.empty(100, 5, device=cuda); pb = torch.empty(100, 8, device=cuda)
    C.check(C.load().mb200_union_rois(C.ptr(r), C.ptr(p), 100, C.ptr(u), C.ptr(pb), C.cur_stream()), "union")
    assert np.array_equal(u.cpu().numpy(), O.union_rois(rois, pairs))
    assert np.array_equal(pb.cpu().numpy(), np.concatenate([rois[pairs[:, 0], 1:], rois[pairs[:, 1], 1:]], 1))


# ------------------------------------------------------------------------------- sgemm
@pytest.mark.parametrize("ta,tb", [(0, 0), (0, 1), (1, 0), (1, 1)])
def test_sgemm(cuda, ta, tb):
    import motifs_cabi as C
    torch.manual_seed(0)
    M, N, K = 123, 77, 201
    A = torch.randn(K, M, device=cuda) if ta else torch.randn(M, K, device=cuda)
    B = torch.randn(N, K, device=cuda) if tb else torch.randn(K, N, device=cuda)
    Cm = torch.randn(M, N, device=cuda)
    ref = 0.5 * ((A.t() if ta else A).double() @ (B.t() if tb else B).double()) + 2.0 * Cm.double()
    rc = C.load().mb200_sgemm(ta, tb, M, N, K, 0.5, C.ptr(A), A.stride(0), C.ptr(B), B.stride(0), 2.0, C.ptr(Cm), N,
                              C.cur_stream())
    assert rc == 1
    assert torch.allclose(Cm.double(), ref, rtol=1e-5, atol=1e-4)


# ------------------------------------------------------------------------------- highway LSTM
def lstm_inputs(rng, T, B, In, H, L, lengths):
    from lib.lstm.highway_lstm_cuda.alternating_highway_lstm import AlternatingHighwayLSTM
    torch.manual_seed(int(rng.randint(1 << 30)))
    m = AlternatingHighwayLSTM(In, H, L, recurrent_dropout_probability=0.2)
    with torch.no_grad():
        m.bias.add_(0.1 * torch.randn_like(m.bias))
    x = torch.randn(T, B, In)
    for b, l in enumerate(lengths):
        x[l:, b] = 0
    drop = (torch.rand(L, B, H) > 0.2).float() / 0.8
    return m, x, drop


@pytest.mark.parametrize("T,B,In,H,L,lengths", [
    (5, 3, 12, 16, 2, [5, 3, 2]),
    (7, 6, 40, 64, 4, [7, 7, 5, 4, 2, 1]),
    (20, 6, 712, 512, 4, [20, 17, 12, 9, 9, 3]),      # edge-context shape (SURVEY §8a a8)
    (9, 40, 33, 128, 3, list(range(40, 0, -1))[:40]),  # more rows than one batch tile; lengths > T clipped below
])
def test_highway_lstm_forward_backward_vs_oracle(cuda, T, B, In, H, L, lengths):
    from torch.nn.utils.rnn import pack_padded_sequence, pad_packed_sequence
    lengths = sorted([min(l, T) for l in lengths], reverse=True)
    lengths[0] = T
    rng = np.random.RandomState(T * 1000 + B)
    m, x, drop = lstm_inputs(rng, T, B, In, H, L, lengths)
    # oracle (CPU, autograd)
    xo = x.clone().requires_grad_(True)
    wo = m.weight.detach().clone().requires_grad_(True)
    bo = m.bias.detach().clone().requires_grad_(True)
    out_o = oracle_lstm(xo, lengths, wo, bo, drop, H, L)
    gout = torch.randn(T, B, H)
    for b, l in enumerate(lengths):
        gout[l:, b] = 0
    (out_o * gout).sum().backward()
    # product
    mc = m.to(cuda).train()
    xc = x.to(cuda).requires_grad_(True)
    packed = pack_padded_sequence(xc, lengths)
    out_p, _ = mc(packed, dropout_weights=drop.to(cuda))
    out_c, _ = pad_packed_sequence(out_p, total_length=T)
    # fp32, different summation order in the K=In / K=H dot products: 2e-5 abs on O(1) values
    np.testing.assert_allclose(out_c.detach().cpu().numpy(), out_o.detach().numpy(), rtol=1e-4, atol=2e-5)
    (out_c * gout.to(cuda)).sum().backward()
    np.testing.assert_allclose(xc.grad.cpu().numpy(), xo.grad.numpy(), rtol=1e-3, atol=1e-4)
    scale = float(wo.grad.abs().max())
    np.testing.assert_allclose(mc.weight.grad.cpu().numpy(), wo.grad.numpy(), rtol=1e-3, atol=1e-4 * max(1.0, scale))
    np.testing.assert_allclose(mc.bias.grad.cpu().numpy(), bo.grad.numpy(), rtol=1e-3, atol=1e-4 * max(1.0, scale))


LSTM_REFERENCE_DIMS = (11, 6, 100, 64, 2)          # T, B, In, H, L
LSTM_REFERENCE_LENGTHS = [11, 9, 9, 4, 2, 1]


def lstm_reference_case(cuda):
    T, B, In, H, L = LSTM_REFERENCE_DIMS
    m, x, drop = lstm_inputs(np.random.RandomState(4), T, B, In, H, L, LSTM_REFERENCE_LENGTHS)
    return m.weight.detach().to(cuda), m.bias.detach().to(cuda), x.to(cuda), drop.to(cuda)


def lstm_launch(lib, handle, w, bias, x, drop):
    """A library's highway_lstm_forward_ongpu (training mode, gates saved) on the LSTM_REFERENCE_* case; returns
    h, c [L,T+1,B,H] and gates [L,T,B,6H] as numpy."""
    import motifs_cabi as C
    T, B, In, H, L = LSTM_REFERENCE_DIMS
    cuda = x.device
    len_host = (ctypes.c_int * B)(*LSTM_REFERENCE_LENGTHS)
    h = torch.zeros(L, T + 1, B, H, device=cuda); c = torch.zeros(L, T + 1, B, H, device=cuda)
    gates = torch.zeros(L, T, B, 6 * H, device=cuda)
    ti = torch.zeros(B, 6 * H, device=cuda); th = torch.zeros(B, 5 * H, device=cuda)
    lib.highway_lstm_forward_ongpu(In, H, B, L, T, C.ptr(x), len_host, C.ptr(h), C.ptr(c), C.ptr(ti), C.ptr(th),
                                   C.ptr(w), C.ptr(bias), C.ptr(drop), C.ptr(gates), 1, C.cur_stream(), handle)
    torch.cuda.synchronize()
    return h.cpu().numpy(), c.cpu().numpy(), gates.cpu().numpy()


def lstm_covered_gates(gates):
    """The gate rows the reference writes, flattened: rows >= covered(t) of step t are left untouched by it."""
    T = LSTM_REFERENCE_DIMS[0]
    cov = [sum(1 for l in LSTM_REFERENCE_LENGTHS if l > t) for t in range(T)]
    return np.concatenate([gates[:, t, :cov[t]].reshape(-1) for t in range(T)])


def test_highway_lstm_eval_and_drop_in_symbol_vs_reference_kernel(cuda):
    """highway_lstm_forward_ongpu of this library vs the oracle and vs what the reference's (cuBLAS-based) kernels
    compiled unmodified computed on the same inputs (tests/golden/make_golden_kernels.py): h and c whole, the covered
    gate rows on a seeded sample."""
    import motifs_cabi as C
    T, B, In, H, L = LSTM_REFERENCE_DIMS
    w, bias, x, drop = lstm_reference_case(cuda)
    h1, c1, g1 = lstm_launch(C.load(), None, w, bias, x, drop)
    out_o, h_o, c_o, g_o = oracle_lstm(x.cpu(), LSTM_REFERENCE_LENGTHS, w.cpu(), bias.cpu(), drop.cpu(), H, L,
                                       return_all=True)
    np.testing.assert_allclose(h1, h_o.numpy(), rtol=1e-4, atol=2e-5)
    np.testing.assert_allclose(c1, c_o.numpy(), rtol=1e-4, atol=2e-5)
    np.testing.assert_allclose(g1, g_o.numpy(), rtol=1e-4, atol=2e-5)
    gold = np.load(REF_KERNELS_GOLDEN)
    np.testing.assert_allclose(h1, gold["lstm_h"], rtol=1e-4, atol=2e-5)
    np.testing.assert_allclose(c1, gold["lstm_c"], rtol=1e-4, atol=2e-5)
    cg = lstm_covered_gates(g1)
    np.testing.assert_allclose(cg[golden_sample(cg.size, gold["lstm_gates_sample"].size, 3)], gold["lstm_gates_sample"],
                               rtol=1e-4, atol=2e-5)


# ------------------------------------------------------------------------------- train-time assignments
def _synthetic_detections(rng, num_im=3, per_im=30, gt_per_im=8):
    gt_boxes, gt_classes, gt_rels, rois, labels, im_inds = [], [], [], [], [], []
    for im in range(num_im):
        gb = rand_boxes(rng, gt_per_im, lo=40, hi=250)
        gc = rng.randint(1, 151, gt_per_im)
        gt_boxes.append(gb); gt_classes.append(np.stack([np.full(gt_per_im, im), gc], 1))
        pairs = [(a, b) for a in range(gt_per_im) for b in range(gt_per_im) if a != b]
        sel = rng.choice(len(pairs), 6, replace=False)
        gt_rels.append(np.array([[im, pairs[k][0], pairs[k][1], rng.randint(1, 51)] for k in sel]))
        # detections: jittered copies of GT boxes (matching labels) + random boxes (label 0)
        src = rng.randint(0, gt_per_im, per_im // 2)
        jit = gb[src] + rng.uniform(-6, 6, (per_im // 2, 4)).astype(np.float32)
        rnd = rand_boxes(rng, per_im - per_im // 2, lo=30, hi=200)
        rois.append(np.concatenate([jit, rnd]).astype(np.float32))
        labels.append(np.concatenate([gc[src], np.zeros(per_im - per_im // 2, np.int64)]))
        im_inds.append(np.full(per_im, im))
    return (np.concatenate(im_inds), np.concatenate(rois), np.concatenate(labels).astype(np.int64),
            np.concatenate(gt_boxes).astype(np.float32), np.concatenate(gt_classes).astype(np.int64),
            np.concatenate(gt_rels).astype(np.int64))


def test_rel_assignments_identical_to_oracle(cuda):
    from lib.fpn.proposal_assignments.rel_assignments import rel_assignments
    from oracle import host
    rng = np.random.RandomState(21)
    im_inds, rois, labels, gt_boxes, gt_classes, gt_rels = _synthetic_detections(rng)
    for nspg, fno in [(1, True), (4, False)]:
        got = rel_assignments(torch.from_numpy(im_inds).to(cuda), torch.from_numpy(rois).to(cuda),
                              torch.from_numpy(labels).to(cuda), torch.from_numpy(gt_boxes).to(cuda),
                              torch.from_numpy(gt_classes).to(cuda), torch.from_numpy(gt_rels).to(cuda), 0,
                              num_sample_per_gt=nspg, filter_non_overlap=fno, rng=np.random.RandomState(5))
        exp = host.rel_assignments(im_inds, rois, labels, gt_boxes, gt_classes, gt_rels, 0, np.random.RandomState(5),
                                   num_sample_per_gt=nspg, filter_non_overlap=fno)
        assert got.dtype == torch.int64 and np.array_equal(got.cpu().numpy(), exp)


def test_proposal_assignments_det_identical_to_oracle(cuda):
    from lib.fpn.proposal_assignments.proposal_assignments_det import proposal_assignments_det
    from oracle import host
    rng = np.random.RandomState(22)
    im_inds, rois, labels, gt_boxes, gt_classes, gt_rels = _synthetic_detections(rng, num_im=2, per_im=400, gt_per_im=10)
    rois5 = np.concatenate([im_inds[:, None].astype(np.float32), rois], 1)
    r, l, t = proposal_assignments_det(torch.from_numpy(rois5).to(cuda), torch.from_numpy(gt_boxes).to(cuda),
                                       torch.from_numpy(gt_classes).to(cuda), 0, rng=np.random.RandomState(9))
    er, el, et = host.proposal_assignments_det(rois5, gt_boxes, gt_classes, 0, np.random.RandomState(9))
    assert np.array_equal(r.cpu().numpy(), er) and np.array_equal(l.cpu().numpy(), el) and np.array_equal(t.cpu().numpy(), et)


def test_maxpool3s2_matches_torch(cuda):
    from lib.get_union_boxes import _MaxPool3s2
    torch.manual_seed(0)
    for shape in [(3, 5, 14, 14), (2, 4, 27, 27), (1, 2, 7, 9)]:
        x = torch.randn(*shape, device=cuda).clamp_min(0).requires_grad_(True)   # post-ReLU: many tied zeros
        y = _MaxPool3s2.apply(x)
        ref_in = x.detach().clone().requires_grad_(True)
        ref = torch.nn.functional.max_pool2d(ref_in, 3, 2, 1)
        assert torch.equal(y, ref)
        g = torch.randn_like(ref)
        y.backward(g); ref.backward(g)
        assert torch.equal(x.grad, ref_in.grad)


# ------------------------------------------------------------------------------- RPN anchor targets (a13)
def test_anchor_target_layer_matches_reference_fixture(cuda, golden):
    """lib/fpn/anchor_targets.py:16-105 on the warp-per-anchor kernels vs the REFERENCE's own function run with the same
    numpy RNG state (tests/golden/make_golden.py): anchors, (h, w, A) indices, box targets and labels identical."""
    from lib.fpn.anchor_targets import anchor_target_layer
    np.random.seed(7)
    anchors, inds, targets, labels = anchor_target_layer(golden["at_gt"], (592, 592))
    assert np.array_equal(anchors, golden["at_anchors"])
    assert np.array_equal(inds, golden["at_inds"])
    assert np.array_equal(targets, golden["at_targets"])
    assert np.array_equal(labels, golden["at_labels"])


@pytest.mark.parametrize("G", [1, 7, 40, 97])
def test_anchor_labels_device_vs_oracle(cuda, G):
    """Labels before subsampling, first arg-max and max overlap vs the oracle (numpy float64) for GT counts that span
    one lane stride to several, including a GT box outside every anchor (its column maximum is 0: every anchor with a zero
    overlap 'attains' it, as in the reference, anchor_targets.py:57-58)."""
    from lib.fpn.anchor_targets import anchor_labels_device
    from oracle import host, ops
    rng = np.random.RandomState(G)
    ans = host.generate_anchors().reshape(-1, 4)
    inside = np.where((ans[:, 0] >= 0) & (ans[:, 1] >= 0) & (ans[:, 2] < 592) & (ans[:, 3] < 592))[0]
    good = ans[inside]
    x1 = rng.uniform(0, 450, G); y1 = rng.uniform(0, 450, G)
    gt = np.stack([x1, y1, np.minimum(x1 + rng.uniform(16, 300, G), 591), np.minimum(y1 + rng.uniform(16, 300, G), 591)], 1)
    gt = gt.astype(np.float32).astype(np.float64)
    if G >= 7:
        gt[3] = [5000, 5000, 5100, 5100]
        gt[5] = gt[2]                                  # duplicate GT box: arg-max must be the FIRST of the two
    labels, arg, mx = anchor_labels_device(torch.from_numpy(good).to(cuda), torch.from_numpy(gt).to(cuda))
    ov = ops.bbox_overlaps_f64(good, gt)
    want_arg = ov.argmax(1)
    want_mx = ov[np.arange(len(good)), want_arg]
    want = -np.ones(len(good), dtype=np.int64)
    want[want_mx < 0.3] = 0
    want[np.where(ov == ov.max(0)[None])[0]] = 1
    want[want_mx >= 0.7] = 1
    assert np.array_equal(mx.cpu().numpy(), want_mx)
    assert np.array_equal(arg.cpu().numpy(), want_arg)
    assert np.array_equal(labels.cpu().numpy(), want)


# ------------------------------------------------------------------------------- decoder commitment (a9 / f3)
@pytest.mark.parametrize("N,seed", [(1, 0), (20, 1), (64, 2), (64, 3)])
def test_decoder_commit_kernel_identical_to_host_loop(cuda, N, seed):
    """lib/lstm/decoder_rnn.py:230-247 (overlap-aware greedy label commitment of SGDet eval) as one device kernel vs the
    reference's host loop restated with numpy: identical commitments, including exact ties of the probabilities (first
    arg-max in row-major order) and boxes that overlap the winner at IoU >= 0.3 in the winner's class."""
    import motifs_cabi as C
    from oracle import ops
    rng = np.random.RandomState(seed)
    Cn = 151
    x1 = rng.uniform(0, 300, (N, 1)); y1 = rng.uniform(0, 300, (N, 1))
    base = np.concatenate([x1, y1, x1 + rng.uniform(40, 250, (N, 1)), y1 + rng.uniform(40, 250, (N, 1))], 1)
    boxes = (base[:, None, :] + rng.randn(N, Cn, 4) * 6).astype(np.float32)            # class-specific refinements
    boxes[..., 2:] = np.maximum(boxes[..., 2:], boxes[..., :2] + 1)
    logits = rng.randn(N, Cn).astype(np.float32) * 3
    if seed == 3:                                                                      # exact ties
        logits = np.round(logits)
    probs = torch.softmax(torch.from_numpy(logits), 1).numpy()
    is_overlap = ops.nms_overlaps(boxes) >= np.float32(0.3)
    sampled = probs.copy(); sampled[:, 0] = 0
    want = np.zeros(N, dtype=np.int64)
    for _ in range(N):
        bi, ci = np.unravel_index(sampled.argmax(), sampled.shape)
        want[int(bi)] = int(ci)
        sampled[is_overlap[bi, :, ci], ci] = 0.0
        sampled[bi] = -1.0
    got = torch.empty(N, dtype=torch.long, device=cuda)
    b = torch.from_numpy(boxes).to(cuda); p = torch.from_numpy(probs).to(cuda)
    C.check(C.load().mb200_decoder_commit(C.ptr(b), C.ptr(p), N, Cn, 0.3, C.ptr(got), C.cur_stream()), "mb200_decoder_commit")
    assert np.array_equal(got.cpu().numpy(), want)


@pytest.mark.parametrize("T,B,In,H,L", [(6, 256, 40, 128, 2), (5, 200, 712, 512, 2), (4, 64, 33, 64, 1), (3, 130, 20, 192, 3)])
def test_highway_lstm_tensor_core_recurrence(cuda, T, B, In, H, L):
    """csrc/lstm_tc.cu (per-step [B,H] x [H,5H] on tcgen05, bf16x3, weight slices resident in shared memory; used for
    B >= 48) against the oracle and against the SIMT kernels on the same inputs: ragged lengths, both directions, training
    mode (gates saved, backward through the unchanged SIMT backward kernel)."""
    from torch.nn.utils.rnn import pack_padded_sequence, pad_packed_sequence
    import lib.lstm.highway_lstm_cuda.alternating_highway_lstm as AH
    assert AH.use_tensor_core_recurrence(H, B)
    lengths = sorted([max(1, T - (i * T) // B) for i in range(B)], reverse=True)
    lengths[0] = T
    rng = np.random.RandomState(T * 100 + B)
    m, x, drop = lstm_inputs(rng, T, B, In, H, L, lengths)
    gout = torch.randn(T, B, H)
    for b, l in enumerate(lengths):
        gout[l:, b] = 0
    mc = m.to(cuda).train()

    def run(tc):
        AH.TC_RECURRENCE = tc
        try:
            mc.zero_grad()
            xc = x.to(cuda).requires_grad_(True)
            out_p, _ = mc(pack_padded_sequence(xc, lengths), dropout_weights=drop.to(cuda))
            out_c, _ = pad_packed_sequence(out_p, total_length=T)
            (out_c * gout.to(cuda)).sum().backward()
            return out_c.detach().cpu(), xc.grad.cpu(), mc.weight.grad.detach().cpu().clone(), mc.bias.grad.detach().cpu().clone()
        finally:
            AH.TC_RECURRENCE = True
    o_tc, gx_tc, gw_tc, gb_tc = run(True)
    o_si, gx_si, gw_si, gb_si = run(False)
    np.testing.assert_allclose(o_tc.numpy(), o_si.numpy(), rtol=1e-4, atol=3e-5)
    scale = float(gw_si.abs().max())
    np.testing.assert_allclose(gx_tc.numpy(), gx_si.numpy(), rtol=1e-3, atol=2e-4)
    np.testing.assert_allclose(gw_tc.numpy(), gw_si.numpy(), rtol=1e-3, atol=2e-4 * max(1.0, scale))
    np.testing.assert_allclose(gb_tc.numpy(), gb_si.numpy(), rtol=1e-3, atol=2e-4 * max(1.0, scale))
    if B * T * H <= 256 * 6 * 128:                       # the oracle (CPU) on the smallest case
        out_o = oracle_lstm(x, lengths, m.weight.detach().cpu(), m.bias.detach().cpu(), drop, H, L)
        np.testing.assert_allclose(o_tc.numpy(), out_o.detach().numpy(), rtol=1e-4, atol=3e-5)
