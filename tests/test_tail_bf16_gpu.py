"""GPU: the open-vocabulary tail on bfloat16 feature volumes.  Every bfloat16 call f(x) is
compared with f(x.float()), the float32 route it stands in for: labels byte for byte, logits value
for value with the same NaN positions."""
import ctypes

import numpy as np
import pytest
import torch

from tests.test_tail_gpu import SIZES

pytestmark = pytest.mark.gpu
BF = torch.bfloat16
P = ctypes.c_void_p
VOCAB = {5: list(range(4)), 18: list(range(17)),
         67: [k for k, n in enumerate(SIZES) for _ in range(n)]}   # Q -> class reflection


def _cls(Q):
    from veon_b200.tail import class_of_prompt
    return class_of_prompt(VOCAB[Q]).cuda()


def _case(B, C, Q, vol, seed):
    """bfloat16 features, float32 classifier and gate, generated on the device"""
    g = torch.Generator(device="cuda").manual_seed(seed)
    feat = (torch.sigmoid(torch.randn(B, C, *vol, device="cuda", generator=g)) - 0.5).to(BF)
    w = torch.randn(Q, C, device="cuda", generator=g)
    w = 100.0 * w / w.norm(dim=1, keepdim=True)
    gate = torch.randn(B, 2, *vol, device="cuda", generator=g)
    return feat, w, gate


def assert_logits_equal(got, want):
    """equal value for value (an exact zero may differ in sign) with the same NaN positions"""
    na, nb = torch.isnan(got), torch.isnan(want)
    assert torch.equal(na, nb), int((na != nb).sum())
    assert torch.equal(got.masked_fill(na, 0), want.masked_fill(nb, 0)), \
        float((got.masked_fill(na, 0) - want.masked_fill(nb, 0)).abs().max())


def _argmax_both(feat, w, cls, gate, free_label=17):
    from veon_b200.tail import voxel_text_argmax
    got = voxel_text_argmax(feat, w, cls, gate, free_label)
    want = voxel_text_argmax(feat.float(), w, cls, gate, free_label)
    torch.cuda.synchronize()
    return got, want


def _entry_rc(feat, w, cls, gate):
    """return code of veon_voxel_text_argmax_bf16 itself (0 when a kernel of its own ran)"""
    from veon_b200 import _lib
    lib = _lib.load()
    B, C, Z, Y, X = feat.shape
    labels = torch.empty((B, X, Y, Z), dtype=torch.uint8, device="cuda")
    rc = lib.veon_voxel_text_argmax_bf16(P(feat.data_ptr()), P(w.data_ptr()), P(cls.data_ptr()),
                                         P(gate.data_ptr()), B, C, w.shape[0], Z, Y, X, 17,
                                         P(labels.data_ptr()), None,
                                         P(torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return rc


SHAPES = [(1, (16, 200, 200)), (2, (2, 10, 12)), (2, (3, 7, 8))]   # full volume; V % 128 != 0


# ---------------------------------------------------------------- 1, 2: tensor-core path
@pytest.mark.parametrize("B,vol", SHAPES)
@pytest.mark.parametrize("Q", [5, 18, 67])
@pytest.mark.parametrize("C", [64, 512])
def test_labels_equal_the_widened_route(C, Q, B, vol):
    feat, w, gate = _case(B, C, Q, vol, seed=C + Q + B)
    cls = _cls(Q)
    assert _entry_rc(feat, w, cls, gate) == 0
    got, want = _argmax_both(feat, w, cls, gate)
    assert got.dtype == torch.uint8 and got.shape == (B, vol[2], vol[1], vol[0])
    assert torch.equal(got, want), int((got != want).sum())
    assert 0.2 < float((got != 17).float().mean()) < 0.8


@pytest.mark.parametrize("B,vol", SHAPES)
@pytest.mark.parametrize("Q", [5, 18, 67])
@pytest.mark.parametrize("C", [64, 512])
def test_logits_equal_the_widened_route(C, Q, B, vol):
    from veon_b200.tail import semantic_inference_3d
    feat, w, _ = _case(B, C, Q, vol, seed=C * Q + B)
    got = semantic_inference_3d(w, feat)
    want = semantic_inference_3d(w, feat.float())
    torch.cuda.synchronize()
    assert got.dtype == torch.float32 and got.shape == (B, Q, *vol)
    assert_logits_equal(got, want)


@pytest.mark.parametrize("C,Q", [(64, 18), (512, 67), (30, 18)])
def test_nan_and_inf_features(C, Q):
    """NaN, +inf and -inf in the features: the labels of those voxels are free, and the logits
    have NaN exactly where the float32 route has it (tensor-core and FFMA paths)"""
    from veon_b200.tail import semantic_inference_3d
    B, vol = 2, (4, 10, 16)
    feat, w, gate = _case(B, C, Q, vol, seed=Q)
    gate[:, 0] = 1.0
    gate[:, 1] = 0.0                                   # occupied everywhere
    flat = feat.view(B, C, -1)
    for k, val in enumerate((float("nan"), float("inf"), -float("inf"))):
        flat[0, 3 + k, 5 + 40 * k] = val
        flat[1, C - 1 - k, 639 - 7 * k] = val
    cls = _cls(Q)
    got, want = _argmax_both(feat, w, cls, gate, free_label=255)   # 17 is a class at Q >= 18
    assert torch.equal(got, want), int((got != want).sum())
    assert int((got == 255).sum()) == 6
    sem, sem32 = semantic_inference_3d(w, feat), semantic_inference_3d(w, feat.float())
    assert_logits_equal(sem, sem32)
    assert int((~torch.isfinite(sem)).any(dim=1).sum()) == 6


@pytest.mark.parametrize("Q_per_class", [1, 3])
def test_ties_and_near_ties(Q_per_class):
    """exact ties between classes (first class wins) and the near-tie construction of
    test_near_tie_labels on bfloat16 features: logit gaps of 1e-6 .. 1e-3 relative"""
    from veon_b200.tail import class_of_prompt
    C, B, vol, n_cls = 512, 2, (4, 40, 50), 6
    refl = [k for k in range(n_cls) for _ in range(Q_per_class)]
    cls = class_of_prompt(refl).cuda()
    gate = torch.zeros(B, 2, *vol, device="cuda")
    gate[:, 0] = 1.0
    for eps in (1e-6, 1e-5, 1e-4, 1e-3):
        g = torch.Generator().manual_seed(int(-np.log10(eps)) * 10 + Q_per_class)
        base = torch.randn(1, C, generator=g)
        rows = base + eps * base.norm() * torch.nn.functional.normalize(
            torch.randn(n_cls * Q_per_class + 1, C, generator=g), dim=1)
        w = (100.0 * rows / rows.norm(dim=1, keepdim=True)).float().cuda()
        feat = (torch.sigmoid(torch.randn(B, C, *vol, generator=g)) - 0.5).cuda().to(BF)
        got, want = _argmax_both(feat, w, cls, gate)
        assert torch.equal(got, want), (eps, int((got != want).sum()))
        w[Q_per_class] = w[0]                          # class 1 ties class 0 exactly
        got, want = _argmax_both(feat, w, cls, gate)
        assert torch.equal(got, want), (eps, int((got != want).sum()))
        if Q_per_class == 1:
            assert not bool((got == 1).any())          # the first of two equal classes wins
    zero = torch.zeros(B, C, *vol, device="cuda", dtype=BF)    # every logit 0: class 0
    got, want = _argmax_both(zero, w, cls, gate)
    assert torch.equal(got, want) and bool((got == 0).all())


# ---------------------------------------------------------------- 3: routes
@pytest.mark.parametrize("C,Q,vol", [(30, 18, (4, 10, 16)),     # C % 32 != 0
                                     (64, 130, (4, 10, 16)),    # Q > 128
                                     (64, 18, (3, 5, 7))])      # V % 4 != 0
def test_ffma_shapes_take_the_bf16_ffma_kernel(C, Q, vol):
    from veon_b200.tail import class_of_prompt, semantic_inference_3d
    feat, w, gate = _case(2, C, Q, vol, seed=C + Q)
    cls = class_of_prompt(list(range(Q - 1))).cuda()
    assert _entry_rc(feat, w, cls, gate) == 0
    got, want = _argmax_both(feat, w, cls, gate)
    assert torch.equal(got, want)
    assert_logits_equal(semantic_inference_3d(w, feat), semantic_inference_3d(w, feat.float()))


def test_loader_misfits_are_widened_in_python():
    """V % 8 == 4, and a bfloat16 view 8- but not 16-byte aligned: the bfloat16 entry returns
    VEON_E_UNSUPPORTED and the Python layer takes the float32 route"""
    from veon_b200 import _lib
    from veon_b200.tail import semantic_inference_3d
    C, Q = 64, 18
    cls = _cls(Q)
    feat, w, gate = _case(2, C, Q, (2, 2, 5), seed=1)               # V = 20
    assert _entry_rc(feat, w, cls, gate) == _lib.E_UNSUPPORTED
    got, want = _argmax_both(feat, w, cls, gate)
    assert torch.equal(got, want)
    assert_logits_equal(semantic_inference_3d(w, feat), semantic_inference_3d(w, feat.float()))
    vol = (4, 10, 16)
    src, w, gate = _case(2, C, Q, vol, seed=2)
    store = torch.empty(src.numel() + 4, dtype=BF, device="cuda")
    feat = store[4:].view(src.shape)                                 # 8 bytes past a 16-byte line
    feat.copy_(src)
    assert feat.is_contiguous() and feat.data_ptr() % 16 == 8
    assert _entry_rc(feat, w, cls, gate) == _lib.E_UNSUPPORTED
    got, want = _argmax_both(feat, w, cls, gate)
    assert torch.equal(got, want)
    assert torch.equal(got, _argmax_both(src, w, cls, gate)[0])
    assert_logits_equal(semantic_inference_3d(w, feat), semantic_inference_3d(w, src.float()))


# ---------------------------------------------------------------- 4: decoder resolution
@pytest.mark.parametrize("Q", [18, 67])
def test_lowres_route_equals_the_widened_route(Q):
    from veon_b200.tail import voxel_text_argmax_lowres
    feat, w, gate = _case(2, 512, Q, (8, 100, 100), seed=Q)
    cls = _cls(Q)
    got = voxel_text_argmax_lowres(feat, w, cls, gate, occ_size=(16, 200, 200))
    want = voxel_text_argmax_lowres(feat.float(), w, cls, gate, occ_size=(16, 200, 200))
    torch.cuda.synchronize()
    assert got.shape == (2, 200, 200, 16)
    assert torch.equal(got, want), int((got != want).sum())
    assert 0.2 < float((got != 17).float().mean()) < 0.8


# ---------------------------------------------------------------- 5: no widening copy
def test_bf16_call_makes_no_float32_copy():
    from veon_b200.tail import voxel_text_argmax
    feat, w, gate = _case(1, 512, 18, (16, 200, 200), seed=5)
    cls = _cls(18)
    voxel_text_argmax(feat, w, cls, gate)              # warm-up: the classifier image buffer
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    voxel_text_argmax(feat, w, cls, gate)
    torch.cuda.synchronize()
    grown = torch.cuda.max_memory_allocated() - base
    assert grown < feat.numel() * 2, grown             # a float32 copy would be numel * 4


# ---------------------------------------------------------------- 6: prepared classifier image
def test_prepared_classifier_image_and_null_agree():
    from veon_b200 import _lib
    lib = _lib.load()
    B, C, Q, (Z, Y, X) = 2, 256, 67, (4, 30, 52)
    feat, w, gate = _case(B, C, Q, (Z, Y, X), seed=11)
    cls = _cls(Q)
    st = P(torch.cuda.current_stream().cuda_stream)
    need = lib.veon_text_classifier_image_bytes(Q, C)
    image = torch.empty(need, dtype=torch.uint8, device="cuda")
    assert lib.veon_text_classifier_image(P(w.data_ptr()), Q, C, P(image.data_ptr()), need, st) == 0
    labels = [torch.empty((B, X, Y, Z), dtype=torch.uint8, device="cuda") for _ in range(2)]
    logits = [torch.empty((B, Q, Z, Y, X), device="cuda") for _ in range(2)]
    for out, img in ((labels[0], P(image.data_ptr())), (labels[1], None)):
        assert lib.veon_voxel_text_argmax_bf16(P(feat.data_ptr()), P(w.data_ptr()), P(cls.data_ptr()),
                                               P(gate.data_ptr()), B, C, Q, Z, Y, X, 17,
                                               P(out.data_ptr()), img, st) == 0
    for out, img in ((logits[0], P(image.data_ptr())), (logits[1], None)):
        assert lib.veon_semantic_inference_3d_bf16(P(w.data_ptr()), P(feat.data_ptr()), B, C, Q, Z,
                                                   Y, X, P(out.data_ptr()), img, st) == 0
    torch.cuda.synchronize()
    assert torch.equal(labels[0], labels[1])
    assert_logits_equal(logits[0], logits[1])
    got, want = _argmax_both(feat, w, cls, gate)
    assert torch.equal(labels[0], want)


# ---------------------------------------------------------------- 7: CUDA graph
def test_bf16_call_in_a_cuda_graph():
    from veon_b200.tail import voxel_text_argmax
    feat, w, gate = _case(2, 512, 67, (4, 40, 50), seed=7)
    cls = _cls(67)
    eager = voxel_text_argmax(feat, w, cls, gate)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        voxel_text_argmax(feat, w, cls, gate)          # warm-up on the capture stream
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = voxel_text_argmax(feat, w, cls, gate)
    out.fill_(255)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, eager)
    feat.copy_(feat.flip(-1))                          # new inputs, same buffers
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, voxel_text_argmax(feat, w, cls, gate))


# ---------------------------------------------------------------- 8: end to end
def test_bf16_neck_volume_feeds_the_tail():
    """LSSViewTransformer(dtype=bfloat16)'s volume straight into the tail: the labels of the same
    volume widened"""
    from tests.test_channels_last_gpu import _neck_inputs
    from veon_b200 import synthetic as S
    from veon_b200.tail import semantic_inference_3d
    from veon_b200.view_transformer import LSSViewTransformer
    cfg = S.CONFIGS["small"]
    B, C, Q = 2, 64, 18
    img, metas, depth, feat = _neck_inputs(cfg, B, C, seed=8)
    neck = LSSViewTransformer(cfg.grid_config, cfg.input_size, cfg.downsample, 8, C,
                              collapse_z=False, dtype=BF)
    vol = neck.view_transform([img] + metas, depth, feat * 0.05)[0]
    assert vol.dtype == BF and vol.shape == (B, C, 16, 200, 200)
    g = torch.Generator(device="cuda").manual_seed(9)
    w = torch.randn(Q, C, device="cuda", generator=g)
    w = 100.0 * w / w.norm(dim=1, keepdim=True)
    gate_w = torch.randn(2, C, device="cuda", generator=g)
    gate = torch.einsum("kc,bczyx->bkzyx", gate_w, vol.float())
    got, want = _argmax_both(vol, w, _cls(Q), gate)
    assert torch.equal(got, want), int((got != want).sum())
    assert 0.001 < float((got != 17).float().mean()) < 0.9
    assert_logits_equal(semantic_inference_3d(w, vol), semantic_inference_3d(w, vol.float()))
