"""GPU: the open-vocabulary tail on channels-last feature volumes.  Every call f(x) on a
channels_last_3d volume is compared with f(x.contiguous()) through the same public function, in
float32 and bfloat16: labels byte for byte, logits bit for bit (compared as int32, which covers
NaN payloads and the sign of zero)."""
import ctypes

import numpy as np
import pytest
import torch

from tests.test_tail_gpu import SIZES

pytestmark = pytest.mark.gpu
BF = torch.bfloat16
CL3 = torch.channels_last_3d
P = ctypes.c_void_p
VOCAB = {5: list(range(4)), 18: list(range(17)),
         67: [k for k, n in enumerate(SIZES) for _ in range(n)]}   # Q -> class reflection
DTYPES = [torch.float32, BF]


def _cls(Q):
    from veon_b200.tail import class_of_prompt
    return class_of_prompt(VOCAB[Q]).cuda()


def _case(B, C, Q, vol, seed, dtype):
    """a channels-last feature volume of `dtype`, float32 classifier and gate"""
    g = torch.Generator(device="cuda").manual_seed(seed)
    feat = (torch.sigmoid(torch.randn(B, C, *vol, device="cuda", generator=g)) - 0.5).to(dtype)
    w = torch.randn(Q, C, device="cuda", generator=g)
    w = 100.0 * w / w.norm(dim=1, keepdim=True)
    gate = torch.randn(B, 2, *vol, device="cuda", generator=g)
    return _to_cl(feat), w, gate


def _to_cl(x):
    x = x.contiguous(memory_format=CL3)
    assert not x.is_contiguous() and x.is_contiguous(memory_format=CL3)
    return x


def assert_bits_equal(got, want):
    assert got.dtype == want.dtype == torch.float32 and got.shape == want.shape
    assert got.is_contiguous() and want.is_contiguous()
    gi, wi = got.view(torch.int32), want.view(torch.int32)
    assert torch.equal(gi, wi), int((gi != wi).sum())


def _argmax_both(feat, w, cls, gate, free_label=17):
    from veon_b200.tail import voxel_text_argmax
    got = voxel_text_argmax(feat, w, cls, gate, free_label)
    want = voxel_text_argmax(feat.contiguous(), w, cls, gate, free_label)
    torch.cuda.synchronize()
    return got, want


def _logits_both(w, feat):
    from veon_b200.tail import semantic_inference_3d
    got = semantic_inference_3d(w, feat)
    want = semantic_inference_3d(w, feat.contiguous())
    torch.cuda.synchronize()
    return got, want


def _entry_rc(feat, w, cls, gate):
    """return code of veon_voxel_text_argmax_cl / _cl_bf16 itself (0 when its kernel ran)"""
    from veon_b200 import _lib
    lib = _lib.load()
    B, C, Z, Y, X = feat.shape
    fn = lib.veon_voxel_text_argmax_cl_bf16 if feat.dtype == BF else lib.veon_voxel_text_argmax_cl
    labels = torch.empty((B, X, Y, Z), dtype=torch.uint8, device="cuda")
    rc = fn(P(feat.data_ptr()), P(w.data_ptr()), P(cls.data_ptr()), P(gate.data_ptr()), B, C,
            w.shape[0], Z, Y, X, 17, P(labels.data_ptr()), None,
            P(torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return rc


# full volume; V % 128 != 0 with V % 8 == 0; V % 128 != 0 with V % 8 == 4
SHAPES = [(1, (16, 200, 200)), (2, (2, 10, 12)), (2, (3, 10, 10))]


# ---------------------------------------------------------------- tensor-core path
@pytest.mark.parametrize("B,vol", SHAPES)
@pytest.mark.parametrize("Q", [5, 18, 67])
@pytest.mark.parametrize("C", [64, 512])
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "bf16"])
def test_labels_equal_the_contiguous_route(dtype, C, Q, B, vol):
    feat, w, gate = _case(B, C, Q, vol, seed=C + Q + B, dtype=dtype)
    cls = _cls(Q)
    assert _entry_rc(feat, w, cls, gate) == 0
    got, want = _argmax_both(feat, w, cls, gate)
    assert got.dtype == torch.uint8 and got.shape == (B, vol[2], vol[1], vol[0])
    assert torch.equal(got, want), int((got != want).sum())
    assert 0.2 < float((got != 17).float().mean()) < 0.8


@pytest.mark.parametrize("B,vol", SHAPES)
@pytest.mark.parametrize("Q", [5, 18, 67])
@pytest.mark.parametrize("C", [64, 512])
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "bf16"])
def test_logits_equal_the_contiguous_route(dtype, C, Q, B, vol):
    feat, w, _ = _case(B, C, Q, vol, seed=C * Q + B, dtype=dtype)
    got, want = _logits_both(w, feat)
    assert got.shape == (B, Q, *vol)
    assert_bits_equal(got, want)


def test_bf16_v8_remainder_runs_natively_with_the_widened_bits():
    """V % 8 == 4: the channels-first bfloat16 call widens and runs float32 tcgen05; the
    channels-last call runs its own bfloat16 kernel and gives the same bits"""
    from veon_b200 import _lib
    C, Q = 64, 18
    feat, w, gate = _case(2, C, Q, (2, 2, 5), seed=3, dtype=BF)            # V = 20
    cls = _cls(Q)
    assert _entry_rc(feat, w, cls, gate) == 0
    contiguous = feat.contiguous()
    lib = _lib.load()
    B, _, Z, Y, X = feat.shape
    labels = torch.empty((B, X, Y, Z), dtype=torch.uint8, device="cuda")
    assert lib.veon_voxel_text_argmax_bf16(
        P(contiguous.data_ptr()), P(w.data_ptr()), P(cls.data_ptr()), P(gate.data_ptr()), B, C, Q,
        Z, Y, X, 17, P(labels.data_ptr()), None,
        P(torch.cuda.current_stream().cuda_stream)) == _lib.E_UNSUPPORTED
    got, want = _argmax_both(feat, w, cls, gate)
    assert torch.equal(got, want)
    assert_bits_equal(*_logits_both(w, feat))


@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "bf16"])
@pytest.mark.parametrize("C,Q", [(64, 18), (512, 67)])
def test_nan_and_inf_features(C, Q, dtype):
    B, vol = 2, (4, 10, 16)
    feat, w, gate = _case(B, C, Q, vol, seed=Q, dtype=dtype)
    gate[:, 0] = 1.0
    gate[:, 1] = 0.0                                   # occupied everywhere
    flat = feat.contiguous().view(B, C, -1)
    for k, val in enumerate((float("nan"), float("inf"), -float("inf"))):
        flat[0, 3 + k, 5 + 40 * k] = val
        flat[1, C - 1 - k, 639 - 7 * k] = val
    feat = _to_cl(flat.view(B, C, *vol))
    cls = _cls(Q)
    got, want = _argmax_both(feat, w, cls, gate, free_label=255)   # 17 is a class at Q >= 18
    assert torch.equal(got, want), int((got != want).sum())
    assert int((got == 255).sum()) == 6
    sem, sem_c = _logits_both(w, feat)
    assert_bits_equal(sem, sem_c)
    assert int((~torch.isfinite(sem)).any(dim=1).sum()) == 6


@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "bf16"])
@pytest.mark.parametrize("Q_per_class", [1, 3])
def test_ties_and_near_ties(Q_per_class, dtype):
    """exact ties between classes (first class wins) and logit gaps of 1e-6 .. 1e-3 relative"""
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
        feat = _to_cl((torch.sigmoid(torch.randn(B, C, *vol, generator=g)) - 0.5).cuda().to(dtype))
        got, want = _argmax_both(feat, w, cls, gate)
        assert torch.equal(got, want), (eps, int((got != want).sum()))
        assert_bits_equal(*_logits_both(w, feat))
        w[Q_per_class] = w[0]                          # class 1 ties class 0 exactly
        got, want = _argmax_both(feat, w, cls, gate)
        assert torch.equal(got, want), (eps, int((got != want).sum()))
        if Q_per_class == 1:
            assert not bool((got == 1).any())          # the first of two equal classes wins
    zero = _to_cl(torch.zeros(B, C, *vol, device="cuda", dtype=dtype))   # every logit 0: class 0
    got, want = _argmax_both(zero, w, cls, gate)
    assert torch.equal(got, want) and bool((got == 0).all())
    assert_bits_equal(*_logits_both(w, zero))


# ---------------------------------------------------------------- routes the kernel does not take
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "bf16"])
@pytest.mark.parametrize("C,Q,vol", [(30, 18, (4, 10, 16)),     # C % 32 != 0
                                     (64, 130, (4, 10, 16)),    # Q > 128
                                     (64, 18, (3, 5, 7))])      # V % 4 != 0
def test_ffma_shapes_are_copied(C, Q, vol, dtype):
    from veon_b200 import _lib
    from veon_b200.tail import class_of_prompt
    feat, w, gate = _case(2, C, Q, vol, seed=C + Q, dtype=dtype)
    cls = class_of_prompt(list(range(Q - 1))).cuda()
    assert _entry_rc(feat, w, cls, gate) == _lib.E_UNSUPPORTED
    got, want = _argmax_both(feat, w, cls, gate)
    assert torch.equal(got, want)
    assert_bits_equal(*_logits_both(w, feat))


@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "bf16"])
def test_misaligned_volume_is_copied(dtype):
    """a channels-last view 4 bytes past a 16-byte line"""
    from veon_b200 import _lib
    B, C, Q, vol = 2, 64, 18, (4, 10, 16)
    src, w, gate = _case(B, C, Q, vol, seed=4, dtype=dtype)
    off = 4 // src.element_size()
    store = torch.empty(src.numel() + off, dtype=dtype, device="cuda")
    feat = store[off:].view(B, *vol, C).permute(0, 4, 1, 2, 3)
    feat.copy_(src)
    assert feat.is_contiguous(memory_format=CL3) and not feat.is_contiguous()
    assert feat.data_ptr() % 16 == 4
    cls = _cls(Q)
    assert _entry_rc(feat, w, cls, gate) == _lib.E_UNSUPPORTED
    got, want = _argmax_both(feat, w, cls, gate)
    assert torch.equal(got, want)
    assert torch.equal(got, _argmax_both(src, w, cls, gate)[0])
    assert_bits_equal(*_logits_both(w, feat))


# ---------------------------------------------------------------- decoder resolution
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "bf16"])
@pytest.mark.parametrize("Q,B,vol,occ", [(18, 2, (8, 100, 100), (16, 200, 200)),
                                         (67, 2, (8, 100, 100), (16, 200, 200)),
                                         (18, 2, (2, 10, 14), (4, 20, 28))])   # V % 128 != 0
def test_lowres_route_equals_the_contiguous_route(Q, B, vol, occ, dtype):
    from veon_b200.tail import voxel_text_argmax_lowres
    feat, w, gate = _case(B, 512, Q, vol, seed=Q, dtype=dtype)
    cls = _cls(Q)
    got = voxel_text_argmax_lowres(feat, w, cls, gate, occ_size=occ)
    want = voxel_text_argmax_lowres(feat.contiguous(), w, cls, gate, occ_size=occ)
    torch.cuda.synchronize()
    assert got.shape == (B, occ[2], occ[1], occ[0])
    assert torch.equal(got, want), int((got != want).sum())
    assert 0.2 < float((got != 17).float().mean()) < 0.8


# ---------------------------------------------------------------- no contiguous copy
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "bf16"])
def test_channels_last_call_makes_no_copy(dtype):
    from veon_b200.tail import semantic_inference_3d, voxel_text_argmax, voxel_text_argmax_lowres
    feat, w, gate = _case(1, 512, 18, (16, 200, 200), seed=5, dtype=dtype)
    cls = _cls(18)
    nbytes = feat.numel() * feat.element_size()

    def grown(fn):
        fn()                                           # warm-up: the classifier image buffer
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        fn()
        torch.cuda.synchronize()
        return torch.cuda.max_memory_allocated() - base

    assert grown(lambda: voxel_text_argmax(feat, w, cls, gate)) < nbytes // 8
    logits_bytes = 18 * 16 * 200 * 200 * 4             # the returned logits
    assert grown(lambda: semantic_inference_3d(w, feat)) < logits_bytes + nbytes // 8
    lr, lr_w, lr_gate = _case(2, 512, 18, (8, 100, 100), seed=6, dtype=dtype)
    ws = torch.empty(2 * 18 * 8 * 100 * 100, dtype=torch.float32, device="cuda")
    lr_bytes = lr.numel() * lr.element_size()
    assert grown(lambda: voxel_text_argmax_lowres(lr, lr_w, cls, lr_gate, workspace=ws)) < \
        lr_bytes // 8


# ---------------------------------------------------------------- prepared classifier image
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "bf16"])
def test_prepared_classifier_image_and_null_agree(dtype):
    from veon_b200 import _lib
    lib = _lib.load()
    B, C, Q, (Z, Y, X) = 2, 256, 67, (4, 30, 52)
    feat, w, gate = _case(B, C, Q, (Z, Y, X), seed=11, dtype=dtype)
    cls = _cls(Q)
    sfx = "_cl_bf16" if dtype == BF else "_cl"
    st = P(torch.cuda.current_stream().cuda_stream)
    need = lib.veon_text_classifier_image_bytes(Q, C)
    image = torch.empty(need, dtype=torch.uint8, device="cuda")
    assert lib.veon_text_classifier_image(P(w.data_ptr()), Q, C, P(image.data_ptr()), need, st) == 0
    labels = [torch.empty((B, X, Y, Z), dtype=torch.uint8, device="cuda") for _ in range(2)]
    logits = [torch.empty((B, Q, Z, Y, X), device="cuda") for _ in range(2)]
    for out, img in ((labels[0], P(image.data_ptr())), (labels[1], None)):
        assert getattr(lib, "veon_voxel_text_argmax" + sfx)(
            P(feat.data_ptr()), P(w.data_ptr()), P(cls.data_ptr()), P(gate.data_ptr()), B, C, Q,
            Z, Y, X, 17, P(out.data_ptr()), img, st) == 0
    for out, img in ((logits[0], P(image.data_ptr())), (logits[1], None)):
        assert getattr(lib, "veon_semantic_inference_3d" + sfx)(
            P(w.data_ptr()), P(feat.data_ptr()), B, C, Q, Z, Y, X, P(out.data_ptr()), img, st) == 0
    torch.cuda.synchronize()
    assert torch.equal(labels[0], labels[1])
    assert_bits_equal(logits[0], logits[1])
    got, want = _argmax_both(feat, w, cls, gate)
    assert torch.equal(labels[0], want)
    assert_bits_equal(logits[0], _logits_both(w, feat)[1])


# ---------------------------------------------------------------- CUDA graph
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "bf16"])
def test_channels_last_call_in_a_cuda_graph(dtype):
    from veon_b200.tail import voxel_text_argmax
    feat, w, gate = _case(2, 512, 67, (4, 40, 50), seed=7, dtype=dtype)
    cls = _cls(67)
    eager = voxel_text_argmax(feat.contiguous(), w, cls, gate)
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
    assert torch.equal(out, voxel_text_argmax(feat.contiguous(), w, cls, gate))


# ---------------------------------------------------------------- end to end
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "bf16"])
def test_channels_last_neck_volume_feeds_the_tail(dtype):
    """LSSViewTransformer(memory_format=channels_last_3d)'s volume straight into the tail"""
    from tests.test_channels_last_gpu import _neck_inputs
    from veon_b200 import synthetic as S
    from veon_b200.view_transformer import LSSViewTransformer
    cfg = S.CONFIGS["small"]
    B, C, Q = 2, 64, 18
    img, metas, depth, feat = _neck_inputs(cfg, B, C, seed=8)
    neck = LSSViewTransformer(cfg.grid_config, cfg.input_size, cfg.downsample, 8, C,
                              collapse_z=False, memory_format=CL3, dtype=dtype)
    vol = neck.view_transform([img] + metas, depth, feat * 0.05)[0]
    assert vol.dtype == dtype and vol.shape == (B, C, 16, 200, 200)
    assert vol.is_contiguous(memory_format=CL3) and not vol.is_contiguous()
    g = torch.Generator(device="cuda").manual_seed(9)
    w = torch.randn(Q, C, device="cuda", generator=g)
    w = 100.0 * w / w.norm(dim=1, keepdim=True)
    gate_w = torch.randn(2, C, device="cuda", generator=g)
    gate = torch.einsum("kc,bczyx->bkzyx", gate_w, vol.float()).contiguous()
    got, want = _argmax_both(vol, w, _cls(Q), gate)
    assert torch.equal(got, want), int((got != want).sum())
    assert 0.001 < float((got != 17).float().mean()) < 0.9
    assert_bits_equal(*_logits_both(w, vol))
