"""Open-vocabulary classification tail on libveonlift.

Mirrors three reference sites (SURVEY.md 8a rows a13-a15) as ONE fused call:

    semantic_inference_3d(ov_classifier_weight, feat_occ)   san_in_veon_temporal.py:257-259
    _merge_classes_prob(sem_occ, dim=1, ...)                san_in_veon_entry_temporal.py:273-297
    simple_test label rule                                  veon_temporal.py:223-229,240

and, for the decoder-resolution route (SURVEY.md 8f-4), the two up-samplings in front of them
(san_in_veon_temporal.py:196-207): `voxel_text_argmax_lowres` classifies the low-resolution
volume and interpolates the Q logit channels instead of the C feature channels.
`semantic_inference_3d` is the reference method of that name on its own (logits out).

The three feature-volume entries read a bfloat16 volume as it is (the pooling's bfloat16 output,
or a 3D decoder's under autocast): half the bytes of the float32 copy they used to make, and the
same results as that float32 route, byte for byte for the labels and value for value for the
logits.  Other dtypes are widened to float32; the classifier and the gate always are.

A float32 or bfloat16 volume in `torch.channels_last_3d` (a 3D decoder running its conv3d in that
layout, or the pooling's channels-last output) is read as it is too, with the bits of the same
call on its contiguous copy; shapes the channels-last kernel does not take are copied first.
"""
import ctypes

import torch

from . import _lib
from ._lib import require_cuda, stream_ptr

__all__ = ["class_of_prompt", "voxel_text_argmax", "semantic_inference_3d", "classify_logits",
           "upsample_classify", "voxel_text_argmax_lowres", "prepare_vocabulary",
           "point_text_argmax"]


def class_of_prompt(class_reflection, mode="nuscenes", background=True):
    """Merged class id of each classifier row: contiguous runs of equal
    `class_reflection` form one class and the extra trailing background row is
    its own class (san_in_veon_entry_temporal.py:273-286).

    background=False: the grouping of the LOSS-side `_merge_classes_prob`
    (loss/occ_loss_utils/occ3d_nuscenes.py:249-265): no trailing row.

    mode: the reference moves the background/free class to index 0 for "semkitti"
    (san_in_veon_entry_temporal.py:288-293: `merged[0] = merged.pop(-1)`).  That re-ordering
    is not expressible as the non-decreasing row -> class map the fused kernels take, so only
    "nuscenes" is supported here and "semkitti" is refused instead of being silently wrong."""
    if mode != "nuscenes":
        raise NotImplementedError(
            "class_of_prompt: only mode='nuscenes' (free class last) is supported; the "
            "reference's semkitti branch moves the free class to index 0")
    refl = [int(v) for v in class_reflection]
    n = len(refl) + (1 if background else 0)
    last_mergeable = n - 2 if background else n - 1
    out = []
    k = 0
    i = 0
    while i < n:
        j = i
        while j < last_mergeable and refl[i] == refl[j + 1]:
            j += 1
        out.extend([k] * (j - i + 1))
        k += 1
        i = j + 1
    return torch.tensor(out, dtype=torch.int32)


def prepare_vocabulary(text_embeddings, bg_embed, logit_scale):
    """The classifier weight the tail multiplies with -- `SANInVeonTemporal.prepare_vocabulary`
    (san_in_veon_temporal.py:261-266) on top of `LearnableBgOvClassifier.
    get_classifier_by_vocabulary` (clip_utils/classifier.py:107-112):

        W = exp(logit_scale) * L2-normalise(cat([text_embeddings, bg_embed]), dim=-1), detached.

    text_embeddings [Q-1, C]: one row per prompt, what the CLIP text encoder + template
    averaging produced (open_clip, un-vendored: outside this path); bg_embed [1, C] the
    learnable background embedding; logit_scale the CLIP log-temperature (scalar tensor or
    float; exp(.) ~ 100).  Init-time only: plain torch ops, device-agnostic."""
    emb = torch.cat([torch.as_tensor(text_embeddings).float(),
                     torch.as_tensor(bg_embed).float().reshape(1, -1)], dim=0)
    emb = torch.nn.functional.normalize(emb, p=2, dim=-1)
    scale = torch.as_tensor(logit_scale, dtype=torch.float32, device=emb.device).exp()
    return (scale * emb).clone().detach()


def _features(t):
    """(volume, entry-point suffix): a bfloat16 volume is read as it is (contiguous bfloat16,
    the `_bf16` entries), anything else as float32"""
    t = t.detach()
    if t.dtype == torch.bfloat16:
        return t.contiguous(), "_bf16"
    return t.contiguous().float(), ""


def _channels_last(t):
    """a 5-D float32 / bfloat16 volume stored [B,Z,Y,X,C] (channels_last_3d, not contiguous)"""
    return (t.dim() == 5 and t.dtype in (torch.float32, torch.bfloat16) and not t.is_contiguous()
            and t.is_contiguous(memory_format=torch.channels_last_3d))


def _call_features(lib, name, feat, call):
    """call(entry, volume) on the volume's own dtype; where the bfloat16 entry returns
    VEON_E_UNSUPPORTED (the float32 route would take the tensor cores, whose bfloat16 loader
    needs V % 8 == 0 and a 16-byte aligned volume) the volume is widened and the float32 entry
    called, which is what the bfloat16 entry stands in for.

    A channels-last volume goes as it is to the `_cl` / `_cl_bf16` entry, which gives the bits of
    the contiguous route; where that entry returns VEON_E_UNSUPPORTED (a shape the channels-first
    call runs on the FFMA kernel, or a volume that is not 16-byte aligned) the volume is made
    contiguous in its own dtype and takes the route above."""
    feat = feat.detach()
    if _channels_last(feat):
        suffix = "_cl_bf16" if feat.dtype == torch.bfloat16 else "_cl"
        rc = call(getattr(lib, name + suffix), feat)
        if rc != _lib.E_UNSUPPORTED:
            _lib.check(rc, name + suffix)
            return
    feat, suffix = _features(feat)
    rc = call(getattr(lib, name + suffix), feat)
    if suffix and rc == _lib.E_UNSUPPORTED:
        suffix = ""
        rc = call(getattr(lib, name), feat.float())
    _lib.check(rc, name + suffix)


def voxel_text_argmax(feat_occ, ov_classifier_weight, prompt_class, bin_occ, free_label=17):
    """feat_occ [B,C,Z,Y,X] f32 or bf16, ov_classifier_weight [Q,C] f32, prompt_class
    [Q] int32 (from `class_of_prompt`), bin_occ [B,2,Z,Y,X] f32 ->
    uint8 occupancy labels [B,X,Y,Z] (free voxels = `free_label`).  A bfloat16 feat_occ is read
    without a float32 copy and gives the labels of `feat_occ.float()`.  A channels_last_3d
    feat_occ (float32 or bfloat16) is read without a contiguous copy where the tensor cores take
    the shape, and gives the labels of `feat_occ.contiguous()`."""
    require_cuda(feat_occ, ov_classifier_weight, prompt_class, bin_occ)
    lib = _lib.load()
    w = ov_classifier_weight.detach().contiguous().float()
    cls = prompt_class.contiguous().int()
    bin_occ = bin_occ.detach().contiguous().float()
    B, C, Z, Y, X = feat_occ.shape
    Q = w.shape[0]
    if w.shape[1] != C or cls.numel() != Q or tuple(bin_occ.shape) != (B, 2, Z, Y, X):
        raise ValueError("inconsistent tail shapes")
    dev = feat_occ.device
    with torch.cuda.device(dev):
        labels = torch.empty((B, X, Y, Z), dtype=torch.uint8, device=dev)
        image = _classifier_image(lib, w, dev)
        _call_features(lib, "veon_voxel_text_argmax", feat_occ, lambda fn, feat: fn(
            ctypes.c_void_p(feat.data_ptr()), ctypes.c_void_p(w.data_ptr()),
            ctypes.c_void_p(cls.data_ptr()), ctypes.c_void_p(bin_occ.data_ptr()),
            B, C, Q, Z, Y, X, int(free_label), ctypes.c_void_p(labels.data_ptr()),
            image, stream_ptr(dev)))
    return labels


_IMAGE_BUFFERS = {}


def _classifier_image(lib, w, dev):
    """The classifier in the tail kernel's tensor-core operand form
    (`veon_text_classifier_image`), rebuilt on the current stream into a buffer kept per
    (device, stream); None when the tensor-core path does not take the shape."""
    Q, C = w.shape
    need = lib.veon_text_classifier_image_bytes(int(Q), int(C))
    if need == 0:
        return None
    stream = torch.cuda.current_stream(dev)
    key = (dev.index, stream.cuda_stream)
    buf = _IMAGE_BUFFERS.get(key)
    if buf is None or buf.numel() < need:
        buf = torch.empty(need, dtype=torch.uint8, device=dev)
        _IMAGE_BUFFERS[key] = buf
    rc = lib.veon_text_classifier_image(ctypes.c_void_p(w.data_ptr()), int(Q), int(C),
                                        ctypes.c_void_p(buf.data_ptr()), ctypes.c_size_t(buf.numel()),
                                        ctypes.c_void_p(stream.cuda_stream))
    _lib.check(rc, "veon_text_classifier_image")
    return ctypes.c_void_p(buf.data_ptr())


def semantic_inference_3d(ov_classifier_weight, mask_pred):
    """`SANInVeonTemporal.semantic_inference_3d` (san_in_veon_temporal.py:257-259):
    einsum("qc,bczhw->bqzhw") of the [Q,C] classifier and a [B,C,Z,Y,X] volume -> [B,Q,Z,Y,X]
    f32 (no gradient: the reference's weight is a detached constant and this entry serves the
    inference route).  A bfloat16 volume is read without a float32 copy and gives the logits of
    `mask_pred.float()` (NaN where those are NaN; only the sign of an exact zero may differ).
    A channels_last_3d volume (float32 or bfloat16) is read without a contiguous copy where the
    tensor cores take the shape, and gives the logits of `mask_pred.contiguous()` bit for bit;
    the logits are contiguous [B,Q,Z,Y,X] either way."""
    require_cuda(ov_classifier_weight, mask_pred)
    lib = _lib.load()
    w = ov_classifier_weight.detach().contiguous().float()
    B, C, Z, Y, X = mask_pred.shape
    Q = w.shape[0]
    if w.shape[1] != C:
        raise ValueError("inconsistent tail shapes")
    dev = mask_pred.device
    with torch.cuda.device(dev):
        sem = torch.empty((B, Q, Z, Y, X), dtype=torch.float32, device=dev)
        image = _classifier_image(lib, w, dev)
        _call_features(lib, "veon_semantic_inference_3d", mask_pred, lambda fn, feat: fn(
            ctypes.c_void_p(w.data_ptr()), ctypes.c_void_p(feat.data_ptr()), B, C, Q, Z, Y, X,
            ctypes.c_void_p(sem.data_ptr()), image, stream_ptr(dev)))
    return sem


def _sample_contiguous(t):
    """float32 view whose samples are contiguous blocks (any batch stride), else a copy"""
    t = t.detach()
    if t.dtype != torch.float32:
        t = t.float()
    inner = 1
    for size, stride in zip(reversed(t.shape[1:]), reversed(t.stride()[1:])):
        if size != 1 and stride != inner:
            return t.contiguous()
        inner *= size
    if t.shape[0] > 1 and t.stride(0) < inner:
        return t.contiguous()
    return t


def classify_logits(sem_occ, bin_occ, prompt_class, free_label=17):
    """`_merge_classes_prob` + the label rule on ready-made logits
    (san_in_veon_entry_temporal.py:273-297, veon_temporal.py:223-229,240): sem_occ [B,Q,Z,Y,X],
    bin_occ [B,2,Z,Y,X] -> uint8 [B,X,Y,Z].  Channel slices of a larger volume are taken as
    they are (no copy)."""
    require_cuda(sem_occ, bin_occ, prompt_class)
    lib = _lib.load()
    sem = _sample_contiguous(sem_occ)
    gate = _sample_contiguous(bin_occ)
    cls = prompt_class.contiguous().int()
    B, Q, Z, Y, X = sem.shape
    if tuple(gate.shape) != (B, 2, Z, Y, X) or cls.numel() != Q:
        raise ValueError("inconsistent tail shapes")
    dev = sem.device
    with torch.cuda.device(dev):
        labels = torch.empty((B, X, Y, Z), dtype=torch.uint8, device=dev)
        rc = lib.veon_classify_logits(
            ctypes.c_void_p(sem.data_ptr()), sem.stride(0), ctypes.c_void_p(gate.data_ptr()),
            gate.stride(0), ctypes.c_void_p(cls.data_ptr()), B, Q, Z, Y, X, int(free_label),
            ctypes.c_void_p(labels.data_ptr()), stream_ptr(dev))
    _lib.check(rc, "veon_classify_logits")
    return labels


def upsample_classify(sem_occ_lr, bin_occ_lr, prompt_class, occ_size, free_label=17):
    """Low-resolution logits [B,Q,Zi,Yi,Xi] and gate [B,2,Zi,Yi,Xi] -> trilinear
    (align_corners=False) to `occ_size` = (Z,Y,X), class merge, arg-max, gate -> uint8 [B,X,Y,Z]."""
    require_cuda(sem_occ_lr, bin_occ_lr, prompt_class)
    lib = _lib.load()
    sem = sem_occ_lr.detach().contiguous().float()
    gate = bin_occ_lr.detach().contiguous().float()
    cls = prompt_class.contiguous().int()
    B, Q, Zi, Yi, Xi = sem.shape
    Z, Y, X = (int(v) for v in occ_size)
    if tuple(gate.shape) != (B, 2, Zi, Yi, Xi) or cls.numel() != Q:
        raise ValueError("inconsistent tail shapes")
    dev = sem.device
    with torch.cuda.device(dev):
        labels = torch.empty((B, X, Y, Z), dtype=torch.uint8, device=dev)
        rc = lib.veon_upsample_classify(
            ctypes.c_void_p(sem.data_ptr()), ctypes.c_void_p(gate.data_ptr()),
            ctypes.c_void_p(cls.data_ptr()), B, Q, Zi, Yi, Xi, Z, Y, X, int(free_label),
            ctypes.c_void_p(labels.data_ptr()), stream_ptr(dev))
    _lib.check(rc, "veon_upsample_classify")
    return labels


def voxel_text_argmax_lowres(feat_occ_lr, ov_classifier_weight, prompt_class, bin_occ_lr,
                             occ_size=(16, 200, 200), free_label=17, workspace=None):
    """The whole inference tail from the decoder's outputs (san_in_veon_temporal.py:196-208 +
    the merge and label rule): feat_occ_lr [B,C,Zi,Yi,Xi], bin_occ_lr [B,2,Zi,Yi,Xi] ->
    uint8 labels [B,X,Y,Z] on the `occ_size` grid.  `workspace`: optional float32 CUDA tensor of
    at least B*Q*Zi*Yi*Xi elements to hold the low-resolution logits (allocated if absent).
    A bfloat16 feat_occ_lr is read without a float32 copy and gives the labels of
    `feat_occ_lr.float()`; bin_occ_lr is taken as float32.  A channels_last_3d feat_occ_lr
    (float32 or bfloat16) is read without a contiguous copy where the tensor cores take the shape,
    and gives the labels of `feat_occ_lr.contiguous()`; bin_occ_lr is made contiguous."""
    require_cuda(feat_occ_lr, ov_classifier_weight, prompt_class, bin_occ_lr)
    lib = _lib.load()
    w = ov_classifier_weight.detach().contiguous().float()
    cls = prompt_class.contiguous().int()
    gate = bin_occ_lr.detach().contiguous().float()
    B, C, Zi, Yi, Xi = feat_occ_lr.shape
    Q = w.shape[0]
    Z, Y, X = (int(v) for v in occ_size)
    if w.shape[1] != C or cls.numel() != Q or tuple(gate.shape) != (B, 2, Zi, Yi, Xi):
        raise ValueError("inconsistent tail shapes")
    dev = feat_occ_lr.device
    need = lib.veon_voxel_text_argmax_lowres_workspace_bytes(B, Q, Zi, Yi, Xi)
    with torch.cuda.device(dev):
        if workspace is None:
            workspace = torch.empty(need // 4, dtype=torch.float32, device=dev)
        ws_bytes = workspace.numel() * workspace.element_size()
        labels = torch.empty((B, X, Y, Z), dtype=torch.uint8, device=dev)
        image = _classifier_image(lib, w, dev)
        _call_features(lib, "veon_voxel_text_argmax_lowres", feat_occ_lr, lambda fn, feat: fn(
            ctypes.c_void_p(feat.data_ptr()), ctypes.c_void_p(w.data_ptr()),
            ctypes.c_void_p(cls.data_ptr()), ctypes.c_void_p(gate.data_ptr()),
            B, C, Q, Zi, Yi, Xi, Z, Y, X, int(free_label), ctypes.c_void_p(labels.data_ptr()),
            ctypes.c_void_p(workspace.data_ptr()), ws_bytes, image, stream_ptr(dev)))
    return labels


def point_text_argmax(pred_feat, ov_classifier_weight, class_reflection):
    """The training-time voxel x text arg-max of `Proj2Dto3DLoss`
    (loss/occ_loss_utils/occ3d_nuscenes.py:472-482) for a POINT LIST:

        pred_probs_3d      = einsum('nc,dc->nd', pred_feat, ov_classifier_weight[:-1])
        pred_indices_3d    = max(pred_probs_3d, dim=1).indices
        pred_indices_3d_ds = max(_merge_classes_prob(pred_probs_3d, 1, class_reflection), 1).indices

    pred_feat [N, C] (rows = the selected voxels), ov_classifier_weight [Q, C] INCLUDING the
    trailing background row (dropped here, as the reference does), class_reflection: the Q-1
    class ids.  Returns (pred_indices_3d, pred_indices_3d_ds), int64 [N].  The [N, Q-1] logits
    are not returned (the reference uses them for nothing else).

    How: the point rows are turned into a [C, N] operand (own transpose kernel), the logits come
    from the tcgen05 3xTF32 kernel of the inference tail, one pass over them takes both
    arg-maxes."""
    require_cuda(pred_feat, ov_classifier_weight)
    lib = _lib.load()
    f = pred_feat.detach().contiguous().float()
    w = ov_classifier_weight.detach()[:-1].contiguous().float()
    N, C = f.shape
    Q = w.shape[0]
    if w.shape[1] != C or len(class_reflection) != Q:
        raise ValueError("inconsistent point_text_argmax shapes")
    dev = f.device
    cls = class_of_prompt(class_reflection, background=False).to(dev)
    with torch.cuda.device(dev):
        p_idx = torch.empty(N, dtype=torch.int64, device=dev)
        c_idx = torch.empty(N, dtype=torch.int64, device=dev)
        if N == 0:
            return p_idx, c_idx
        ldn = (N + 3) // 4 * 4                      # the tensor path wants V % 4 == 0
        ft = torch.zeros((C, ldn), dtype=torch.float32, device=dev) if ldn != N else \
            torch.empty((C, ldn), dtype=torch.float32, device=dev)
        if ldn == N:
            rc = lib.veon_transpose_batched(ctypes.c_void_p(f.data_ptr()), 1, N, C,
                                            ctypes.c_void_p(ft.data_ptr()), stream_ptr(dev))
            _lib.check(rc, "veon_transpose_batched")
        else:
            ft[:, :N] = f.t()
        logits = semantic_inference_3d(w, ft.view(1, C, 1, 1, ldn))      # [1, Q, 1, 1, ldn]
        rc = lib.veon_point_text_argmax(ctypes.c_void_p(logits.data_ptr()),
                                        ctypes.c_void_p(cls.data_ptr()), Q, N, ldn,
                                        ctypes.c_void_p(p_idx.data_ptr()),
                                        ctypes.c_void_p(c_idx.data_ptr()), stream_ptr(dev))
    _lib.check(rc, "veon_point_text_argmax")
    return p_idx, c_idx
