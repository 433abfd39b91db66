"""ctypes binding of libcutie_b200.so -- the hand-written sm_100a kernels behind the C-ABI in
include/cutie_b200.h.  Every function here takes CUDA torch tensors (PyTorch owns all memory, kernels
borrow pointers), enqueues on torch.cuda.current_stream() and never synchronises.

There is NO fallback: if the shared library is missing, or a tensor is not a CUDA fp32/int tensor,
these functions raise.  (tests/ swap this module's functions for oracle-backed CPU emulations to
exercise the host logic without a GPU; the product never does.)
"""
import ctypes
import os
from typing import List, NamedTuple, Optional, Sequence, Tuple

import torch

_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'lib', 'libcutie_b200.so')
_lib = None

USAGE_FIXED_POINT_BITS = 40     # usage accumulators are uint64 fixed point, 2^-40 resolution

LAUNCH_COUNT = 0                # number of cutie_b200 CUDA kernels enqueued so far (bench.py reports the delta)
PROFILE = None                  # set to a list to collect (name, start_event, end_event) per C-ABI call


class _call:
    """Counts the kernels a C-ABI call launches and, when PROFILE is a list, brackets it with CUDA events
    on the launching stream (bench.py's live per-kernel timing)."""

    def __init__(self, name: str, launches: int):
        self.name, self.launches = name, launches

    def __enter__(self):
        global LAUNCH_COUNT
        LAUNCH_COUNT += self.launches
        if PROFILE is not None:
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e0.record()
        return self

    def __exit__(self, *exc):
        if PROFILE is not None and exc[0] is None:
            e1 = torch.cuda.Event(enable_timing=True)
            e1.record()
            PROFILE.append((self.name, self.e0, e1))
        return False


class KernelError(RuntimeError):
    pass


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            raise KernelError(f'{_LIB_PATH} not found: build it with `python __graft_entry__.py build` '
                              '(there is no CPU or PyTorch fallback for the Cutie hot path)')
        _lib = ctypes.CDLL(_LIB_PATH)
        _lib.cutie_b200_last_error.restype = ctypes.c_char_p
        _lib.cutie_affinity_workspace_bytes.restype = ctypes.c_size_t
        _lib.cutie_affinity_workspace_bytes.argtypes = [ctypes.c_int64] * 3 + [ctypes.c_int]
    return _lib


def _check(status: int, what: str):
    if status != 0:
        msg = lib().cutie_b200_last_error()
        raise KernelError(f'{what} failed (status {status}): {msg.decode() if msg else "?"}')


def _stream() -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t: Optional[torch.Tensor], dtype=torch.float32) -> ctypes.c_void_p:
    if t is None:
        return ctypes.c_void_p(0)
    if not t.is_cuda:
        raise KernelError('cutie_b200 kernels need CUDA tensors (no CPU path exists)')
    if t.device.index != torch.cuda.current_device():
        # launches go to torch.cuda.current_stream() of the CURRENT device: a tensor living elsewhere would be
        # dereferenced by a kernel running on the wrong GPU
        raise KernelError(f'tensor on cuda:{t.device.index} but the current device is cuda:{torch.cuda.current_device()} '
                          '(wrap the call in torch.cuda.device(tensor.device))')
    if t.dtype != dtype:
        raise KernelError(f'expected {dtype}, got {t.dtype}')
    return ctypes.c_void_p(t.data_ptr())


def _i64(v) -> ctypes.c_int64:
    return ctypes.c_int64(int(v))


class BankSegment(NamedTuple):
    """One physically contiguous run of memory tokens (token-major).

    key [B, n, CK], shrinkage [B, n], values: per-object list of [B, n, CV]; the token axis and the
    channel axis are contiguous, the batch stride is arbitrary (views into the arena).
    """
    key: torch.Tensor
    shrinkage: torch.Tensor
    values: Tuple[torch.Tensor, ...] = ()
    # optional: the tcgen05 operand image of the ARENA this run lives in ([B, tiles, KEY_IMAGE_FLOATS], built by
    # bank_key_image) and the run's first physical token index inside that arena
    key_image: Optional[torch.Tensor] = None
    phys_begin: int = 0
    # the key centre [B, 64] the image was built with (bank_key_image(..., mu)); all segments of a call share it
    key_mu: Optional[torch.Tensor] = None

    @property
    def n(self) -> int:
        return self.key.shape[1]


KEY_IMAGE_TILE = 128            # tokens per image tile (the filter's MMA N)
KEY_IMAGE_FLOATS = 9216         # 36864 bytes of FP16 operands: 2 swizzled [128 x 128 B] K-blocks + one [128 x 32 B] tail block


def _rows_view_ok(t: torch.Tensor):
    if t.dim() == 3:
        assert t.stride(2) == 1 and t.stride(1) == t.shape[2], 'token-major rows must be dense'
    else:
        assert t.stride(1) == 1


# ---------------------------------------------------------------------------------------------
# memory readout (SURVEY.md section 8 rows a4, a5, a6)
# ---------------------------------------------------------------------------------------------
def kpad_for(top_k: int) -> int:
    if top_k <= 32:
        return 32
    if top_k <= 64:
        return 64
    raise KernelError('top_k > 64 is not supported by the sm_100a top-k kernels')


def affinity_topk(segments: Sequence[BankSegment], qk: torch.Tensor, qe: torch.Tensor, top_k: int,
                  usage_acc: Optional[torch.Tensor] = None, want_sim: bool = False,
                  seed_idx: Optional[torch.Tensor] = None):
    """Anisotropic-L2 similarity of every query against every memory token of `segments`, exact
    top-k per query, softmax over the k winners.

    qk, qe: [B, CK, Q] (channel-major, as the key projection emits them).
    Returns (idx int32 [B,Q,kpad], w f32 [B,Q,kpad], sim f32 [B,Q,kpad] or None); entries >= top_k are
    (-1, 0).  idx counts tokens across `segments` in order.  Winners are ordered by descending
    similarity, ties toward the lower index.  If usage_acc (int64 [B, N_total], zeroed by the caller) is
    given, w * 2^40 is accumulated per token (deterministic integer adds).
    seed_idx (int32 [B, Q, kpad], image plan only): per query top_k distinct token indices of THIS bank (-1 = none) --
    typically the previous frame's winners; their exact energies tighten the candidate filter's threshold.  The
    result never depends on them (any k distinct tokens bound the k-th smallest energy from above).
    """
    B, CK, Q = qk.shape
    n_total = sum(s.n for s in segments)
    if n_total < top_k:
        raise KernelError(f'selected index k out of range: top_k={top_k} > {n_total} memory tokens')
    kpad = kpad_for(top_k)
    dev = qk.device
    idx = torch.empty(B, Q, kpad, dtype=torch.int32, device=dev)
    w = torch.empty(B, Q, kpad, dtype=torch.float32, device=dev)
    sim = torch.empty(B, Q, kpad, dtype=torch.float32, device=dev) if want_sim else None
    L = lib()
    ws_bytes = L.cutie_affinity_workspace_bytes(B, Q, n_total, top_k)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    ns = len(segments)
    assert 1 <= ns <= 4
    for s in segments:
        _rows_view_ok(s.key), _rows_view_ok(s.shrinkage)
        assert s.key.shape[2] == CK
    assert qk.is_contiguous() and qe.is_contiguous()
    PA, IA = ctypes.c_void_p * ns, ctypes.c_int64 * ns
    plan = L.cutie_affinity_plan(_i64(n_total), ctypes.c_int(top_k))
    with_img = all(s.key_image is not None for s in segments)
    if with_img:
        for s in segments:
            assert s.key_image.dtype == torch.float32 and s.key_image.shape[2] == KEY_IMAGE_FLOATS
            assert s.key_image.stride(2) == 1 and s.key_image.stride(1) == KEY_IMAGE_FLOATS
            assert (s.phys_begin + s.n + KEY_IMAGE_TILE - 1) // KEY_IMAGE_TILE <= s.key_image.shape[1]
        mu = segments[0].key_mu
        for s in segments:
            assert (s.key_mu is None) == (mu is None) and (mu is None or s.key_mu.data_ptr() == mu.data_ptr()), \
                'all key images of one read must have been built with the same key centre'
        if mu is not None:
            assert mu.shape == (B, CK) and mu.is_contiguous()
        if seed_idx is not None:
            assert seed_idx.shape == (B, Q, kpad) and seed_idx.is_contiguous()
        img_args = (PA(*[s.key_image.data_ptr() for s in segments]), IA(*[s.key_image.stride(0) for s in segments]),
                    IA(*[s.phys_begin for s in segments]), _ptr(mu), _ptr(seed_idx, torch.int32))
    else:
        img_args = (None, None, None, None, None)
    # launches: exact scan (small banks, or no key images) = scan + merge; FP16 image plan = sample pass, threshold,
    # filter pass, re-rank
    with _call('affinity_topk', 4 if (plan and with_img) else 2):
        st = L.cutie_affinity_topk_img(
            ctypes.c_int(ns), PA(*[s.key.data_ptr() for s in segments]),
            PA(*[s.shrinkage.data_ptr() for s in segments]), IA(*[s.n for s in segments]),
            IA(*[s.key.stride(0) for s in segments]), IA(*[s.shrinkage.stride(0) for s in segments]),
            *img_args, _ptr(qk), _ptr(qe), _i64(B), _i64(CK), _i64(Q), ctypes.c_int(top_k), ctypes.c_int(kpad),
            _ptr(idx, torch.int32), _ptr(w), _ptr(sim), _ptr(usage_acc, torch.int64), _i64(n_total),
            _ptr(ws, torch.uint8), ctypes.c_size_t(ws_bytes), _stream())
    _check(st, 'cutie_affinity_topk')
    if KEEP_LAST_WORKSPACE:
        global _LAST_WS
        _LAST_WS = (ws, B, Q, n_total, top_k)
    return idx, w, sim


KEEP_LAST_WORKSPACE = False     # diagnostics: keep the workspace of the last affinity_topk call alive
_LAST_WS = None


def last_candidate_counts() -> Optional[torch.Tensor]:
    """Diagnostics (KEEP_LAST_WORKSPACE = True): per-query number of candidates the last filtered affinity_topk call
    handed to the exact re-rank, int32 [B, Q]; None if the last call was an exact scan."""
    if _LAST_WS is None:
        return None
    ws, B, Q, n_total, top_k = _LAST_WS
    f = lib().cutie_debug_ws_count_offset
    f.restype = ctypes.c_int64
    off = int(f(_i64(B), _i64(Q), _i64(n_total), ctypes.c_int(top_k)))
    if off < 0:
        return None
    return ws[off:off + 4 * B * Q].view(torch.int32).view(B, Q).clone()


def set_tc_min_tokens(n: int):
    """Banks with fewer tokens than n use the exact fp32 scan only; larger ones with key images take the FP16 filter
    plan (default 6144; negative restores the default)."""
    lib().cutie_set_tc_min_tokens(_i64(n))


def phase_timing(enable: bool):
    """Record per-launch device times inside the filtered affinity plan (diagnostics)."""
    lib().cutie_debug_phase_timing(ctypes.c_int(1 if enable else 0))


def phase_times(calls_ago: int = 0):
    """[ms per phase] of the filtered affinity call `calls_ago` calls back: sample pass, threshold select, filter pass,
    re-rank."""
    buf = (ctypes.c_float * 16)()
    n = lib().cutie_debug_phase_times(_i64(calls_ago), buf, ctypes.c_int(16))
    return [float(buf[i]) for i in range(n)]


def image_level_launches() -> int:
    """How many FP16 filter passes over a key image this process has run so far (one per filtered affinity call)."""
    f = lib().cutie_debug_image_level_launches
    f.restype = ctypes.c_int64
    return int(f())


def affinity_plan(n_total: int, top_k: int) -> int:
    """0 = exact fp32 scan; 1 = FP16 filter over the key images + exact re-rank of the survivors (calls with images)."""
    return int(lib().cutie_affinity_plan(_i64(n_total), ctypes.c_int(top_k)))


def topk_merge(part_val: torch.Tensor, part_idx: torch.Tensor, top_k: int, n_total: int,
               usage_acc: Optional[torch.Tensor] = None, want_sim: bool = False):
    """Merge per-shard sorted candidate lists [B, parts, Q, kpad] (dead slots: idx < 0) into the global
    top-k + softmax.  Same outputs as affinity_topk; idx are whatever index space part_idx uses."""
    B, parts, Q, kpad = part_val.shape
    assert part_val.is_contiguous() and part_idx.is_contiguous() and kpad == kpad_for(top_k)
    dev = part_val.device
    idx = torch.empty(B, Q, kpad, dtype=torch.int32, device=dev)
    w = torch.empty(B, Q, kpad, dtype=torch.float32, device=dev)
    sim = torch.empty(B, Q, kpad, dtype=torch.float32, device=dev) if want_sim else None
    with _call('topk_merge', 1):
        st = lib().cutie_topk_merge(_ptr(part_val), _ptr(part_idx, torch.int32), _i64(B), _i64(parts), _i64(Q),
                                    ctypes.c_int(top_k), ctypes.c_int(kpad), _ptr(idx, torch.int32), _ptr(w),
                                    _ptr(sim), _ptr(usage_acc, torch.int64), _i64(n_total), _stream())
    _check(st, 'cutie_topk_merge')
    return idx, w, sim


def readout_gather(idx: torch.Tensor, w: torch.Tensor, segments: Sequence[BankSegment],
                   out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out[b,k,c,q] = sum_j w[b,q,j] * V_k[idx[b,q,j], c]  ->  [B, K, CV, Q] (a6, evaluated sparsely)."""
    B, Q, kpad = idx.shape
    K = len(segments[0].values)
    CV = segments[0].values[0].shape[2]
    if out is None:
        out = torch.empty(B, K, CV, Q, dtype=torch.float32, device=idx.device)
    ns = len(segments)
    ptrs, strides = [], []
    for s in segments:
        assert len(s.values) == K
        for v in s.values:
            _rows_view_ok(v)
            ptrs.append(v.data_ptr())
            strides.append(v.stride(0))
    PA, IA, IS = ctypes.c_void_p * (ns * K), ctypes.c_int64 * (ns * K), ctypes.c_int64 * ns
    _L = lib()
    with _call('readout_gather', 1):
        st = _L.cutie_readout_gather(_ptr(idx, torch.int32), _ptr(w), _i64(B), _i64(Q), ctypes.c_int(kpad),
                                        ctypes.c_int(ns), IS(*[s.n for s in segments]), PA(*ptrs), IA(*strides),
                                        _i64(K), _i64(CV), _ptr(out), _stream())
    _check(st, 'cutie_readout_gather')
    return out


def usage_commit(use_cnt: torch.Tensor, life_cnt: torch.Tensor, usage_acc: torch.Tensor, acc_offset: int):
    """use_cnt[b,i] += usage_acc[b, acc_offset+i] * 2^-40 ; life_cnt[b,i] += 1   (kv_memory_store.py:151-162)."""
    B, n = use_cnt.shape
    if n == 0:
        return
    with _call('usage_commit', 1):
        st = lib().cutie_usage_commit(_ptr(use_cnt), _i64(use_cnt.stride(0)), _ptr(life_cnt), _i64(life_cnt.stride(0)),
                                      _ptr(usage_acc, torch.int64), _i64(usage_acc.stride(0)), _i64(acc_offset),
                                      _i64(B), _i64(n), _stream())
    _check(st, 'cutie_usage_commit')


# ---------------------------------------------------------------------------------------------
# memory bank maintenance (a17, a18)
# ---------------------------------------------------------------------------------------------
def bank_append(src: torch.Tensor, dst_rows: torch.Tensor):
    """dst_rows[b, i, c] = src[b, c, i]: channel-major feature map [B, C, n] -> token-major rows [B, n, C]."""
    B, C, n = src.shape
    assert dst_rows.shape == (B, n, C)
    _rows_view_ok(dst_rows)
    assert src.stride(2) == 1 and src.stride(1) == n
    with _call('bank_append', 1):
        st = lib().cutie_bank_append(_ptr(src), _i64(src.stride(0)), _ptr(dst_rows), _i64(dst_rows.stride(0)),
                                     _i64(B), _i64(C), _i64(n), _stream())
    _check(st, 'cutie_bank_append')


def upsample2x_add(g: torch.Tensor, skip: torch.Tensor) -> torch.Tensor:
    """bilinear x2 (align_corners=False) of every object's feature map plus the shared skip feature:
    g [B,K,C,h,w], skip [B,C,2h,2w] -> [B,K,C,2h,2w] (the mask decoder's UpsampleBlock input)."""
    B, K, C, h, w = g.shape
    assert skip.shape == (B, C, 2 * h, 2 * w)
    g, skip = g.contiguous(), skip.contiguous()
    out = torch.empty(B, K, C, 2 * h, 2 * w, dtype=torch.float32, device=g.device)
    with _call('upsample2x_add', 1):
        st = lib().cutie_upsample2x_add(_ptr(g), _ptr(skip), _ptr(out), _i64(B), _i64(K), _i64(C), _i64(h), _i64(w),
                                        _stream())
    _check(st, 'cutie_upsample2x_add')
    return out


def bias_act_(y: torch.Tensor, bias: torch.Tensor, z: Optional[torch.Tensor] = None, relu: bool = False) -> torch.Tensor:
    """In place y = act(y + bias[c] (+ z)) for a dense [N,C,H,W] tensor in NCHW or channels-last storage: the epilogue
    of a cuDNN convolution called without its bias (one float4 stream instead of ATen's broadcast add + add + clamp)."""
    assert y.dim() == 4 and y.dtype == torch.float32
    N, C, H, W = y.shape
    if y.is_contiguous():
        cl = False
    elif y.is_contiguous(memory_format=torch.channels_last):
        cl = True
    else:
        raise KernelError('bias_act_: y must be dense NCHW or channels-last')
    if z is not None:
        assert z.shape == y.shape
        if z.stride() != y.stride():            # other storage order: one copy into y's layout
            z = torch.empty_like(y).copy_(z)
    bias = bias.detach()
    assert bias.shape == (C,) and bias.is_contiguous()
    with _call('bias_act', 1):
        st = lib().cutie_bias_act(_ptr(y), _ptr(bias), _ptr(z), _i64(N), _i64(C), _i64(H * W), int(cl), int(bool(relu)),
                                  _stream())
    _check(st, 'cutie_bias_act')
    return y


def bias_relu_maxpool(y: torch.Tensor, bias: torch.Tensor) -> torch.Tensor:
    """relu(max_pool2d(y, 3, stride=2, padding=1) + bias[c]) == max_pool2d(relu(y + bias), 3, 2, 1) for a bias-less
    convolution output y [N,C,H,W] (dense NCHW, or channels-last with C % 4 == 0); the result keeps y's storage order."""
    assert y.dim() == 4 and y.dtype == torch.float32
    N, C, H, W = y.shape
    Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    if y.is_contiguous():
        cl = False
    elif y.is_contiguous(memory_format=torch.channels_last) and C % 4 == 0:
        cl = True
    else:
        y, cl = y.contiguous(), False
    out = torch.empty(N, C, Ho, Wo, dtype=torch.float32, device=y.device,
                      memory_format=torch.channels_last if cl else torch.contiguous_format)
    bias = bias.detach()
    assert bias.shape == (C,) and bias.is_contiguous()
    with _call('bias_relu_maxpool', 1):
        st = lib().cutie_bias_relu_maxpool(_ptr(y), _ptr(bias), _ptr(out), _i64(N), _i64(C), _i64(H), _i64(W), int(cl),
                                           _stream())
    _check(st, 'cutie_bias_relu_maxpool')
    return out


SEGMENT_TAIL_MAX_CHANNELS = 16


def segment_tail(x: torch.Tensor):
    """Decoder logits x [B,K,h,w] (stride 4) -> (logits [B,1+K,4h,4w], prob [B,1+K,4h,4w]): sigmoid, soft aggregation
    (background = prod(1-p), clamp, log-odds), bilinear x4, softmax over channels."""
    B, K, h, w = x.shape
    assert x.dtype == torch.float32 and K + 1 <= SEGMENT_TAIL_MAX_CHANNELS
    x = x.contiguous()
    agg = torch.empty(B, K + 1, h, w, dtype=torch.float32, device=x.device)
    logits = torch.empty(B, K + 1, 4 * h, 4 * w, dtype=torch.float32, device=x.device)
    prob = torch.empty_like(logits)
    with _call('segment_tail', 2):
        st = lib().cutie_segment_tail(_ptr(x), _ptr(agg), _ptr(logits), _ptr(prob), _i64(B), _i64(K), _i64(h), _i64(w),
                                      _stream())
    _check(st, 'cutie_segment_tail')
    return logits, prob


def conv3x3_c1(x: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor, relu_input: bool = False) -> torch.Tensor:
    """F.conv2d(relu(x) if relu_input else x, weight, bias, padding=1) for weight [1,C,3,3]: x [N,C,H,W] -> [N,1,H,W]."""
    N, C, H, W = x.shape
    assert x.dtype == torch.float32 and tuple(weight.shape) == (1, C, 3, 3) and bias.numel() == 1
    x = x.contiguous()
    w = weight.detach().contiguous()
    out = torch.empty(N, 1, H, W, dtype=torch.float32, device=x.device)
    with _call('conv3x3_c1', 1):
        st = lib().cutie_conv3x3_c1(_ptr(x), _ptr(w), _ptr(bias.detach()), _ptr(out), _i64(N), _i64(C), _i64(H), _i64(W),
                                    int(bool(relu_input)), _stream())
    _check(st, 'cutie_conv3x3_c1')
    return out


def conv_tc_eligible(weight: torch.Tensor, stride=(1, 1), padding=(1, 1), dilation=(1, 1), groups: int = 1) -> bool:
    """Geometries cutie_conv_tc implements: 3x3 / zero pad 1 and 1x1 / no pad, stride 1 or 2, Cin % 32 == 0;
    output channels go in tiles of 128 (a partial tile costs a full one, so layers with fewer than 64 output channels stay
    with the library)."""
    if weight.dim() != 4 or groups != 1 or tuple(dilation) != (1, 1) or weight.shape[0] < 64 or weight.shape[1] % 32:
        return False
    k = tuple(weight.shape[2:])
    if k == (3, 3):
        return tuple(stride) in ((1, 1), (2, 2)) and tuple(padding) == (1, 1)
    if k == (1, 1):
        return tuple(stride) in ((1, 1), (2, 2)) and tuple(padding) == (0, 0)
    return False


def conv_weight_image(weight: torch.Tensor) -> torch.Tensor:
    """The layer's tcgen05 operand image (tf32 hi | lo planes per (128-channel tile, 32-channel chunk, tap), swizzled):
    built once per weight version, 2x the weight bytes."""
    Cout, Cin, k = weight.shape[0], weight.shape[1], weight.shape[2]
    assert weight.dtype == torch.float32 and weight.shape[2] == weight.shape[3] and k in (1, 3) and Cin % 32 == 0
    lib().cutie_conv_weight_image_bytes.restype = ctypes.c_int64
    nbytes = lib().cutie_conv_weight_image_bytes(_i64(Cout), _i64(Cin), int(k))
    img = torch.empty(nbytes // 4, dtype=torch.float32, device=weight.device)
    w = weight.detach().contiguous()
    with _call('conv_weight_image', 1):
        st = lib().cutie_conv_weight_image(_ptr(w), _i64(Cout), _i64(Cin), int(k), _ptr(img), _stream())
    _check(st, 'cutie_conv_weight_image')
    return img


def _ncp_strides(t: torch.Tensor):
    """(image, channel, pixel) element strides of a dense NCHW or channels-last [N, C, H, W] tensor, else None."""
    N, C, H, W = t.shape
    sn, sc, sh, sw = t.stride()
    if W > 1 and sh != sw * W and H > 1:
        return None
    if H == 1 and W == 1:
        return (sn, sc, 1)
    return (sn, sc, sw if W > 1 else sh)


def conv_tc(x: torch.Tensor, weight_image: torch.Tensor, bias: Optional[torch.Tensor], cout: int, ksize: int = 3,
            stride: int = 1, residual: Optional[torch.Tensor] = None, relu_in: bool = False,
            relu_out: bool = False, units_per_cta: Optional[int] = None,
            counters: Optional[torch.Tensor] = None) -> torch.Tensor:
    """act(bias + conv(pre(x)) [+ residual]) on the tensor cores with 3xTF32 splitting (fp32-class accuracy).
    x [N, Cin, H, W] dense NCHW or channels-last (the output takes the same memory format) -> [N, cout, H', W'].
    Layers with fewer output tiles than SMs are spread evenly over the SMs in (tile, input chunk) units (cutie_conv_plan):
    `units_per_cta` overrides the plan's share size (tests); `counters`: the layer's own zeroed int32 tile counters (the
    kernel leaves them zero), else a fresh zeroed buffer per call."""
    N, Cin, H, W = x.shape
    assert x.dtype == torch.float32 and ksize in (1, 3)
    cl = x.is_contiguous(memory_format=torch.channels_last) and not x.is_contiguous()
    if not cl:
        x = x.contiguous()
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    out = torch.empty(N, cout, Ho, Wo, dtype=torch.float32, device=x.device,
                      memory_format=torch.channels_last if cl else torch.contiguous_format)
    zs = None
    if residual is not None:
        assert tuple(residual.shape) == (N, cout, Ho, Wo)
        zs = _ncp_strides(residual)
        if zs is None:
            residual = residual.contiguous()
            zs = _ncp_strides(residual)
    arr = lambda t: (ctypes.c_int64 * 3)(*t)
    plan = (ctypes.c_int64 * 6)()
    q = int(units_per_cta) if units_per_cta else 0
    _check(lib().cutie_conv_plan(_i64(N), _i64(Cin), _i64(cout), _i64(H), _i64(W), int(ksize), int(stride), q, plan),
           'cutie_conv_plan')
    ntile, ws_floats = int(plan[0]), int(plan[5])
    ws = cnt = None
    if ws_floats:
        ws = torch.empty(ws_floats, dtype=torch.float32, device=x.device)
        cnt = counters if counters is not None and counters.numel() >= ntile else torch.zeros(ntile, dtype=torch.int32, device=x.device)
    with _call('conv_tc', 1):
        st = lib().cutie_conv_tc(_ptr(x), arr(_ncp_strides(x)), _ptr(weight_image),
                                 _ptr(bias.detach() if bias is not None else None), _ptr(residual),
                                 arr(zs) if zs is not None else None, _i64(N), _i64(Cin), _i64(cout), _i64(H), _i64(W),
                                 int(ksize), int(stride), int(bool(relu_in)), int(bool(relu_out)), _ptr(out),
                                 arr(_ncp_strides(out)), q, _ptr(ws), _ptr(cnt, torch.int32), _stream())
    _check(st, 'cutie_conv_tc')
    return out


def area_pool(x: torch.Tensor, f: int) -> torch.Tensor:
    """F.interpolate(x, scale_factor=1/f, mode='area') for [..., H, W] with H % f == W % f == 0."""
    H, W = x.shape[-2:]
    assert x.dtype == torch.float32 and H % f == 0 and W % f == 0
    x = x.contiguous()
    out = torch.empty(*x.shape[:-2], H // f, W // f, dtype=torch.float32, device=x.device)
    planes = x.numel() // (H * W)
    with _call('area_pool', 1):
        st = lib().cutie_area_pool(_ptr(x), _ptr(out), _i64(planes), _i64(H), _i64(W), _i64(f), _stream())
    _check(st, 'cutie_area_pool')
    return out


def eca_scale_add_(y: torch.Tensor, x: torch.Tensor, conv1d_weight: torch.Tensor) -> torch.Tensor:
    """In place y = y * sigmoid(conv1d(mean_hw(y))) + x -- the tail of ChannelAttnResBlock (the spatial mean stays an
    ATen reduction).  y [N,C,H,W] dense NCHW or channels-last; x same shape; conv1d_weight [1,1,k]."""
    assert y.dim() == 4 and y.dtype == torch.float32 and x.shape == y.shape
    N, C, H, W = y.shape
    if y.is_contiguous():
        cl = False
    elif y.is_contiguous(memory_format=torch.channels_last):
        cl = True
    else:
        raise KernelError('eca_scale_add_: y must be dense NCHW or channels-last')
    if x.stride() != y.stride():
        x = torch.empty_like(y).copy_(x)
    w = conv1d_weight.detach().reshape(-1)
    mean = y.mean(dim=(2, 3)).contiguous()
    gate = torch.empty_like(mean)
    with _call('eca_scale_add', 2):
        st = lib().cutie_eca_scale_add(_ptr(y), _ptr(x), _ptr(mean), _ptr(w), _ptr(gate), _i64(N), _i64(C), _i64(H * W),
                                       _i64(w.numel()), int(cl), _stream())
    _check(st, 'cutie_eca_scale_add')
    return y


def gated_update(h: torch.Tensor, v: torch.Tensor) -> torch.Tensor:
    """GRU-like sensory update: h [B,K,d,H,W], v [B,K,3d,H,W] = [forget | update | candidate] -> [B,K,d,H,W]."""
    B, K, d, H, W = h.shape
    assert v.shape == (B, K, 3 * d, H, W) and h.dtype == torch.float32 and v.dtype == torch.float32
    h, v = h.contiguous(), v.contiguous()
    out = torch.empty_like(h)
    with _call('gated_update', 1):
        st = lib().cutie_gated_update(_ptr(v), _ptr(h), _ptr(out), _i64(B * K), _i64(d), _i64(H * W), _stream())
    _check(st, 'cutie_gated_update')
    return out


def prob_to_mask(prob: torch.Tensor, lut: torch.Tensor) -> torch.Tensor:
    """lut[argmax over channels] of a [C,H,W] probability map (any plane/row strides, unit pixel stride) -> int64 [H,W]."""
    C, H, W = prob.shape
    assert prob.stride(2) == 1 and lut.dtype == torch.int64 and lut.numel() >= C and lut.is_contiguous()
    out = torch.empty(H, W, dtype=torch.int64, device=prob.device)
    with _call('prob_to_mask', 1):
        st = lib().cutie_prob_to_mask(_ptr(prob), _i64(prob.stride(0)), _i64(prob.stride(1)), _i64(C), _i64(H), _i64(W),
                                      _ptr(lut, torch.int64), _ptr(out, torch.int64), _stream())
    _check(st, 'cutie_prob_to_mask')
    return out


def key_image_tiles(capacity: int) -> int:
    """Image tiles needed for an arena of `capacity` tokens."""
    return (int(capacity) + KEY_IMAGE_TILE - 1) // KEY_IMAGE_TILE


def bank_key_image(key_arena: torch.Tensor, shr_arena: torch.Tensor, phys_begin: int, n: int, image: torch.Tensor,
                   mu: Optional[torch.Tensor] = None):
    """(Re)build the tcgen05 operand image for tokens [phys_begin, phys_begin + n) of an arena.

    key_arena [B, cap, 64] and shr_arena [B, cap] token-major, image [B, tiles, KEY_IMAGE_FLOATS]: every
    128-token physical tile holds [shr k'^2 | shr k' | error-bound tail], k' = k - mu (mu [B, 64]: the bank's key centre,
    None = 0; the filter subtracts the same mu from the query keys), in the swizzled shared-memory layout of
    the FP16 affinity filter (csrc/tc_operand_f16.cuh), so the filter fetches a tile with one 36 KB bulk copy.
    (The tensor's dtype is float32 only as a container: 9216 floats = 36864 bytes of f16 operands per tile.)"""
    B, cap, CK = key_arena.shape
    assert CK == 64 and shr_arena.shape == (B, cap) and image.shape[0] == B and image.shape[2] == KEY_IMAGE_FLOATS
    _rows_view_ok(key_arena), _rows_view_ok(shr_arena)
    assert image.stride(2) == 1 and image.stride(1) == KEY_IMAGE_FLOATS
    assert 0 <= phys_begin and phys_begin + n <= cap
    assert mu is None or (mu.shape == (B, CK) and mu.is_contiguous())
    with _call('bank_key_image', 1):
        st = lib().cutie_bank_key_image(_ptr(key_arena), _i64(key_arena.stride(0)), _ptr(shr_arena),
                                        _i64(shr_arena.stride(0)), _i64(B), _i64(phys_begin), _i64(n), _ptr(image),
                                        _i64(image.stride(0)), _i64(image.shape[1]), _ptr(mu), _stream())
    _check(st, 'cutie_bank_key_image')


def bank_export(rows: torch.Tensor, dst: torch.Tensor):
    """dst[b, c, i] = rows[b, i, c] (token-major -> channel-major; used for the reference-shaped views)."""
    B, n, C = rows.shape
    assert dst.shape == (B, C, n) and dst.is_contiguous()
    _rows_view_ok(rows)
    with _call('bank_export', 1):
        st = lib().cutie_bank_export(_ptr(rows), _i64(rows.stride(0)), _ptr(dst), _i64(dst.stride(0)),
                                     _i64(B), _i64(C), _i64(n), _stream())
    _check(st, 'cutie_bank_export')


def bank_gather(segments_rows: Sequence[torch.Tensor], index: torch.Tensor, dst_rows: torch.Tensor):
    """dst_rows[b, j, :] = concat(segments_rows)[b, index[b, j], :]   (token-major gather; a18 eviction /
    prototype selection).  index int64 [B, m]."""
    B, m = index.shape
    C = dst_rows.shape[2]
    assert dst_rows.shape[:2] == (B, m)
    ns = len(segments_rows)
    assert 1 <= ns <= 4
    for r in segments_rows:
        _rows_view_ok(r)
    _rows_view_ok(dst_rows)
    PA, IA = ctypes.c_void_p * ns, ctypes.c_int64 * ns
    with _call('bank_gather', 1):
        st = lib().cutie_bank_gather(ctypes.c_int(ns), PA(*[r.data_ptr() for r in segments_rows]),
                                     IA(*[r.shape[1] for r in segments_rows]), IA(*[r.stride(0) for r in segments_rows]),
                                     _ptr(index, torch.int64), _ptr(dst_rows), _i64(dst_rows.stride(0)),
                                     _i64(B), _i64(m), _i64(C), _stream())
    _check(st, 'cutie_bank_gather')


def consolidate(segments: Sequence[BankSegment], proto_key: torch.Tensor, proto_sel: torch.Tensor,
                out_values: Sequence[torch.Tensor], out_shrinkage: torch.Tensor,
                stats: Optional[Tuple[torch.Tensor, torch.Tensor]] = None):
    """Potentiation (memory_manager.py:345-356): dense max-subtracted softmax over all candidate tokens
    of `segments` for each prototype, then weighted sums of candidate values and shrinkage.

    proto_key, proto_sel: [B, P, CK] token-major.  out_values[k]: [B, P, CV] rows; out_shrinkage [B, P].
    stats = (out_max, out_sumexp), both [B, P] dense (key-sharded memory): the softmax statistics of THIS shard of the
    candidates, by which its results are normalised -- what the shards exchange to combine them (inference/sharded.py).
    """
    B, P, CK = proto_key.shape
    ns = len(segments)
    K = len(out_values)
    n_total = sum(s.n for s in segments)
    ws = torch.empty(B * P * n_total, dtype=torch.float32, device=proto_key.device)
    PA, IA = ctypes.c_void_p * ns, ctypes.c_int64 * ns
    VA, VI = ctypes.c_void_p * (ns * K), ctypes.c_int64 * (ns * K)
    OA, OI = ctypes.c_void_p * K, ctypes.c_int64 * K
    vp, vs = [], []
    for s in segments:
        for v in s.values:
            vp.append(v.data_ptr()), vs.append(v.stride(0))
    for t in (proto_key, proto_sel):
        _rows_view_ok(t)
    if stats is not None:
        for t in stats:
            assert t.shape == (B, P) and t.is_contiguous() and t.dtype == torch.float32
    with _call('consolidate', 1):
        st = lib().cutie_consolidate_partial(
            ctypes.c_int(ns), PA(*[s.key.data_ptr() for s in segments]), PA(*[s.shrinkage.data_ptr() for s in segments]),
            IA(*[s.n for s in segments]), IA(*[s.key.stride(0) for s in segments]),
            IA(*[s.shrinkage.stride(0) for s in segments]), VA(*vp), VI(*vs), _i64(K),
            _ptr(proto_key), _i64(proto_key.stride(0)), _ptr(proto_sel), _i64(proto_sel.stride(0)),
            _i64(B), _i64(P), _i64(CK), _i64(out_values[0].shape[2] if K else 0),
            OA(*[v.data_ptr() for v in out_values]), OI(*[v.stride(0) for v in out_values]),
            _ptr(out_shrinkage), _i64(out_shrinkage.stride(0)), _ptr(stats[0] if stats else None),
            _ptr(stats[1] if stats else None), _ptr(ws), _i64(n_total), _stream())
    _check(st, 'cutie_consolidate_partial')


def obj_summary_accumulate(acc: torch.Tensor, new: torch.Tensor):
    """acc += new  (streaming object-memory sum, memory_manager.py:252-271).  Both [B, Q, E+1] dense."""
    assert acc.is_contiguous() and new.is_contiguous() and acc.shape == new.shape
    with _call('obj_summary_accumulate', 1):
        st = lib().cutie_obj_summary_accumulate(_ptr(acc), _ptr(new), _i64(acc.numel()), _stream())
    _check(st, 'cutie_obj_summary_accumulate')


# ---------------------------------------------------------------------------------------------
# object transformer (a9-a15)
# ---------------------------------------------------------------------------------------------
def qt_linear(x: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor], *,
              ln: Optional[Tuple[torch.Tensor, torch.Tensor]] = None, pe: Optional[torch.Tensor] = None,
              summary_norm: bool = False, relu: bool = False, residual: Optional[torch.Tensor] = None,
              residual_mod: int = 0, xhat_out: Optional[torch.Tensor] = None,
              out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Skinny fused linear for the [B*K*16, 256] query tile:
         xin = x                                   (or sums/(area+1e-4) if summary_norm: x is [M, Kd+1])
         xin = LayerNorm(xin; ln) if ln else xin   (xhat_out <- this, if given)
         xin = xin + pe if pe is not None
         y   = xin @ weight^T + bias ; relu ; + residual[m % residual_mod if residual_mod else m]
    x [M, Kd(+1)], weight [N, Kd] (row-major, may be a row-slice view), returns y [M, N].
    """
    M = x.shape[0]
    N, Kd = weight.shape
    assert weight.stride(1) == 1
    assert x.is_contiguous() and x.shape[1] == Kd + (1 if summary_norm else 0)
    if out is None:
        out = torch.empty(M, N, dtype=torch.float32, device=x.device)
    if ln is not None:
        assert Kd == 256, 'fused LayerNorm supports embed_dim 256'
    with _call('qt_linear', 1):
        st = lib().cutie_qt_linear(
            _ptr(x), _i64(M), _i64(Kd), _ptr(weight), _i64(weight.stride(0)), _i64(N), _ptr(bias),
            _ptr(ln[0] if ln else None), _ptr(ln[1] if ln else None), _ptr(pe), ctypes.c_int(int(summary_norm)),
            ctypes.c_int(int(relu)), _ptr(residual), _i64(residual_mod), _ptr(xhat_out), _ptr(out), _stream())
    _check(st, 'cutie_qt_linear')
    return out


def qt_head_fold(a: torch.Tensor, weight: torch.Tensor, *, transpose_w: bool, scale: float,
                 bias_vec: Optional[torch.Tensor] = None, num_heads: int = 8):
    """Per-head fold of a projected [M, E] tile into the other side's input space:
         out[m, h, c] = scale * sum_{d<E/H} a[m, h*d_h + d] * Wx[h*d_h + d, c],  Wx = W or W^T
         dots[m, h]   = scale * sum_d a[m, h*d_h + d] * bias_vec[h*d_h + d]   (if bias_vec)
    Returns (out [M, H, E], dots [M, H] or None).
    """
    M, E = a.shape
    assert weight.shape == (E, E) and weight.stride(1) == 1
    out = torch.empty(M, num_heads, E, dtype=torch.float32, device=a.device)
    dots = torch.empty(M, num_heads, dtype=torch.float32, device=a.device) if bias_vec is not None else None
    with _call('qt_head_fold', 1):
        st = lib().cutie_qt_head_fold(_ptr(a), _i64(M), _i64(E), ctypes.c_int(num_heads), _ptr(weight),
                                      _i64(weight.stride(0)), ctypes.c_int(int(transpose_w)), ctypes.c_float(scale),
                                      _ptr(bias_vec), _ptr(out), _ptr(dots), _stream())
    _check(st, 'cutie_qt_head_fold')
    return out, dots


def qt_self_attention(qk: torch.Tensor, v: torch.Tensor, num_queries: int, num_heads: int = 8) -> torch.Tensor:
    """softmax(Q_h K_h^T / sqrt(d)) V_h for every (object, head); qk [M, 2E] = [Q | K], v [M, E] -> [M, E]."""
    M, E2 = qk.shape
    E = E2 // 2
    out = torch.empty(M, E, dtype=torch.float32, device=qk.device)
    with _call('qt_self_attention', 1):
        st = lib().cutie_qt_self_attention(_ptr(qk), _ptr(v), _i64(M), _i64(E), ctypes.c_int(num_queries),
                                           ctypes.c_int(num_heads), _ptr(out), _stream())
    _check(st, 'cutie_qt_self_attention')
    return out


def qt_aux_mask(pixel: torch.Tensor, w: torch.Tensor, b: torch.Tensor, B: int, K: int):
    """mask_pred + sigmoid + aggregate + foreground test (a15) in one pass over pixel [B*K, E, HW].
    Returns (aux_logits f32 [B,K,HW], fg uint8 [B,K,HW], fg_count int32 [B*K])."""
    BK, E, HW = pixel.shape
    assert pixel.is_contiguous(), 'pixel must be channel-major contiguous [B*K, E, HW]'
    dev = pixel.device
    logits = torch.empty(B, K, HW, dtype=torch.float32, device=dev)
    fg = torch.empty(B, K, HW, dtype=torch.uint8, device=dev)
    cnt = torch.zeros(BK, dtype=torch.int32, device=dev)
    with _call('qt_aux_mask', 1):
        st = lib().cutie_qt_aux_mask(_ptr(pixel), _ptr(w), _ptr(b), _i64(B), _i64(K), _i64(E), _i64(HW),
                                     _ptr(logits), _ptr(fg, torch.uint8), _ptr(cnt, torch.int32), _stream())
    _check(st, 'cutie_qt_aux_mask')
    return logits, fg, cnt


def qt_pixel_to_query_tiles(qfold: torch.Tensor, pixel: torch.Tensor, pixel_pe: torch.Tensor, fg: torch.Tensor,
                            fg_count: torch.Tensor, num_queries: int, num_heads: int = 8):
    """The tensor-core half of qt_pixel_to_query only: per 64-pixel tile and object the tile-local softmax statistics and
    Z = P . pixel^T go to a workspace; the merge + value projection then runs as QtChain.p2q_combine inside the next fused
    query chain.  Returns (workspace, tiles)."""
    M, H, E = qfold.shape
    BK, _, HW = pixel.shape
    assert pixel.is_contiguous() and pixel_pe.is_contiguous() and qfold.is_contiguous() and fg.is_contiguous()
    L = lib()
    L.cutie_qt_pixel_to_query_splits.restype = ctypes.c_int
    L.cutie_qt_pixel_to_query_workspace_floats.restype = ctypes.c_int64
    splits = L.cutie_qt_pixel_to_query_splits(_i64(BK), _i64(HW), ctypes.c_int(num_heads))
    ws = torch.empty(int(L.cutie_qt_pixel_to_query_workspace_floats(_i64(BK), _i64(HW))), dtype=torch.float32,
                     device=pixel.device)
    with _call('qt_pixel_to_query', 1):
        st = L.cutie_qt_pixel_to_query(_ptr(qfold), _ptr(pixel), _ptr(pixel_pe), _ptr(fg, torch.uint8),
                                       _ptr(fg_count, torch.int32), _ptr(None), _i64(0), _ptr(None),
                                       _i64(BK), _i64(E), _i64(HW), ctypes.c_int(num_queries), ctypes.c_int(num_heads),
                                       ctypes.c_int(splits), _ptr(ws), _ptr(None), _stream())
    _check(st, 'cutie_qt_pixel_to_query')
    return ws, int(splits)


def qt_pixel_to_query(qfold: torch.Tensor, pixel: torch.Tensor, pixel_pe: torch.Tensor, fg: torch.Tensor,
                      fg_count: torch.Tensor, wv: torch.Tensor, bv: torch.Tensor, num_queries: int,
                      num_heads: int = 8) -> torch.Tensor:
    """read_from_pixel attention core (a11) for all objects/heads, on the tensor cores (csrc/qt_tc.cu):
         scores[(i,h), p] = qfold[m=(bk,i), h, :] . (pixel+pixel_pe)[bk, :, p]  (scale pre-folded)
         foreground queries (i < Q/2) see only fg pixels, background queries only non-fg (a15 rules),
         P = softmax_p(scores), Z = P . pixel^T, attn[m, h*d+e] = Z[(i,h), :] . wv[h*d+e, :] + bv[h*d+e]
    Returns attn [M, E] (to be passed through the output projection by qt_linear).  One CTA per 64-pixel tile and
    object (tile-local softmax), then a combine kernel; the tile count is fixed by HW (deterministic)."""
    M, H, E = qfold.shape
    BK, _, HW = pixel.shape
    assert pixel.is_contiguous() and pixel_pe.is_contiguous() and qfold.is_contiguous() and fg.is_contiguous()
    dev = pixel.device
    out = torch.empty(M, E, dtype=torch.float32, device=dev)
    L = lib()
    L.cutie_qt_pixel_to_query_splits.restype = ctypes.c_int
    L.cutie_qt_pixel_to_query_workspace_floats.restype = ctypes.c_int64
    splits = L.cutie_qt_pixel_to_query_splits(_i64(BK), _i64(HW), ctypes.c_int(num_heads))
    ws = torch.empty(int(L.cutie_qt_pixel_to_query_workspace_floats(_i64(BK), _i64(HW))), dtype=torch.float32, device=dev)
    with _call('qt_pixel_to_query', 2):
        st = L.cutie_qt_pixel_to_query(_ptr(qfold), _ptr(pixel), _ptr(pixel_pe), _ptr(fg, torch.uint8),
                                       _ptr(fg_count, torch.int32), _ptr(wv), _i64(wv.stride(0)), _ptr(bv),
                                       _i64(BK), _i64(E), _i64(HW), ctypes.c_int(num_queries), ctypes.c_int(num_heads),
                                       ctypes.c_int(splits), _ptr(ws), _ptr(out), _stream())
    _check(st, 'cutie_qt_pixel_to_query')
    return out


def qt_query_to_pixel(kfold: torch.Tensor, kdots: torch.Tensor, vfold: torch.Tensor, out_bias: torch.Tensor,
                      pixel: torch.Tensor, pixel_pe: torch.Tensor, num_queries: int, num_heads: int = 8,
                      out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """read_from_query (a13) fully fused on the pixel side, channel-major in and out:
         s[p, (j,h)] = (pixel+pixel_pe)[:, p] . kfold[(bk,j), h, :] + kdots[(bk,j), h]
         P = softmax over the Q queries j within each head
         out[:, p] = pixel[:, p] + out_bias + sum_{j,h} P[p,(j,h)] * vfold[(bk,j), h, :]
    """
    BK, E, HW = pixel.shape
    assert pixel.is_contiguous() and pixel_pe.is_contiguous() and kfold.is_contiguous() and vfold.is_contiguous()
    if out is None:
        out = torch.empty_like(pixel)
    with _call('qt_query_to_pixel', 1):
        st = lib().cutie_qt_query_to_pixel(_ptr(kfold), _ptr(kdots), _ptr(vfold), _ptr(out_bias), _ptr(pixel),
                                           _ptr(pixel_pe), _i64(BK), _i64(E), _i64(HW), ctypes.c_int(num_queries),
                                           ctypes.c_int(num_heads), _ptr(out), _stream())
    _check(st, 'cutie_qt_query_to_pixel')
    return out


# ---------------------------------------------------------------------------------------------
# the query-side chain of a transformer block as one launch (cutie_qt_chain)
# ---------------------------------------------------------------------------------------------
QT_CHAIN_MAX_OPS = 16
QT_CHAIN_MAX_TILES = 1024           # pixel tiles the in-chain combine can merge (64 pixels each)
_QT_LINEAR, _QT_HEAD_FOLD, _QT_SELF_ATTENTION, _QT_P2Q_COMBINE = 0, 1, 2, 3
_QT_SYNC = {}                        # device index -> 4 x uint32 grid-barrier counters (zero between launches)


class _QtOp(ctypes.Structure):       # mirrors `cutie_qt_op` (include/cutie_b200.h)
    _fields_ = [('kind', ctypes.c_int32), ('phase', ctypes.c_int32), ('inp', ctypes.c_void_p * 8),
                ('out', ctypes.c_void_p * 2), ('i', ctypes.c_int64 * 6), ('f', ctypes.c_float),
                ('reserved', ctypes.c_int32)]


class QtChain:
    """Records qt_linear / qt_head_fold / qt_self_attention / combine ops (same arguments and semantics as the stand-alone
    wrappers) and runs them as ONE persistent launch.  Ops recorded between two barrier() calls form a phase: they must
    not depend on each other; an op may consume the outputs of earlier phases.  Outputs are allocated at record time and
    hold their values after run()."""

    def __init__(self):
        self.ops = []                # (name, args, kwargs, outs, phase)
        self.phase = 0
        self.prefetch = []

    def barrier(self):
        self.phase += 1

    def linear(self, x, weight, bias, *, ln=None, pe=None, summary_norm=False, relu=False, residual=None, residual_mod=0,
               want_xhat=False):
        M = x.shape[0]
        N, Kd = weight.shape
        assert weight.stride(1) == 1 and x.is_contiguous() and x.shape[1] == Kd + (1 if summary_norm else 0)
        assert ln is None or Kd == 256, 'fused LayerNorm supports embed_dim 256'
        out = torch.empty(M, N, dtype=torch.float32, device=x.device)
        xhat = torch.empty(M, Kd, dtype=torch.float32, device=x.device) if want_xhat else None
        self.ops.append(('qt_linear', (x, weight, bias), dict(ln=ln, pe=pe, summary_norm=summary_norm, relu=relu,
                                                              residual=residual, residual_mod=residual_mod,
                                                              xhat_out=xhat), (out,), self.phase))
        self.prefetch.append(weight)
        return (out, xhat) if want_xhat else out

    def head_fold(self, a, weight, *, transpose_w, scale, bias_vec=None, num_heads=8):
        M, E = a.shape
        assert weight.shape == (E, E) and weight.stride(1) == 1 and num_heads == 8 and E == 256
        out = torch.empty(M, num_heads, E, dtype=torch.float32, device=a.device)
        dots = torch.empty(M, num_heads, dtype=torch.float32, device=a.device) if bias_vec is not None else None
        self.ops.append(('qt_head_fold', (a, weight), dict(transpose_w=transpose_w, scale=scale, bias_vec=bias_vec,
                                                           num_heads=num_heads), (out, dots), self.phase))
        self.prefetch.append(weight)
        return out, dots

    def self_attention(self, qk, v, num_queries, num_heads=8):
        M, E2 = qk.shape
        assert E2 == 512 and num_queries == 16 and num_heads == 8 and M % 16 == 0
        out = torch.empty(M, E2 // 2, dtype=torch.float32, device=qk.device)
        self.ops.append(('qt_self_attention', (qk, v, num_queries, num_heads), {}, (out,), self.phase))
        return out

    def p2q_combine(self, ws, tiles, wv, bv, BK, num_queries=16, num_heads=8):
        assert tiles <= QT_CHAIN_MAX_TILES and wv.stride(1) == 1
        out = torch.empty(BK * num_queries, 256, dtype=torch.float32, device=wv.device)
        self.ops.append(('qt_p2q_combine', (ws, tiles, wv, bv, BK, num_queries, num_heads), {}, (out,), self.phase))
        return out

    def run(self):
        if self.ops:
            qt_chain_run(self)


def _vp(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def qt_chain_run(chain: QtChain):
    """One cutie_qt_chain launch for the recorded ops."""
    n = len(chain.ops)
    if n > QT_CHAIN_MAX_OPS:
        raise KernelError(f'a query chain holds at most {QT_CHAIN_MAX_OPS} ops, got {n}')
    arr = (_QtOp * n)()
    dev = None
    for o, (name, args, kw, outs, phase) in zip(arr, chain.ops):
        o.phase = phase
        if name == 'qt_linear':
            x, w, b = args
            ln = kw['ln']
            o.kind = _QT_LINEAR
            ins = (x, w, b, ln[0] if ln else None, ln[1] if ln else None, kw['pe'], kw['residual'])
            o.i[:] = (x.shape[0], w.shape[1], w.stride(0), w.shape[0],
                      (1 if kw['summary_norm'] else 0) | (2 if kw['relu'] else 0), kw['residual_mod'])
            o.out[0], o.out[1] = _ptr(outs[0]), _ptr(kw['xhat_out'])
        elif name == 'qt_head_fold':
            a, w = args
            o.kind = _QT_HEAD_FOLD
            ins = (a, w, kw['bias_vec'])
            o.i[:] = (a.shape[0], w.stride(0), int(kw['transpose_w']), 0, 0, 0)
            o.f = float(kw['scale'])
            o.out[0], o.out[1] = _ptr(outs[0]), _ptr(outs[1])
        elif name == 'qt_self_attention':
            qk, v = args[:2]
            o.kind = _QT_SELF_ATTENTION
            ins = (qk, v)
            o.i[:] = (qk.shape[0], 0, 0, 0, 0, 0)
            o.out[0] = _ptr(outs[0])
        else:
            ws, tiles, wv, bv, BK = args[:5]
            o.kind = _QT_P2Q_COMBINE
            ins = (ws, wv, bv)
            o.i[:] = (tiles, wv.stride(0), BK, 0, 0, 0)
            o.out[0] = _ptr(outs[0])
        for j, t in enumerate(ins):
            o.inp[j] = _ptr(t)
        dev = outs[0].device
    sync = _QT_SYNC.get(dev.index)
    if sync is None:
        if torch.cuda.is_current_stream_capturing():
            raise KernelError('the first query chain of a device must run outside CUDA-graph capture (it allocates the '
                              'grid-barrier counters); warm the model up eagerly once')
        sync = _QT_SYNC[dev.index] = torch.zeros(4, dtype=torch.int32, device=dev)
    pf = [w for w in chain.prefetch if w.is_contiguous()][:16]
    PA, IA = ctypes.c_void_p * max(len(pf), 1), ctypes.c_int64 * max(len(pf), 1)
    with _call('qt_chain', 1):
        st = lib().cutie_qt_chain(arr, ctypes.c_int(n), PA(*[w.data_ptr() for w in pf]),
                                  IA(*[w.numel() * 4 for w in pf]), ctypes.c_int(len(pf)),
                                  _ptr(sync, torch.int32), _stream())
    _check(st, 'cutie_qt_chain')
