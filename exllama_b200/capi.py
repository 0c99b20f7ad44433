"""ctypes binding of libexl_b200.so -- the C ABI declared in include/exl_b200.h.

This is the thinnest possible host side: torch is used only for device memory and streams
(tensor.data_ptr(), torch.cuda.current_stream()).  There is no CPU fallback: if the library is
missing or no sm_100 device is present, calls raise.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("EXL_B200_LIB", os.path.join(_HERE, "libexl_b200.so"))   # env override: dev experiments only
_lib = None

vp, i32, i64, f32 = C.c_void_p, C.c_int, C.c_int64, C.c_float

# name -> (restype, argtypes); mirrors include/exl_b200.h one to one
SIGNATURES = {
    "exl_last_error": (C.c_char_p, []),
    "exl_version": (i32, []),
    "exl_set_tuning_params": (i32, [i32] * 9),
    "exl_prepare_buffers": (i32, [i32, vp, i64, vp, i64, vp, i32, vp, i64]),
    "exl_cleanup": (i32, []),
    "exl_make_q4": (i32, [vp, vp, vp, vp, i32, i32, i32, i32, vp, C.POINTER(vp)]),
    "exl_q4_info": (i32, [vp] + [C.POINTER(i32)] * 6),
    "exl_q4_get_x_map_host": (i32, [vp, vp]),
    "exl_q4_matmul": (i32, [vp, i32, vp, vp, i32, i32, vp]),
    "exl_q4_reconstruct": (i32, [vp, vp, vp]),
    "exl_q4_matmul_lora": (i32, [vp, i32, vp, vp, vp, vp, i32, vp, vp]),
    "exl_column_remap": (i32, [vp, vp, i32, i32, vp, vp]),
    "exl_half_matmul": (i32, [vp, vp, vp, i32, i32, i32, vp]),
    "exl_half_matmul_cublas": (i32, [vp, vp, vp, i32, i32, i32, i32, vp]),
    "exl_rms_norm": (i32, [vp, vp, vp, f32, i32, i32, i32, vp]),
    "exl_rope": (i32, [vp, vp, vp, i32, i32, i32, i32, i32, vp]),
    "exl_silu_mul": (i32, [vp, vp, i32, i32, vp]),
    "exl_update_cache": (i32, [vp, vp, vp, vp, i32, i32, i32, i32, i32, vp]),
    "exl_q4_attn": (i32, [vp, vp, f32, vp, vp, vp, vp, vp, vp, vp, vp] + [i32] * 7 + [vp, vp, i32] +
                    [vp, vp, i32] * 3 + [vp, i32, vp]),
    "exl_q4_attn_2": (i32, [vp, vp, vp, i32, vp, vp, i32, vp, vp]),
    "exl_q4_mlp": (i32, [vp, vp, f32, vp, vp, vp, i32, i32] + [vp, vp, i32] * 3 + [vp, i32, vp]),
    "exl_tp_status": (i32, [i32, C.POINTER(C.c_uint)]),
    "exl_decode_attn": (i32, [vp, vp, vp, vp, i32, i32, i32, i32, i32, vp]),
    "exl_q4_attn_2_tp": (i32, [vp, vp, vp, i32, i32, vp]),
    "exl_tp_workspace_alloc": (i32, [i32, C.POINTER(vp), vp]),
    "exl_tp_workspace_open": (i32, [i32, vp, C.POINTER(vp)]),
    "exl_tp_init": (i32, [i32, i32, i32, C.POINTER(vp)]),
    "exl_q4_attn_2_ar": (i32, [vp, vp, vp, i32, vp]),
    "exl_q4_mlp_ar": (i32, [vp, vp, f32, vp, vp, vp, i32, i32, i32, vp]),
    "exl_q4_mlp_tp": (i32, [vp, vp, f32, vp, vp, vp, i32, i32, i32, i32, vp]),
    "exl_rep_penalty": (i32, [i32, vp, vp, f32, i32, i32, i32]),
    "exl_apply_rep_penalty": (i32, [i32, vp, f32, i32, i32, i32, vp]),
    "exl_q4_matmul_host": (i32, [vp, i32, vp, vp, vp, vp, vp]),
    "exl_decode_plan_create": (i32, [vp, C.POINTER(vp)]),
    "exl_decode_plan_destroy": (i32, [vp]),
    "exl_decode_plan_info": (i32, [vp, C.POINTER(i32), C.POINTER(i32), C.POINTER(i64), C.POINTER(i64)]),
    "exl_decode_step": (i32, [vp, vp, i32, vp, vp, vp]),
    "exl_decode_plan_trace": (i32, [vp, vp, i64]),
    "exl_decode_plan_ipc_export": (i32, [vp, vp]),
    "exl_decode_plan_ipc_import": (i32, [vp, vp, i32]),
    "exl_launch_count": (i64, []),
    "exl_last_q4_path": (C.c_char_p, []),
    "exl_last_tc_config": (C.c_char_p, []),
    "exl_last_gemv_config": (C.c_char_p, []),
}


class ExlError(RuntimeError):
    pass


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ExlError(f"{LIB_PATH} is missing: run `python -m exllama_b200._build` (there is no CPU fallback)")
        _lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(_lib, name)
            fn.restype = res
            fn.argtypes = args
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        raise ExlError(f"exl_b200 error {rc}: {lib().exl_last_error().decode()}")


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class Q4:
    """Owning-side view of an exl_q4_matrix handle; keeps the borrowed tensors alive."""

    def __init__(self, qweight, qzeros, scales, g_idx=None):
        import torch
        assert qweight.is_cuda and qweight.dtype == torch.int32 and qweight.is_contiguous()
        self.qweight, self.qzeros, self.scales = qweight, qzeros, scales
        self.K, self.N, self.groups = qweight.shape[0] * 8, qweight.shape[1], qzeros.shape[0]
        self.device = qweight.device.index or 0
        h = vp()
        g = None
        if g_idx is not None:
            self._g = g_idx.to("cpu", torch.int32).contiguous()
            g = C.c_void_p(self._g.data_ptr())
        with torch.cuda.device(self.device):
            check(lib().exl_make_q4(_ptr(qweight), _ptr(qzeros), _ptr(scales), g, self.K, self.N, self.groups,
                                    self.device, _stream(), C.byref(h)))
        self.handle = h

    def x_map(self):
        import numpy as np
        out = np.empty(self.K, dtype=np.uint32)
        check(lib().exl_q4_get_x_map_host(self.handle, out.ctypes.data_as(vp)))
        return out


def q4_matmul(x, q4: Q4, out=None, no_zero=False, force_path=0):
    import torch
    M = x.shape[0]
    if out is None:
        out = torch.empty((M, q4.N), dtype=torch.float16, device=x.device)
    check(lib().exl_q4_matmul(_ptr(x), M, q4.handle, _ptr(out), int(no_zero), force_path, _stream()))
    return out


def q4_reconstruct(q4: Q4):
    import torch
    out = torch.empty((q4.K, q4.N), dtype=torch.float16, device=q4.qweight.device)
    check(lib().exl_q4_reconstruct(q4.handle, _ptr(out), _stream()))
    return out


def rms_norm(x, w, eps, out=None):
    import torch
    if out is None:
        out = torch.empty_like(x)
    check(lib().exl_rms_norm(_ptr(x), _ptr(w), _ptr(out), eps, x.shape[0], x.shape[1], x.device.index or 0, _stream()))
    return out


def rope_(x, sin, cos, past_len, num_heads, head_dim):
    bsz = x.shape[0]
    rows = x.numel() // head_dim // bsz
    check(lib().exl_rope(_ptr(x), _ptr(sin), _ptr(cos), bsz, rows, head_dim, num_heads, past_len, _stream()))


def silu_mul_(x, y):
    check(lib().exl_silu_mul(_ptr(x), _ptr(y), x.shape[0], x.shape[1], _stream()))


def update_cache(k, v, kc, vc, head_dim, kvh, q_len, max_seq, past_len):
    check(lib().exl_update_cache(_ptr(k), _ptr(v), _ptr(kc), _ptr(vc), head_dim, kvh, q_len, max_seq, past_len, _stream()))


def column_remap(x, x_map):
    import torch
    out = torch.empty_like(x)
    check(lib().exl_column_remap(_ptr(x), _ptr(out), x.shape[0], x.shape[1], _ptr(x_map), _stream()))
    return out


def half_matmul_cublas(x, w, out=None, no_zero=False):
    import torch
    if out is None:
        out = torch.empty((x.shape[0], w.shape[1]), dtype=torch.float16, device=x.device)
    check(lib().exl_half_matmul_cublas(_ptr(x), _ptr(w), _ptr(out), x.shape[0], x.shape[1], w.shape[1], int(no_zero), _stream()))
    return out


def half_matmul(x, w, out):
    check(lib().exl_half_matmul(_ptr(x), _ptr(w), _ptr(out), x.shape[0], x.shape[1], w.shape[1], _stream()))
    return out


def q4_attn(x, rms_w, eps, q, k, v, qp: Q4, kp: Q4, vp_: Q4, sin, cos, q_len, past_len, num_heads, num_kv_heads,
            head_dim, key_cache, value_cache, max_seq_len):
    bsz, dim = q.shape[0], q.shape[2]
    check(lib().exl_q4_attn(_ptr(x), _ptr(rms_w), eps, _ptr(q), _ptr(k), _ptr(v), qp.handle, kp.handle, vp_.handle,
                            _ptr(sin), _ptr(cos), bsz, q_len, dim, head_dim, num_heads, num_kv_heads, past_len,
                            _ptr(key_cache), _ptr(value_cache), max_seq_len,
                            None, None, 0, None, None, 0, None, None, 0, None, x.device.index or 0, _stream()))


def q4_attn_2(x, attn_output, op: Q4):
    check(lib().exl_q4_attn_2(_ptr(x), _ptr(attn_output), op.handle, x.shape[0], None, None, 0, None, _stream()))


def q4_mlp(x, rms_w, eps, gate: Q4, up: Q4, down: Q4):
    check(lib().exl_q4_mlp(_ptr(x), _ptr(rms_w), eps, gate.handle, up.handle, down.handle, x.shape[0], x.shape[1],
                           None, None, 0, None, None, 0, None, None, 0, None, x.device.index or 0, _stream()))


def decode_attn(q, key_cache, value_cache, num_heads, num_kv_heads, head_dim, seq_len, max_seq_len):
    import torch
    out = torch.empty_like(q)
    check(lib().exl_decode_attn(_ptr(q), _ptr(key_cache), _ptr(value_cache), _ptr(out), num_heads, num_kv_heads, head_dim, seq_len, max_seq_len, _stream()))
    return out


def prepare_buffers(device, temp_state, temp_mlp, temp_zeros_float, temp_dq):
    check(lib().exl_prepare_buffers(device, _ptr(temp_state), temp_state.numel(), _ptr(temp_mlp), temp_mlp.numel(),
                                    _ptr(temp_zeros_float), temp_zeros_float.shape[-1], _ptr(temp_dq), temp_dq.numel()))


def launch_count() -> int:
    return int(lib().exl_launch_count())


def last_q4_path() -> str:
    return lib().exl_last_q4_path().decode()


def last_tc_config() -> str:
    """Tile configuration of the last tcgen05 GEMM launch ("128x128", "256x128", "256x256", "+mc" when multicast ran)."""
    return lib().exl_last_tc_config().decode()


def last_gemv_config() -> str:
    """Decode GEMV launches of the last q4_* call, "; "-separated, each e.g. "rmsnorm+silu_mul cs=2 chunk=8 items=86"
    (prologue+epilogue, cluster size = K split, x staging chunk in 128-k stages, clusters); "none" when it made none."""
    return lib().exl_last_gemv_config().decode()


class _DecodeDesc(C.Structure):
    """struct exl_decode_desc (include/exl_b200.h)"""
    _fields_ = [("n_layers", i32), ("num_heads", i32), ("head_dim", i32), ("max_seq_len", i32), ("vocab", i32), ("rms_eps", f32),
                ("mats", C.POINTER(vp)), ("ln1", C.POINTER(vp)), ("ln2", C.POINTER(vp)), ("key_cache", C.POINTER(vp)),
                ("value_cache", C.POINTER(vp)), ("sin", vp), ("cos", vp), ("final_norm", vp), ("lm_head", vp),
                ("tp_rank", i32), ("tp_world", i32)]


class DecodePlan:
    """exl_decode_plan: the whole decode token as one persistent kernel (csrc/decode_step.cu).

    handles: per layer the 7 Q4 handles (q, k, v, o, gate, up, down) as integers / c_void_p; every tensor passed here is
    borrowed and must outlive the plan."""

    def __init__(self, handles, ln1, ln2, key_cache, value_cache, sin, cos, num_heads, head_dim, max_seq_len, eps,
                 final_norm=None, lm_head=None, tp_rank=0, tp_world=1):
        n = len(handles)
        self._keep = (ln1, ln2, key_cache, value_cache, sin, cos, final_norm, lm_head)
        flat = []
        for hs in handles:
            assert len(hs) == 7
            flat += [h.value if isinstance(h, C.c_void_p) else int(h) for h in hs]
        self._mats = (vp * (7 * n))(*flat)
        arr = lambda ts: (vp * n)(*[t.data_ptr() for t in ts])
        self._a = [arr(ln1), arr(ln2), arr(key_cache), arr(value_cache)]
        d = _DecodeDesc()
        d.n_layers, d.num_heads, d.head_dim, d.max_seq_len = n, num_heads, head_dim, max_seq_len
        d.vocab = lm_head.shape[0] if lm_head is not None else 0
        d.rms_eps = eps
        d.mats = C.cast(self._mats, C.POINTER(vp))
        d.ln1, d.ln2, d.key_cache, d.value_cache = (C.cast(x, C.POINTER(vp)) for x in self._a)
        d.sin, d.cos = sin.data_ptr(), cos.data_ptr()
        d.final_norm = final_norm.data_ptr() if final_norm is not None else None
        d.lm_head = lm_head.data_ptr() if lm_head is not None else None
        d.tp_rank, d.tp_world = tp_rank, tp_world
        self.vocab = d.vocab
        self.tp_world = tp_world
        self.handle = vp()
        check(lib().exl_decode_plan_create(C.byref(d), C.byref(self.handle)))

    def ipc_export(self) -> bytes:
        buf = (C.c_ubyte * 64)()
        check(lib().exl_decode_plan_ipc_export(self.handle, C.cast(buf, vp)))
        return bytes(buf)

    def ipc_import(self, handles):
        """handles: list of `world` 64-byte handles in rank order (as gathered from every rank's ipc_export())."""
        blob = b"".join(bytes(h) for h in handles)
        assert len(blob) == 64 * self.tp_world
        buf = (C.c_ubyte * len(blob)).from_buffer_copy(blob)
        check(lib().exl_decode_plan_ipc_import(self.handle, C.cast(buf, vp), self.tp_world))

    def info(self):
        g, r, s, b = i32(), i32(), i64(), i64()
        check(lib().exl_decode_plan_info(self.handle, C.byref(g), C.byref(r), C.byref(s), C.byref(b)))
        return {"grid": g.value, "ring_stages": r.value, "smem_bytes": s.value, "barriers_per_step": b.value}

    def step(self, x_in, past_len, x_out=None, logits=None):
        check(lib().exl_decode_step(self.handle, _ptr(x_in), past_len, _ptr(x_out), _ptr(logits), _stream()))

    def trace(self):
        """[grid, 4 layers, 24 events] globaltimer stamps (ns) of the last launch (EXL_DS_TRACE=1 at creation)."""
        import numpy as np
        g = self.info()["grid"]
        out = np.zeros((g, 4, 24), dtype=np.uint64)
        check(lib().exl_decode_plan_trace(self.handle, out.ctypes.data_as(vp), out.size))
        return out

    def close(self):
        if self.handle:
            check(lib().exl_decode_plan_destroy(self.handle))
            self.handle = None
