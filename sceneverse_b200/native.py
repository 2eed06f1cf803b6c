"""Thin torch-tensor front-ends of the libsvgps kernels (allocation, stream, status checks)."""
import torch

from . import _lib

_ACT = {None: 0, "none": 0, "relu": 1, "gelu": 2}


def gemm(a, w, bias=None, act=None, residual=None, out_dtype=torch.bfloat16, rowmax=0):
    """epilogue(a @ w.T): a (M,K) bf16, w (N,K) bf16 (nn.Linear layout), bias (N) f32 -> (M,N) (or (M/16,N) with rowmax=16).
    Rows may be strided (last dim contiguous, stride % 8 == 0)."""
    assert a.is_cuda and a.dtype == torch.bfloat16 and w.dtype == torch.bfloat16 and a.dim() == 2 and w.dim() == 2
    assert a.stride(1) == 1 and w.stride(1) == 1
    M, K = a.shape
    N = w.shape[0]
    out = torch.empty((M // rowmax if rowmax else M, N), dtype=out_dtype, device=a.device)
    if bias is not None:
        bias = bias.float().contiguous()
    if residual is not None:
        residual = residual.to(out_dtype).contiguous()
    lib = _lib.gps()
    with torch.cuda.device(a.device):
        st = lib.sv_gemm_bf16(a.data_ptr(), a.stride(0), w.data_ptr(), w.stride(0), M, N, K,
                              bias.data_ptr() if bias is not None else None, _ACT[act],
                              residual.data_ptr() if residual is not None else None, out.data_ptr(), N,
                              1 if out_dtype == torch.float32 else 0, rowmax,
                              torch.cuda.current_stream(a.device).cuda_stream)
    _lib.check(lib, st, "sv_gemm_bf16")
    return out


def _mask_bytes(mask):
    """(B, L) key-padding mask as the uint8 bytes the kernels read: a bool tensor already IS one byte of 0 / 1 per element,
    so it is re-viewed, not copied (32 cast kernels per training step otherwise)."""
    if mask is None:
        return None
    if mask.dtype == torch.bool:
        return mask.contiguous().view(torch.uint8)
    return (mask != 0).contiguous().view(torch.uint8)


def attention(q, k, v, num_heads, key_padding_mask=None, spatial_w=None, spatial_heads=0, pairwise_locs=None,
              return_lse=False, dropout_p=0.0, seed=0):
    """Fused attention forward: q (B,Lq,E), k/v (B,Lk,E) bf16 (views with a contiguous last dim are fine), head dim 64.
    key_padding_mask (B,Lk) bool, True = ignore.  spatial_w (B,Lq,spatial_heads*6) + pairwise_locs (B,Lq,Lk,5) switch on the
    MultiHeadAttentionSpatial 'cond' gate.  Returns (B,Lq,E) bf16."""
    B, Lq, E = q.shape
    Lk = k.shape[1]
    assert E == num_heads * 64 and q.dtype == k.dtype == v.dtype == torch.bfloat16
    assert q.stride(2) == 1 and k.stride(2) == 1 and v.stride(2) == 1
    out = torch.empty((B, Lq, E), dtype=torch.bfloat16, device=q.device)
    kpm = _mask_bytes(key_padding_mask)
    sw = locs = None
    if spatial_w is not None:
        sw = spatial_w.float().contiguous()
        locs = pairwise_locs.float().contiguous()
    lse = torch.empty((B, num_heads, Lq), dtype=torch.float32, device=q.device) if return_lse else None
    lib = _lib.gps()
    with torch.cuda.device(q.device):
        st = lib.sv_attention_fwd_dropout_bf16(
            q.data_ptr(), q.stride(0), q.stride(1), k.data_ptr(), k.stride(0), k.stride(1), v.data_ptr(), v.stride(0),
            v.stride(1), out.data_ptr(), out.stride(0), out.stride(1), kpm.data_ptr() if kpm is not None else None,
            sw.data_ptr() if sw is not None else None, int(spatial_heads), locs.data_ptr() if locs is not None else None,
            B, num_heads, Lq, Lk, 0.125, lse.data_ptr() if lse is not None else None, float(dropout_p), int(seed),
            torch.cuda.current_stream(q.device).cuda_stream)
    _lib.check(lib, st, "sv_attention_fwd_dropout_bf16")
    return (out, lse) if return_lse else out


def attention_backward(q, k, v, out, grad_out, lse, num_heads, key_padding_mask=None, spatial_w=None, pairwise_locs=None,
                       dropout_p=0.0, seed=0, packed_grad=None):
    """Gradients of `attention` (gate requires one weight set per head).  Returns (dq, dk, dv, d_spatial_w or None).
    packed_grad: a (B, L, 3E) bf16 buffer (self-attention on a packed QKV projection): dq / dk / dv are written straight
    into its three column slices and returned as views."""
    B, Lq, E = q.shape
    Lk = k.shape[1]
    dev = q.device
    grad_out = grad_out.to(torch.bfloat16).contiguous()
    out = out.contiguous()
    if packed_grad is not None:
        assert Lq == Lk and packed_grad.shape == (B, Lq, 3 * E) and packed_grad.is_contiguous() and packed_grad.dtype == torch.bfloat16
        dq, dk, dv = packed_grad[..., :E], packed_grad[..., E:2 * E], packed_grad[..., 2 * E:]
        d_rs = 3 * E
    else:
        dq = torch.empty((B, Lq, E), dtype=torch.bfloat16, device=dev)
        dk = torch.empty((B, Lk, E), dtype=torch.bfloat16, device=dev)
        dv = torch.empty((B, Lk, E), dtype=torch.bfloat16, device=dev)
        d_rs = E
    lib = _lib.gps()
    scratch = torch.empty(lib.sv_attention_bwd_scratch_floats(B, num_heads, Lq, Lk), dtype=torch.float32, device=dev)
    kpm = _mask_bytes(key_padding_mask)
    sw = locs = dsw = None
    if spatial_w is not None:
        sw, locs = spatial_w.float().contiguous(), pairwise_locs.float().contiguous()
        dsw = torch.empty_like(sw)
    with torch.cuda.device(dev):
        st = lib.sv_attention_bwd_strided_bf16(
            q.data_ptr(), q.stride(0), q.stride(1), k.data_ptr(), k.stride(0), k.stride(1), v.data_ptr(), v.stride(0),
            v.stride(1), out.data_ptr(), grad_out.data_ptr(), kpm.data_ptr() if kpm is not None else None,
            sw.data_ptr() if sw is not None else None, locs.data_ptr() if locs is not None else None, lse.data_ptr(),
            B, num_heads, Lq, Lk, 0.125, dq.data_ptr(), dk.data_ptr(), dv.data_ptr(), d_rs,
            dsw.data_ptr() if dsw is not None else None, scratch.data_ptr(), float(dropout_p), int(seed),
            torch.cuda.current_stream(dev).cuda_stream)
    _lib.check(lib, st, "sv_attention_bwd_strided_bf16")
    return dq, dk, dv, dsw


def colsum(x):
    """Column sums of a (R, N) bf16 / f32 matrix (rows may be strided) -> (N,) f32; deterministic native kernel."""
    assert x.is_cuda and x.dim() == 2 and x.stride(1) == 1 and x.dtype in (torch.bfloat16, torch.float32)
    R, N = x.shape
    lib = _lib.gps()
    out = torch.empty(N, dtype=torch.float32, device=x.device)
    scratch = torch.empty(lib.sv_colsum_scratch_floats(N), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        st = lib.sv_colsum(x.data_ptr(), x.stride(0), 1 if x.dtype == torch.bfloat16 else 0, R, N, out.data_ptr(),
                           scratch.data_ptr(), torch.cuda.current_stream(x.device).cuda_stream)
    _lib.check(lib, st, "sv_colsum")
    return out


def gemm_ex(a, b, a_transposed=False, b_transposed=False, bias=None, act=None, out_dtype=torch.bfloat16):
    """epilogue(A . B^T) with operands optionally given transposed in memory (no copies):
    a: (M,K), or (K,M) when a_transposed;  b: (N,K), or (K,N) when b_transposed.  bf16 in, bf16 / f32 out (M,N)."""
    assert a.is_cuda and a.dtype == torch.bfloat16 and b.dtype == torch.bfloat16 and a.dim() == 2 and b.dim() == 2
    assert a.stride(1) == 1 and b.stride(1) == 1
    M, K = (a.shape[1], a.shape[0]) if a_transposed else a.shape
    N, Kb = (b.shape[1], b.shape[0]) if b_transposed else b.shape
    assert K == Kb, (a.shape, b.shape)
    out = torch.empty((M, N), dtype=out_dtype, device=a.device)
    if bias is not None:
        bias = bias.float().contiguous()
    lib = _lib.gps()
    with torch.cuda.device(a.device):
        st = lib.sv_gemm_bf16_ex(a.data_ptr(), a.stride(0), 1 if a_transposed else 0, b.data_ptr(), b.stride(0),
                                 1 if b_transposed else 0, M, N, K, bias.data_ptr() if bias is not None else None, _ACT[act],
                                 None, out.data_ptr(), N, 1 if out_dtype == torch.float32 else 0, 0,
                                 torch.cuda.current_stream(a.device).cuda_stream)
    _lib.check(lib, st, "sv_gemm_bf16_ex")
    return out


def _stream(t):
    return torch.cuda.current_stream(t.device).cuda_stream


def _rows_ok(t):
    return t.dim() == 2 and t.stride(1) == 1 and t.stride(0) % 8 == 0 and t.data_ptr() % 16 == 0


def linear_fwd(x, w, bias=None, act=None, dropout_p=0.0, seed=0, out_dtype=torch.bfloat16, want_pre=False, n_out=None,
               out=None):
    """out = dropout(act(x @ w[:n].T + bias)): x (M,K) bf16, w (N,K) bf16, bias (N) f32.  `out` may be a wider buffer
    (M, Np >= N): only the first N columns are written.  want_pre: also return the pre-activation (bf16, same layout)."""
    assert x.dtype == torch.bfloat16 and w.dtype == torch.bfloat16 and _rows_ok(x) and _rows_ok(w), (x.shape, x.stride(), w.shape)
    M, K = x.shape
    N = w.shape[0] if n_out is None else n_out
    if out is None:
        out = torch.empty((M, N), dtype=out_dtype, device=x.device)
    pre = torch.empty_like(out) if want_pre else None
    if bias is not None:
        assert bias.dtype == torch.float32 and bias.is_contiguous()
    lib = _lib.gps()
    with torch.cuda.device(x.device):
        st = lib.sv_linear_fwd_bf16(x.data_ptr(), x.stride(0), w.data_ptr(), w.stride(0), M, N, K,
                                    bias.data_ptr() if bias is not None else None, _ACT[act], float(dropout_p), int(seed),
                                    out.data_ptr(), out.stride(0), 1 if out.dtype == torch.float32 else 0,
                                    pre.data_ptr() if pre is not None else None, _stream(x))
    _lib.check(lib, st, "sv_linear_fwd_bf16")
    return (out, pre) if want_pre else out


def linear_dgrad(g, w, act=None, aux=None, dropout_p=0.0, seed=0, n_red=None, out_dtype=torch.bfloat16):
    """dx (M,Kin) = (g (M,N) @ w (N,Kin)) * act'(aux) [* dropout mask]; n_red > w.shape[0]: g carries zero pad columns."""
    assert g.dtype == torch.bfloat16 and w.dtype == torch.bfloat16 and _rows_ok(g) and _rows_ok(w)
    M = g.shape[0]
    N = g.shape[1] if n_red is None else n_red
    Kin = w.shape[1]
    dx = torch.empty((M, Kin), dtype=out_dtype, device=g.device)
    if aux is not None:
        assert aux.dtype == torch.bfloat16 and aux.shape == (M, Kin) and aux.stride(1) == 1
    lib = _lib.gps()
    with torch.cuda.device(g.device):
        st = lib.sv_linear_dgrad_bf16(g.data_ptr(), g.stride(0), w.data_ptr(), w.stride(0), M, N, Kin, _ACT[act],
                                      aux.data_ptr() if aux is not None else None, aux.stride(0) if aux is not None else 0,
                                      float(dropout_p), int(seed), dx.data_ptr(), dx.stride(0),
                                      1 if out_dtype == torch.float32 else 0, _stream(g))
    _lib.check(lib, st, "sv_linear_dgrad_bf16")
    return dx


def linear_wgrad(g, x, n_out=None, dw=None, db=None, want_db=False, accumulate=False):
    """dw (N,Kin) f32 (+)= g[:, :N].T @ x, db (N) f32 (+)= g[:, :N].sum(0).  accumulate=True adds into the given dw / db (the
    flat gradient buffer), otherwise they are (allocated and) overwritten."""
    assert g.dtype == torch.bfloat16 and x.dtype == torch.bfloat16 and _rows_ok(g) and _rows_ok(x) and g.shape[0] == x.shape[0]
    M, Kin = x.shape
    N = g.shape[1] if n_out is None else n_out
    if dw is None:
        assert not accumulate
        dw = torch.empty((N, Kin), dtype=torch.float32, device=g.device)
    if db is None and want_db:
        assert not accumulate
        db = torch.empty(N, dtype=torch.float32, device=g.device)
    assert dw.dtype == torch.float32 and dw.stride(1) == 1 and dw.shape == (N, Kin)
    lib = _lib.gps()
    with torch.cuda.device(g.device):
        st = lib.sv_linear_wgrad_bf16(g.data_ptr(), g.stride(0), x.data_ptr(), x.stride(0), M, N, Kin, dw.data_ptr(),
                                      dw.stride(0), db.data_ptr() if db is not None else None, 1 if accumulate else 0,
                                      _stream(g))
    _lib.check(lib, st, "sv_linear_wgrad_bf16")
    return dw, db


def act_bwd(g, aux, act):
    """g * act'(aux): (M,N) bf16; relu: aux = forward output, gelu: aux = pre-activation."""
    assert g.dtype == torch.bfloat16 and aux.dtype == torch.bfloat16 and g.shape == aux.shape and _rows_ok(g) and _rows_ok(aux)
    out = torch.empty((g.shape[0], g.shape[1]), dtype=torch.bfloat16, device=g.device)
    lib = _lib.gps()
    with torch.cuda.device(g.device):
        st = lib.sv_act_bwd_bf16(g.data_ptr(), g.stride(0), aux.data_ptr(), aux.stride(0), _ACT[act], g.shape[0], g.shape[1],
                                 out.data_ptr(), out.stride(0), _stream(g))
    _lib.check(lib, st, "sv_act_bwd_bf16")
    return out


def embedding_bwd(grad_out, ids, dw, padding_idx=-1):
    """dw[ids] += grad_out: grad_out (..., D) bf16 | f32, ids (...) int64, dw (V, D) f32 contiguous (accumulated into)."""
    D = grad_out.shape[-1]
    g2 = grad_out.reshape(-1, D)
    if g2.stride(1) != 1:
        g2 = g2.contiguous()
    ids = ids.reshape(-1).contiguous()
    assert ids.dtype == torch.int64 and dw.dtype == torch.float32 and dw.is_contiguous() and dw.shape[1] == D
    assert g2.dtype in (torch.bfloat16, torch.float32) and g2.shape[0] == ids.numel()
    lib = _lib.gps()
    with torch.cuda.device(g2.device):
        st = lib.sv_embedding_bwd(g2.data_ptr(), g2.stride(0), 1 if g2.dtype == torch.bfloat16 else 0, ids.data_ptr(),
                                  ids.numel(), D, dw.shape[0], int(padding_idx if padding_idx is not None else -1),
                                  dw.data_ptr(), _stream(g2))
    _lib.check(lib, st, "sv_embedding_bwd")
    return dw


def gemm_force_ctas(n):
    """0 = heuristic, 1 = single-CTA tiles, 2 = CTA pairs (cta_group::2) wherever the problem has more than 128 rows,
    4 = CTA pairs in multicast clusters of two (experiment); bits 8.. are timing-only profiling switches (svgps.h)."""
    _lib.check(_lib.gps(), _lib.gps().sv_gemm_force_ctas(int(n)), "sv_gemm_force_ctas")
