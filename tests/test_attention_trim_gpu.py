"""Key-padding masks together with weight dropout, and key tiles that hold no unmasked key.

The attention kernels skip every key past the last unmasked one of a scene.  Those keys carry exactly zero weight, so the
forward must be bit-identical to the same scene with the padded keys cut off, and the backward must still write their
dK / dV rows (as zeros): the packed QKV gradient comes from torch.empty and every row of it is read downstream."""
import pytest
import torch

pytestmark = pytest.mark.gpu

B_KENDS = [0, 1, 16, 127, 128, 129, 257, 300]   # suffix masks: 1 + index of the last unmasked key per scene
L, H, E, P, SEED = 300, 12, 768, 0.1, 987654321
ROW_MIX = 0x9E3779B97F4A7C15                       # csrc/attn_common.cuh drop_row_key: seed + row * ROW_MIX


def rand(*shape, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn(*shape, device="cuda", generator=g)


def _mask():
    """(B, L) bool, True = ignore: the suffix masks of B_KENDS plus one scene with holes (first key masked, gaps)."""
    m = torch.zeros(len(B_KENDS) + 1, L, dtype=torch.bool, device="cuda")
    for b, kend in enumerate(B_KENDS):
        m[b, kend:] = True
    hole = m[len(B_KENDS)]
    hole[0] = True
    hole[40:90] = True
    hole[130:131] = True
    hole[200:250] = True
    hole[281:] = True                               # kend = 281
    return m


def _kend(row):
    live = (~row).nonzero()
    return int(live[-1]) + 1 if live.numel() else 0


def _inputs():
    B = len(B_KENDS) + 1
    q, k, v = (rand(B, L, E, seed=s).bfloat16() for s in (1, 2, 3))
    go = rand(B, L, E, seed=4).bfloat16()
    return q, k, v, go, _mask()


def _scene_seed(b):
    """seed under which scene b of a batch of one draws the dropout mask it draws at index b of the full batch"""
    return (SEED + b * H * L * ROW_MIX) % (1 << 64)


def test_forward_bit_equal_to_cut_keys():
    from sceneverse_b200 import native
    q, k, v, _, mask = _inputs()
    out, lse = native.attention(q, k, v, H, key_padding_mask=mask, return_lse=True, dropout_p=P, seed=SEED)
    for b in range(mask.shape[0]):
        kend = _kend(mask[b])
        if kend == 0:
            assert torch.equal(out[b], torch.zeros_like(out[b]))
            assert torch.isinf(lse[b]).all() and (lse[b] > 0).all()
            continue
        o1, l1 = native.attention(q[b:b + 1], k[b:b + 1, :kend], v[b:b + 1, :kend], H,
                                  key_padding_mask=mask[b:b + 1, :kend], return_lse=True, dropout_p=P,
                                  seed=_scene_seed(b))
        assert torch.equal(out[b:b + 1], o1), (b, kend)
        assert torch.equal(lse[b:b + 1], l1), (b, kend)


def test_backward_matches_torch_with_mask_and_dropout():
    import numpy as np
    from sceneverse_b200 import native
    from tests.test_attention_gpu import _dropout_keep
    q, k, v, go, mask = _inputs()
    B = mask.shape[0]
    out, lse = native.attention(q, k, v, H, key_padding_mask=mask, return_lse=True, dropout_p=P, seed=SEED)
    dq, dk, dv, _ = native.attention_backward(q, k, v, out, go, lse, H, key_padding_mask=mask, dropout_p=P, seed=SEED)
    for g in (dq, dk, dv):
        assert torch.isfinite(g.float()).all()
    dead = [b for b in range(B) if _kend(mask[b]) == 0]
    for b in dead:                                   # every key masked: no gradient at all
        for g in (dq, dk, dv):
            assert torch.equal(g[b], torch.zeros_like(g[b]))
    for g in (dk, dv):                               # masked keys get exactly zero gradient
        assert (g.float().masked_select(mask[..., None].expand(-1, -1, E)) == 0).all()
    live = [b for b in range(B) if b not in dead]
    keep = torch.from_numpy(np.ascontiguousarray(_dropout_keep(SEED, B, H, L, L, P))).cuda()[live]
    qf, kf, vf = (t[live].float().requires_grad_(True) for t in (q, k, v))
    n = len(live)
    qh, kh, vh = (t.view(n, L, H, 64).transpose(1, 2) for t in (qf, kf, vf))
    att = ((qh @ kh.transpose(-1, -2)) * 0.125).masked_fill(mask[live][:, None, None, :], float("-inf")).softmax(-1)
    want = ((att * keep / (1 - P)) @ vh).transpose(1, 2).reshape(n, L, E)
    want.backward(go[live].float())
    assert (out[live].float() - want).abs().max().item() / want.abs().max().item() < 2e-2
    for g, w, name in zip((dq, dk, dv), (qf.grad, kf.grad, vf.grad), "qkv"):
        err = (g[live].float() - w).abs().max().item() / (w.abs().max().item() + 1e-9)
        assert err < 3e-2, (name, err)


@pytest.mark.parametrize("p", [0.0, P])
def test_packed_gradient_rows_of_masked_keys_are_written(p):
    from sceneverse_b200 import native
    q, k, v, go, mask = _inputs()
    B = mask.shape[0]
    out, lse = native.attention(q, k, v, H, key_padding_mask=mask, return_lse=True, dropout_p=p, seed=SEED)
    packed = torch.full((B, L, 3 * E), float("nan"), dtype=torch.bfloat16, device="cuda")
    dq, dk, dv, _ = native.attention_backward(q, k, v, out, go, lse, H, key_padding_mask=mask, dropout_p=p, seed=SEED,
                                              packed_grad=packed)
    assert not torch.isnan(packed.float()).any()
    sel = mask[..., None].expand(-1, -1, E)
    for g in (dk, dv):
        assert (g.float().masked_select(sel) == 0).all()
    ref = native.attention_backward(q, k, v, out, go, lse, H, key_padding_mask=mask, dropout_p=p, seed=SEED)
    for g, r in zip((dq, dk, dv), ref[:3]):
        assert torch.equal(g, r)
