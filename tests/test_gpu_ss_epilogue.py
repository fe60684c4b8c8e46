"""The staged, coalesced epilogue of the persistent prologue GEMMs (ss_store_staged) stores exactly what the thread-per-row stores
(ss_store_row, backend bit 11 = +2048) store: the GEMM on its own at ragged shapes (C, its fp16x3 image, image only), and the whole B=100
prologue (every plain-mode product, single CTAs and CTA pairs) followed by the greedy decode."""
import numpy as np
import pytest
import torch

from gvd_b200 import capi, synth

pytestmark = pytest.mark.gpu

ROW_STORE = 2048


@pytest.fixture(autouse=True)
def _restore_backend():
    prev = capi.get_backend()
    yield
    capi.set_backend(prev)


def _decode_f16x3(img, N, scale):
    M, Np = img.shape
    h = img.cpu().numpy().view(np.float16).astype(np.float64).reshape(M, Np // 32, 2, 16, 2)
    v = (h[:, :, 0] + h[:, :, 1]).reshape(M, Np) / scale
    return v[:, :N], v[:, N:]


# 256-column tiles with a partial last tile and image padding that is not a multiple of 32 (601: tiles 256 + 256 + 89, pitch 608; odd
# ldc = scalar tail), M not a multiple of 256 (the pair's row tiles), 128- and 64-column tiles
@pytest.mark.parametrize("M,N,K", [(20000, 601, 300), (3000, 2600, 96), (20000, 520, 64), (10000, 300, 64), (5000, 200, 36)])
@pytest.mark.parametrize("act", [0, 1])
@pytest.mark.parametrize("ss_backend", [923, 1947])
def test_linear_f16ss_staged_epilogue(M, N, K, act, ss_backend):
    g = torch.Generator().manual_seed(M + 5 * N)
    A = torch.randn(M, K, generator=g).cuda()
    W = (torch.randn(N, K, generator=g) / K ** 0.5).cuda()
    b = torch.randn(N, generator=g).cuda()
    out = {}
    for flags in (ss_backend, ss_backend | ROW_STORE):
        capi.set_backend(flags)
        C, img = capi.op_linear_f16ss(A, W, b, act, want_img=True)
        _, img_only = capi.op_linear_f16ss(A, W, b, act, want_img=True, want_c=False)
        out[flags] = (C, img, img_only)
    torch.cuda.synchronize()
    C, img, img_only = out[ss_backend]
    for x, y in zip(out[ss_backend], out[ss_backend | ROW_STORE]):
        assert torch.equal(x, y)
    assert torch.equal(img_only, img)
    ref = A.double() @ W.double().t() + b.double()
    if act:
        ref = ref.clamp(min=0)
    scale = max(1.0, float(ref.abs().max()))
    assert float((C.double() - ref).abs().max()) <= 2e-5 * scale
    val, pad = _decode_f16x3(img, N, 4.0)
    assert float(np.abs(val - C.cpu().double().numpy()).max()) <= 2.0 ** -20 * scale and not pad.any()


@pytest.mark.parametrize("ss_backend", [923, 1947])
def test_prologue_staged_epilogue_bit_identical(ss_backend):
    B, T = 100, 10
    opt = synth.make_opt(t_attn_size=T)
    nm = capi.NativeModel(opt)
    nm.load_state_dict(synth.make_state_dict(opt))
    inp = synth.make_inputs(opt, B, seed=1234, masked=False)
    keys = ("segs_feat", "ppls", "num", "ppls_feat", "sample_idx", "pnt_mask")
    dev = {k: inp[k].cuda() for k in keys}
    BR, H, A = B * nm.R, opt.rnn_size, opt.att_hid_size
    NCp = (opt.detect_size + 1 + 3) // 4 * 4
    shapes = {"g_pool": (BR, 2048), "pool_embed": (BR, H), "pool_feats": (BR, H), "p_pool_feats": (BR, A), "simT": (BR, NCp)}
    got = {}
    for flags in (ss_backend, ss_backend | ROW_STORE):
        capi.set_backend(flags)
        sim = nm.prologue(*(dev[k] for k in keys), want_sim=True)
        res = {k: nm.workspace_tensor(B, T, k, s).clone() for k, s in shapes.items()}
        res["seq"], res["logp"], res["att2"] = nm.decode_greedy(B, T, dev["pnt_mask"])
        res["sim"] = sim
        got[flags] = res
    torch.cuda.synchronize()
    for k, v in got[ss_backend].items():
        assert torch.equal(v, got[ss_backend | ROW_STORE][k]), k
