"""The training path (tp_forward_train + tp_backward through autograd) at the batch sizes and widths it runs at, against PyTorch
autograd over the oracle's torch port IN FLOAT64 ON THE GPU (weights = the module's bf16 parameters, inputs = the same bf16
tensors, both converted to fp64; parameter gradients are sums over crops, so the reference runs in chunks of crops and adds
its fp64 gradients).

Gates (the repository's existing ones): forward rel-RMS <= 4e-3, max-abs <= 5e-3 and per-row rel-RMS <= 1.2e-2 (the `_check` of
test_fullsize_gpu.py); every parameter gradient <= 3 % rel-RMS + an absolute floor of 1 % of the k branch's first-layer bias
gradient (ln_k_1.bias and the k slice of in_proj_bias are analytically zero: the softmax is shift-invariant per window), and
<= 1.5 % rel-RMS for every gradient whose RMS is well above that floor.

What the shapes reach that the other gradient tests do not: the split-K weight gradients (R = 576 N >= 16384 rows, N >= 29), the
transposing fallbacks for hidden % 256 != 0 and widths that are not multiples of 64, the 13B width (5120), scale factors 1 / 8 / 12,
the two-pass GELU plan (TP_TRAIN_DUAL=0), crop-strided [:, 1:] CLIP views, fp32 master parameters, and buffers left unwritten.
"""
import ctypes as C
import json

import pytest
import torch

from oracle import torch_port

pytestmark = pytest.mark.gpu

REL_RMS_TOL = 4e-3
MAX_ABS_TOL = 5e-3
GRAD_TOL = 3e-2            # every gradient, on top of the floor
GRAD_TOL_STRICT = 1.5e-2   # every non-degenerate gradient

ROWS_PER_KBLOCK = 64       # kBlockK: rows of one k-block of the wgrads that contract over the batch
WGRAD_SPLITS = 4           # kWgradSplits (tp_train.inl)


@pytest.fixture(autouse=True)
def _free_cache():
    yield
    torch.cuda.empty_cache()


def _state_dict(hidden, seed):
    from tokenpacker_b200 import synthetic as syn
    return {k: torch.from_numpy(v).bfloat16() for k, v in syn.synthetic_state_dict(hidden, seed=seed).items()}


def _module(hidden, s, seed, dtype=torch.bfloat16):
    from tokenpacker_b200 import TokenPackerB200
    m = TokenPackerB200(hidden_size=hidden, scale_factor=s)
    m.load_state_dict(_state_dict(hidden, seed))
    return m.to("cuda", dtype).train()


def _inputs(n, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x0 = torch.randn(n, 576, 1024, device="cuda", generator=g).bfloat16()
    xm = torch.randn(n, 576, 4096, device="cuda", generator=g).bfloat16()
    return x0, xm


def _grad_out(n, s, hidden, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn(n, (24 // s) ** 2, hidden, device="cuda", generator=g).bfloat16()


def _train_step(m, x0, xm, grad_out):
    """One training forward + backward of the module with the given output gradient: (output, {parameter name: gradient})."""
    for p in m.parameters():
        p.grad = None
    out = m((x0, xm))
    assert out.requires_grad
    out.backward(grad_out)
    return out.detach(), {k: p.grad for k, p in m.named_parameters()}


def _reference(m, x0, xm, s, grad_out, chunk=8):
    """The same step in fp64 autograd over the torch port: output [N, M, H] and the 23 gradients, summed over chunks of crops."""
    p = {k: v.detach().double().requires_grad_(True) for k, v in m.named_parameters()}
    outs = []
    for i in range(0, x0.shape[0], chunk):
        out = torch_port.forward(p, x0[i:i + chunk].double(), xm[i:i + chunk].double(), s)
        out.backward(grad_out[i:i + chunk].double())
        outs.append(out.detach())
    return torch.cat(outs), {k: v.grad for k, v in p.items()}


def _check_forward(out, ref):
    assert out.shape == ref.shape
    d = out.double() - ref
    rel = float(d.pow(2).mean().sqrt() / ref.pow(2).mean().sqrt())
    mx = float(d.abs().max())
    # per-row check as well: no single crop / token may hide behind the batch average
    row_rel = float((d.pow(2).mean(-1).sqrt() / ref.pow(2).mean(-1).sqrt().clamp_min(1e-6)).max())
    assert rel <= REL_RMS_TOL and mx <= MAX_ABS_TOL and row_rel <= 3 * REL_RMS_TOL, (rel, mx, row_rel)
    return rel, mx


def _check_grads(grads, ref, s):
    """Every gradient against fp64; returns {name: rel-RMS}."""
    err = {}
    for k, r in ref.items():
        g = grads[k]
        assert g is not None and g.shape == r.shape and bool(torch.isfinite(g).all()), k
        err[k] = (float((g.double() - r).pow(2).mean().sqrt()), float(r.pow(2).mean().sqrt()))
    # the absolute floor for the analytically-zero gradients; at s = 1 every window has one key, so the softmax is constant and
    # the whole k and q branches have zero gradient: there the v branch's first-layer bias gradient sets the scale
    floor = 1e-2 * err["k_proj_1.0.bias" if s > 1 else "v_proj_1.0.bias"][1]
    assert floor > 0
    bad = {k: (e, r) for k, (e, r) in err.items() if e > GRAD_TOL * r + floor}
    assert not bad, (bad, err)
    rel = {k: e / r for k, (e, r) in err.items() if r > 30 * floor}
    assert max(rel.values()) < GRAD_TOL_STRICT, rel
    return rel


def _report(label, **kw):
    print(f"measured {label}: " + json.dumps(kw, sort_keys=True, default=lambda v: float(f"{v:.3g}")))


def _split_boundary_crops(n):
    """Crops that hold a row next to a split-K boundary (computed as the host does: k-blocks = ceil(R/64), per split =
    ceil(k-blocks/4), boundary rows i * per * 64), plus the first and the last crop."""
    rows = 576 * n
    kblocks = -(-rows // ROWS_PER_KBLOCK)
    per = -(-kblocks // WGRAD_SPLITS)
    crops = {0, n - 1}
    for i in range(1, WGRAD_SPLITS):
        b = i * per * ROWS_PER_KBLOCK
        if b < rows:
            crops |= {(b - 1) // 576, b // 576}
    return sorted(crops)


@pytest.mark.parametrize("n", [28, 29, 64])
def test_split_k_weight_gradients_at_split_boundaries(n):
    """N = 28 is the last batch whose 1024x1024 wgrads over R = 576 N rows run unsplit; from N = 29 on (R >= 16384) they run
    split-K over 4 k-ranges (N = 29: 261 k-blocks in 66/66/66/63) and splitk_reduce_kernel adds the fp32 partial slices.  A
    gradient with one crop non-zero is that crop's own gradient (crops are independent), so each crop next to a split boundary
    is checked against the fp64 reference of that crop alone: a dropped or doubled 64-row k-block is >= 1/9 of the signal."""
    s, hidden = 2, 256
    m = _module(hidden, s, seed=40 + n)
    x0, xm = _inputs(n, seed=41 + n)
    go = _grad_out(n, s, hidden, seed=42 + n)
    worst = {}
    for c in _split_boundary_crops(n):
        one_hot = torch.zeros_like(go)
        one_hot[c] = go[c]
        _, grads = _train_step(m, x0, xm, one_hot)
        _, ref = _reference(m, x0[c:c + 1], xm[c:c + 1], s, go[c:c + 1])
        for k, v in _check_grads(grads, ref, s).items():
            worst[k] = max(worst.get(k, 0.0), v)
    _report(f"split-K N={n} crops={_split_boundary_crops(n)}", **worst)


def test_benchmark_shape_dense():
    """The benchmark's training step: N = 64, s = 2, H = 4096, every gradient and every output row against fp64."""
    s, hidden, n = 2, 4096, 64
    m = _module(hidden, s, seed=3)
    x0, xm = _inputs(n, seed=4)
    go = _grad_out(n, s, hidden, seed=5)
    out, grads = _train_step(m, x0, xm, go)
    ref_out, ref = _reference(m, x0, xm, s, go)
    rel, mx = _check_forward(out, ref_out)
    _report("dense N=64 H=4096", forward_rel=rel, forward_max_abs=mx, **_check_grads(grads, ref, s))


SHAPES = [(1, 256, 2), (8, 256, 3), (12, 384, 2), (3, 416, 5), (4, 160, 7), (2, 5120, 2), (4, 5120, 3)]


def _shape_case(s, hidden, n):
    m = _module(hidden, s, seed=60 + s)
    x0, xm = _inputs(n, seed=61 + hidden)
    go = _grad_out(n, s, hidden, seed=62)
    out, grads = _train_step(m, x0, xm, go)
    with torch.no_grad():
        out_eval = m((x0, xm))
    ref_out, ref = _reference(m, x0, xm, s, go)
    rel, mx = _check_forward(out, ref_out)
    rel_eval, mx_eval = _check_forward(out_eval, ref_out)
    return dict(forward_rel=rel, forward_max_abs=mx, eval_rel=rel_eval, eval_max_abs=mx_eval, **_check_grads(grads, ref, s))


@pytest.mark.parametrize("s,hidden,n", SHAPES)
def test_shape_matrix(s, hidden, n):
    """Scale factors 1 / 8 / 12 (the streaming window-attention backward), widths that are not multiples of 256 (transposing
    dgrad / wgrad fallbacks for mlp.2, a separate GELU pass for mlp.0) or of 64 (160, 416), the 13B width 5120; Q = N (24/s)^2
    rows that end inside a 256-row tile.  Training forward, eval forward and every gradient against fp64."""
    _report(f"shape s={s} H={hidden} N={n}", **_shape_case(s, hidden, n))


@pytest.mark.parametrize("s,hidden,n", [(2, 256, 3), (2, 4096, 2)])
def test_shape_matrix_two_pass_gelu(s, hidden, n, monkeypatch):
    """TP_TRAIN_DUAL=0: the GELU pre-activations are stored by the GEMMs and GELU runs as its own pass (k/v_proj.0 and mlp.0)."""
    monkeypatch.setenv("TP_TRAIN_DUAL", "0")
    _report(f"two-pass GELU s={s} H={hidden} N={n}", **_shape_case(s, hidden, n))


def _clip_states(n, width, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn(n, 577, width, device="cuda", generator=g).bfloat16()


@pytest.mark.parametrize("n", [3, 30])
@pytest.mark.parametrize("views", ["both", "x0", "xm"])
def test_training_on_clip_views_is_bitwise_equal_to_copies(n, views):
    """The vision tower hands over [:, 1:] views of [N, 577, C] hidden states (crop stride 577 C).  Training reads them in
    place (3-D A map of k/v_proj.0, strided point queries); output and all 23 gradients must be bit-identical to the same
    step on contiguous copies.  N = 30 also runs the split-K wgrads."""
    s, hidden = 2, 256
    m = _module(hidden, s, seed=7)
    h0 = _clip_states(n, 1024, seed=8)
    hm = _clip_states(n, 4096, seed=9)
    x0v, xmv = h0[:, 1:], hm[:, 1:]
    assert not x0v.is_contiguous() and x0v.stride(0) == 577 * 1024 and xmv.stride(0) == 577 * 4096
    x0c, xmc = x0v.contiguous(), xmv.contiguous()
    go = _grad_out(n, s, hidden, seed=10)
    out_c, grads_c = _train_step(m, x0c, xmc, go)
    out_v, grads_v = _train_step(m, x0v if views != "xm" else x0c, xmv if views != "x0" else xmc, go)
    assert torch.equal(out_v, out_c)
    for k, g in grads_c.items():
        assert torch.equal(grads_v[k], g), k
    assert float(out_c.float().abs().sum()) > 0 and float(grads_c["k_proj_1.0.weight"].float().abs().sum()) > 0


def test_fp32_master_parameters_give_the_bf16_results():
    """A module holding fp32 copies of bf16-representable weights (mixed-precision masters) computes with the same bf16 bits:
    same output, and fp32 gradients equal to the bf16 module's gradients converted to float."""
    s, hidden, n = 2, 256, 3
    m16 = _module(hidden, s, seed=12)
    m32 = _module(hidden, s, seed=12, dtype=torch.float32)
    x0, xm = _inputs(n, seed=13)
    go = _grad_out(n, s, hidden, seed=14)
    with pytest.warns(UserWarning, match="bf16"):
        out32, g32 = _train_step(m32, x0, xm, go)
    out16, g16 = _train_step(m16, x0, xm, go)
    assert out32.dtype == torch.bfloat16 and torch.equal(out32, out16)
    for k, g in g16.items():
        assert g32[k].dtype == torch.float32 and torch.equal(g32[k], g.float()), k


@pytest.mark.parametrize("s,hidden,n", [(2, 160, 3), (2, 256, 29)])
def test_every_byte_written_and_deterministic(s, hidden, n):
    """tp_forward_train + tp_backward at the C ABI with the saved activations, the backward workspace, the output and the 23
    gradient buffers zero-filled, then filled with 0xFF bytes (NaN in bf16 and fp32), then zero-filled again: a kernel that reads a
    byte nobody wrote shows up as a NaN or as a difference.  These buffers hold data only (activations, LayerNorm statistics,
    column-sum / split-K partials; the training launches use no tile counters), so poisoning can change values but not control
    flow.  H = 160 runs the transposing fallbacks, N = 29 the split-K wgrads."""
    from tokenpacker_b200 import _lib
    lib = _lib.lib
    m = _module(hidden, s, seed=15)
    x0, xm = _inputs(n, seed=16)
    go = _grad_out(n, s, hidden, seed=17)
    params = [p.detach().contiguous() for p in m._raw_params()]
    w = _lib.TpWeights(*[t.data_ptr() for t in params])
    stream = torch.cuda.current_stream().cuda_stream
    pbytes = lib.tp_packed_bytes(hidden)
    packed = torch.zeros(pbytes, dtype=torch.uint8, device="cuda")
    _lib.check(lib.tp_pack_weights_train(C.byref(w), hidden, packed.data_ptr(), pbytes, stream), "tp_pack_weights_train")
    sbytes = lib.tp_train_saved_bytes(n, s, hidden)
    wbytes = lib.tp_backward_workspace_bytes(n, s, hidden)
    results = []
    for fill in (0x00, 0xFF, 0x00):
        saved = torch.full((sbytes,), fill, dtype=torch.uint8, device="cuda")
        ws = torch.full((wbytes,), fill, dtype=torch.uint8, device="cuda")
        out = torch.empty(n, (24 // s) ** 2, hidden, dtype=torch.bfloat16, device="cuda")
        grads = [torch.empty_like(p) for p in params]
        for t in [out] + grads:
            t.view(torch.uint8).fill_(fill)
        g = _lib.TpWeights(*[t.data_ptr() for t in grads])
        _lib.check(lib.tp_forward_train(C.byref(w), packed.data_ptr(), x0.data_ptr(), xm.data_ptr(), n, 576 * 1024, 576 * 4096, s, hidden,
                                        out.data_ptr(), saved.data_ptr(), sbytes, stream), "tp_forward_train")
        _lib.check(lib.tp_backward(C.byref(w), xm.data_ptr(), 576 * 4096, n, s, hidden, go.data_ptr(), saved.data_ptr(), C.byref(g),
                                   ws.data_ptr(), wbytes, stream), "tp_backward")
        torch.cuda.synchronize()
        results.append([out] + grads)
    names = ["output"] + [key for _, key in _lib.WEIGHT_FIELDS]
    for name, a, b, c in zip(names, *results):
        assert bool(torch.isfinite(a.float()).all()) and bool(torch.isfinite(b.float()).all()), name
        assert torch.equal(a, b) and torch.equal(a, c), name
