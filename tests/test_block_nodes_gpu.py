"""-m gpu: the two block autograd nodes of adapter4rec_b200.functional, each run on its own against an fp32 torch
statement of the same block, in every combination the model's callers produce:

  FrozenBlockFunction   out = tail(dropout(F(x)) + res)                      BertSelfOutput, BertLayer, ViTLayer
  AdapterBlockFunction  out = tail(h + W_u act(W_d h + b_d) + b_u [+ inp])   AdapterBlock.fused,
                        h = dropout(F(x)) or x                               BertAdaptedSelfOutput.forward_block

The reference rounds to bf16 where the kernels store bf16, and rebuilds the dropout mask from the (seed, offset) that
DropoutState handed out, so what is left is fp32 summation order and the final rounding.  In the adapter node each
tensor the node stored (h, s, z) is held against the statement computed from the stored tensors before it, and the
reference continues from them, as test_kernels_gpu.test_adapter_ln_fused does for K5.  Each tensor is held to the bound
tests/test_kernels_gpu.py sets for the kernel that writes it.  The node's own return values are compared (grad_fn.apply
runs its backward), so a gradient returned for an input that needs none is caught too."""
import math
import types

import pytest
import torch

import dropout_rng as R
from test_kernels_gpu import _close

pytestmark = pytest.mark.gpu
BF16 = torch.bfloat16
M, H, RANK, INTER = 333, 256, 32, 1024      # ragged M; K5 takes H % 64 == 0 and r % 8 == 0

# (rtol, atol) per returned gradient, after the kernel that writes it: the data-gradient GEMM's LINEAR epilogue (x),
# the LayerNorm backward (res / inp, gamma / beta), the weight-gradient GEMM (w_down, w_up and b_up, which is the ones
# column of dzᵀ·[s | 1]) and the column sum (b_down)
BOUNDS = {"x": (2 ** -7, 2e-2), "res": (2 ** -6, 2e-2), "inp": (2 ** -6, 2e-2),
          "gamma": (1e-3, 1e-2 * math.sqrt(M)), "beta": (1e-3, 1e-2 * math.sqrt(M)),
          "w_down": (1e-3, 2e-3 * math.sqrt(M)), "w_up": (1e-3, 2e-3 * math.sqrt(M)), "b_up": (1e-3, 2e-3 * math.sqrt(M)),
          "b_down": (1e-4, 2e-2)}


@pytest.fixture(autouse=True)
def _keep_dropout_state():
    from adapter4rec_b200 import functional as Fn
    saved = Fn.DropoutState.seed, Fn.DropoutState.counter
    yield
    Fn.DropoutState.seed, Fn.DropoutState.counter = saved


def bf(t):
    return t.to(BF16).float()


def _rand(shape, scale, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.randn(shape, generator=g, device="cuda") * scale).to(BF16)


def _init_linear(lin, scale, seed, trainable):
    with torch.no_grad():
        lin.weight.copy_(_rand(tuple(lin.weight.shape), scale, seed).float())         # bf16-exact fp32 master
        lin.bias.copy_(_rand(tuple(lin.bias.shape), 0.1, seed + 1).float())
    lin.requires_grad_(trainable)
    return lin


def _frozen_f(kind):
    """(dense, intermediate) of F: the frozen H -> H dense, or the frozen FFN pair H -> INTER -> H"""
    from adapter4rec_b200.model.layers import Linear
    if kind == "dense":
        return _init_linear(Linear(H, H).cuda(), H ** -0.5, 11, False), None
    return (_init_linear(Linear(INTER, H).cuda(), INTER ** -0.5, 13, False),
            _init_linear(Linear(H, INTER).cuda(), H ** -0.5, 11, False))


def _layernorm(trainable):
    from adapter4rec_b200.model.layers import LayerNorm
    ln = LayerNorm(H, eps=1e-12).cuda()
    with torch.no_grad():
        ln.weight.copy_(1 + 0.1 * _rand((H,), 1.0, 21).float())
        ln.bias.copy_(0.1 * _rand((H,), 1.0, 22).float())
    return ln.requires_grad_(trainable)


def _dropout(p):
    """hands the next draw a counter past 2^32; returns (keep mask * scale, or 1.0, check of the draw's size)"""
    from adapter4rec_b200 import functional as Fn
    Fn.DropoutState.manual_seed(0xB10C5)
    Fn.DropoutState.counter = off = (1 << 32) + 5
    seed = Fn.DropoutState.seed
    keep = R.element_keep(seed, off, p, torch.arange(M, device="cuda"), H).float() * R.keep_scale(p) if p > 0 else 1.0

    def check_draw():
        assert Fn.DropoutState.counter == off + ((M * H + 3) // 4 if p > 0 else 0), "one draw of F's output, or none"
    return keep, check_draw


def _gelu_grad(u):
    t = u.detach().clone().requires_grad_(True)
    torch.nn.functional.gelu(t).backward(torch.ones_like(t))
    return t.grad


def _f_fwd(x, dense, inter):
    """F(x) up to its last GEMM's epilogue (fp32) and the FFN pre-activation u (bf16-rounded, None for the dense)"""
    u = None
    if inter is not None:
        pre = x @ inter.weight.detach().t() + inter.bias.detach()
        u, x = bf(pre), bf(torch.nn.functional.gelu(pre))
    return x @ dense.weight.detach().t() + dense.bias.detach(), u


def _f_bwd(dh, u, dense, inter, fold):
    if inter is not None:
        dh = bf((dh @ dense.weight.detach()) * _gelu_grad(u))
    w = (dense if inter is None else inter).weight.detach()
    return bf(dh @ w + (0.0 if fold is None else fold))


def _layernorm_ref(z, ln, dout):
    """(LN(z), dz, dgamma, dbeta) in fp32"""
    zf = z.clone().requires_grad_(True)
    g, b = ln.weight.detach().clone().requires_grad_(True), ln.bias.detach().clone().requires_grad_(True)
    y = torch.nn.functional.layer_norm(zf, (H,), g, b, ln.eps)
    y.backward(dout)
    return y.detach(), zf.grad, g.grad, b.grad


def _check(got, want):
    """every value the node's backward returned: the reference where the input needs a gradient, else None"""
    for name, g in got.items():
        if name not in want:
            assert g is None, "%s: a gradient was returned for an input that needs none" % name
    for name, ref in want.items():
        assert got[name] is not None, "%s: no gradient returned" % name
        _close(got[name], ref, *BOUNDS[name], name)


def _cases(shapes):
    """(F, tail, res, ln_trainable, p, x_grad) over the LayerNorm's trainability and the dropout where they exist, and with
    and without a gradient for x, where at least one input of the node needs a gradient (adapters always do)"""
    out = []
    for F, tail, res, adapter in shapes:
        for ln_trainable in ((False, True) if tail == "ln" else (False,)):
            for p in ((0.0, 0.1) if tail == "ln" and F is not None else (0.0,)):
                for x_grad in (True, False):
                    if adapter or x_grad or ln_trainable or res == "other":
                        out.append(pytest.param(F, tail, res, ln_trainable, p, x_grad, id="-".join(map(str, (
                            F, tail, res, "ln_trainable" if ln_trainable else "ln_frozen", p, "dx" if x_grad else "no_dx")))))
    return out


# F, tail, res: BertSelfOutput (dense, LayerNorm, the sub-layer input), BertOutput (FFN, LayerNorm, res is x), ViTOutput
# (FFN, no tail, the skip input), the FFN in front of an adapter wrapper (no tail, no residual)
FROZEN = _cases([("dense", "ln", "other", False), ("ffn", "ln", "x", False), ("ffn", None, "other", False),
                 ("ffn", None, None, False)])


@pytest.mark.parametrize("F,tail,res,ln_trainable,p,x_grad", FROZEN)
def test_frozen_block_node(F, tail, res, ln_trainable, p, x_grad):
    from adapter4rec_b200 import functional as Fn
    dense, inter = _frozen_f(F)
    ln = _layernorm(ln_trainable) if tail == "ln" else None
    x = _rand((M, H), 1.0, 1).requires_grad_(x_grad)
    r = {None: None, "x": x, "other": _rand((M, H), 1.0, 2).requires_grad_(True)}[res]
    keep, check_draw = _dropout(p)
    out = Fn.frozen_block(x, r, dense, intermediate=inter, ln=ln, p=p)
    check_draw()
    dout = _rand((M, H), 1.0, 3)
    got = dict(zip(Fn.FrozenBlockFunction.ARGS, out.grad_fn.apply(dout)))

    acc, u = _f_fwd(x.detach().float(), dense, inter)
    z = bf(acc * keep + (0.0 if r is None else r.detach().float()))
    want = {}
    if ln is None:
        ref_out, dz, dzm = z, dout.float(), dout.float()
    else:
        ref_out, dzf, dg, db = _layernorm_ref(z, ln, dout.float())
        dz, dzm = bf(dzf), bf(dzf * keep)
        if ln_trainable:
            want["gamma"], want["beta"] = dg, db
    if x_grad:
        want["x"] = _f_bwd(dzm, u, dense, inter, dz if res == "x" else None)
    if res == "other":
        want["res"] = dz
    _close(out, ref_out, 2 ** -7, 1e-2 if ln is not None else 2e-2, "out")
    _check(got, want)


# F, tail, inp: AdapterBlock.forward (no tail, no inp: SASRec / ViT adapters; + inp: the enclosing skip connection),
# forward_from_dense (LayerNorm after the wrapper's dense), forward_block (BertSelfOutput: dense; BertOutput: FFN, inp is x)
ADAPTER = _cases([(None, None, None, True), (None, "inp", "other", True), (None, "ln", "other", True),
                  ("dense", "ln", "other", True), ("ffn", "ln", "x", True)])


@pytest.mark.parametrize("F,tail,inp,ln_trainable,p,x_grad", ADAPTER)
@pytest.mark.parametrize("act", ["relu", "gelu"])
def test_adapter_block_node(act, F, tail, inp, ln_trainable, p, x_grad):
    from adapter4rec_b200 import functional as Fn
    from adapter4rec_b200.model.modules import AdapterBlock
    adapter = AdapterBlock(types.SimpleNamespace(adapter_activation="GELU" if act == "gelu" else "RELU"), H, RANK).cuda()
    _init_linear(adapter.fc_down, 0.05, 31, True)
    _init_linear(adapter.fc_up, 0.05, 33, True)
    dense, inter = _frozen_f(F) if F is not None else (None, None)
    ln = _layernorm(ln_trainable) if tail == "ln" else None
    x = _rand((M, H), 1.0, 1).requires_grad_(x_grad)
    i = {None: None, "x": x, "other": _rand((M, H), 1.0, 2).requires_grad_(True)}[inp]
    keep, check_draw = _dropout(p)
    out = Fn.adapter_block(x, i, adapter, ln=ln, dense=dense, intermediate=inter, p=p)
    check_draw()
    dout = _rand((M, H), 1.0, 3)
    got = dict(zip(Fn.AdapterBlockFunction.ARGS, out.grad_fn.apply(dout)))

    h_k, z_k, _, _, _, s_k, _, _, _, _ = out.grad_fn.saved_tensors      # h, z and s as the node's kernels wrote them

    # Each tensor the node stored is held against the fp32 statement computed from the stored tensors before it, to the
    # bound of the kernel that wrote it (test_adapter_ln_fused feeds K5 and its reference the same h and takes the
    # LayerNorm of the kernel's own z).  The epilogues evaluate GELU in a fast form (within 1/8 bf16 ulp), so a bf16 value
    # may round the other way than in fp32 torch; carried further, that flips a ReLU mask or moves a 333-row
    # weight-gradient sum by more than a rounding.
    u = None
    h = x.detach().float()
    if dense is not None:
        acc, u = _f_fwd(h, dense, inter)
        _close(h_k, bf(acc * keep), 2 ** -7, 2e-2, "h")
        h = h_k.float()
    wd, bd = adapter.fc_down.weight.detach(), adapter.fc_down.bias.detach()
    wu, bu = adapter.fc_up.weight.detach(), adapter.fc_up.bias.detach()
    pre = h @ wd.t() + bd
    s = bf(torch.nn.functional.gelu(pre) if act == "gelu" else torch.relu(pre))
    _close(s_k, s, 2 ** -7, 1e-3, "s")
    zsum = h + s @ wu.t() + bu + (0.0 if i is None else i.detach().float())
    s = s_k.float()
    want = {}
    if ln is None:
        _close(out, zsum, 2 ** -7, 2e-2, "out")
        dz = dout.float()
    else:
        _close(z_k, zsum, 2 ** -7, 2e-2, "z")
        ref_out, dzf, dg, db = _layernorm_ref(z_k.float(), ln, dout.float())
        _close(out, ref_out, 2 ** -7, 1e-2, "out")
        dz = bf(dzf)
        if ln_trainable:
            want["gamma"], want["beta"] = dg, db
    ds = bf((dz @ wu) * (_gelu_grad(bf(pre)) if act == "gelu" else (s > 0).float()))
    want.update(w_down=ds.t() @ h, b_down=ds.sum(0), w_up=dz.t() @ s, b_up=dz.sum(0))
    if x_grad:
        dh = bf((ds @ wd + dz) * keep)
        want["x"] = dh if dense is None else _f_bwd(dh, u, dense, inter, dz if inp == "x" else None)
    if inp == "other":
        want["inp"] = dz
    _check(got, want)
