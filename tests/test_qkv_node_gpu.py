"""-m gpu: the fused q|k|v (+ LoRA) projection node (functional.QKVFunction, called through Fn.qkv) run on its own
against an fp32 torch statement of the same projection, in the configurations the model's callers produce:

  qkv = x·[Wq;Wk;Wv]ᵀ + [bq;bk;bv] + Σ_j (x·A_jᵀ)·B_jᵀ / r_j      BertSelfAttention, ViTSelfAttention,
                                                                  MultiHeadedAttention.presum, LoRALinear.forward

The reference rounds to bf16 where the kernels store bf16 (the operands B / r, T, qkv, dT) and continues from the T the
node stored, so what is left is fp32 summation order and the final rounding.  Each tensor is held to the bound
tests/test_kernels_gpu.py sets for the kernel that writes it.  The node's own return values are compared (grad_fn.apply
runs its backward), so a gradient returned for an input that needs none is caught too."""
import math

import pytest
import torch

from test_kernels_gpu import _close

pytestmark = pytest.mark.gpu
BF16 = torch.bfloat16
M, H = 333, 256                 # ragged M
WGRAD = (1e-3, 2e-3 * math.sqrt(M))
# (rtol, atol) per returned gradient, after the kernel that writes it: the data-gradient GEMM (x), the weight-gradient
# GEMM (weight, lora_A, lora_B, and the bias when it is the ones column of dqkvᵀ·[T | 1]) or the column sum (bias)
BOUNDS = {"x": (2 ** -7, 2e-2), "weight": WGRAD, "lora_A": WGRAD, "lora_B": WGRAD, "bias_ones": WGRAD,
          "bias": (1e-4, 2e-2)}


def bf(t):
    return t.to(BF16).float()


def _rand(shape, scale, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.randn(shape, generator=g, device="cuda") * scale).to(BF16)


def _proj(seed, r=None, bias=True, w_train=False, b_train=True):
    """one projection H -> H: a Linear (r None) or a LoRALinear of rank r (r = 0: no LoRA pair, weight trainable),
    parameters bf16-exact"""
    from adapter4rec_b200.model.layers import Linear, LoRALinear
    m = (Linear(H, H, bias=bias) if r is None else LoRALinear(H, H, r=r, bias=bias)).cuda()
    with torch.no_grad():
        for i, (name, p) in enumerate(m.named_parameters()):
            scale = {"weight": H ** -0.5, "bias": 0.1, "lora_A": H ** -0.5, "lora_B": 1.0}[name]
            p.copy_(_rand(tuple(p.shape), scale, seed + i).float())
    if r is None:
        m.weight.requires_grad_(w_train)
    if bias:
        m.bias.requires_grad_(b_train)
    return m


# the projections of each case: BERT / ViT (query, key, value with biases; LoRA on q and v, the key frozen), SASRec
# (bias-free w_Q / w_K / w_V; the image tree's surgery puts r = 4 on w_Q and a LoRALinear(r=0) on w_V), full fine-tuning,
# and a stand-alone LoRALinear
CASES = {
    "frozen": lambda: [_proj(10, b_train=False), _proj(20, b_train=False), _proj(30, b_train=False)],
    "frozen_no_bias": lambda: [_proj(10, bias=False), _proj(20, bias=False), _proj(30, bias=False)],
    "lora_r8": lambda: [_proj(10, r=8), _proj(20, b_train=False), _proj(30, r=8)],
    "lora_r12": lambda: [_proj(10, r=12), _proj(20, b_train=False), _proj(30, r=12)],
    "lora_r32": lambda: [_proj(10, r=32), _proj(20, b_train=False), _proj(30, r=32)],       # ranks fill T: no ones column
    "lora_q4_v0": lambda: [_proj(10, r=4), _proj(20, bias=False, w_train=True), _proj(30, r=0)],
    "standalone_r8": lambda: [_proj(10, r=8)],
    "full_ft": lambda: [_proj(10, w_train=True), _proj(20, w_train=True), _proj(30, w_train=True)],
    "full_ft_frozen_bias": lambda: [_proj(10, w_train=True, b_train=False), _proj(20, w_train=True, b_train=False),
                                    _proj(30, w_train=True, b_train=False)],
}


def _slots(mods):
    slots, off = [], 0
    for j, m in enumerate(mods):
        if getattr(m, "lora_A", None) is not None:
            slots.append((j, off, m.r))
            off += m.r
    return slots, off < 64


def _forward_ref(x, mods, T_k):
    """(T, qkv) in fp32 with bf16 roundings; qkv continues from T_k, the T the node stored"""
    slots, ones = _slots(mods)
    T = torch.zeros((M, 64), device="cuda")
    if ones:
        T[:, 63] = 1.0
    qkv = []
    for j, m in enumerate(mods):
        q = x @ m.weight.detach().t() + (0.0 if m.bias is None else m.bias.detach())
        for jj, o, r in slots:
            if jj == j:
                T[:, o:o + r] = x @ m.lora_A.detach().t()
                q = q + T_k[:, o:o + r] @ bf(m.lora_B.detach() * (1.0 / r)).t()
        qkv.append(q)
    return bf(T), bf(torch.cat(qkv, 1))


def _backward_ref(x, mods, T_k, dqkv, dskip, x_grad):
    """{argument name of QKVFunction: gradient} for every input that needs one"""
    slots, ones = _slots(mods)
    want = {}
    dx = torch.zeros((M, H), device="cuda") if dskip is None else dskip.clone()
    for j, m in enumerate(mods):
        dq = dqkv[:, j * H:(j + 1) * H]
        dx = dx + dq @ m.weight.detach()
        if m.weight.requires_grad:
            want[(j, "weight")] = dq.t() @ x
        if m.bias is not None and m.bias.requires_grad:
            want[(j, "bias")] = dq.sum(0)
        for jj, o, r in slots:
            if jj == j:
                dT = bf(dq @ bf(m.lora_B.detach() * (1.0 / r)))
                dx = dx + dT @ m.lora_A.detach()
                want[(j, "lora_A")] = dT.t() @ x
                want[(j, "lora_B")] = (dq.t() @ T_k[:, o:o + r]) / r
    if x_grad:
        want["x"] = dx
    return want, ones


def _check(got, want, ones):
    for name, g in got.items():
        if name not in want:
            assert g is None, "%s: a gradient was returned for an input that needs none" % (name,)
    for name, ref in want.items():
        assert got[name] is not None, "%s: no gradient returned" % (name,)
        kind = name if isinstance(name, str) else name[1]
        _close(got[name], ref, *BOUNDS["bias_ones" if kind == "bias" and ones else kind], str(name))


PARAMS = [(case, None, True) for case in CASES] + [
    ("lora_r8", "both", True), ("lora_r8", "unused", True), ("lora_r8", "alone", True),
    ("lora_r8", None, False), ("lora_r8", "both", False), ("full_ft", None, False)]


@pytest.mark.parametrize("case,skip,x_grad", PARAMS)
def test_qkv_node(case, skip, x_grad):
    """skip: None (one output), "both" (qkv and the skip output receive gradients), "unused" (only qkv), "alone" (only
    the skip output)"""
    from adapter4rec_b200 import functional as Fn
    mods = CASES[case]()
    x = _rand((M, H), 1.0, 1).requires_grad_(x_grad)
    out = Fn.qkv(x, mods, Fn.QKVCache(), skip=skip is not None)
    qkv, skip_out = out if skip is not None else (out, None)
    if skip is not None and not x_grad:
        assert skip_out is x, "with x needing no gradient the skip input is x itself"
    grad_fn = qkv.grad_fn
    T_k = grad_fn.saved_tensors[1]
    T_ref, qkv_ref = _forward_ref(x.detach().float(), mods, None if T_k is None else T_k.float())
    if T_k is not None:
        _close(T_k, T_ref, 2 ** -7, 1e-2, "T")
    else:
        assert not _slots(mods)[0], "a LoRA projection stores T"
    _close(qkv, qkv_ref, 2 ** -7, 2e-2, "qkv")

    dqkv = None if skip == "alone" else _rand((M, len(mods) * H), 1.0, 2)
    dskip = _rand((M, H), 1.0, 3) if skip in ("both", "alone") and x_grad else None
    with_skip = skip is not None and x_grad
    names = Fn.QKVFunction.args(len(mods))
    got = grad_fn.apply(dqkv, dskip) if with_skip else grad_fn.apply(dqkv)
    assert len(got) == len(names)
    got = dict(zip(names, got))
    if skip == "alone":
        assert got.pop("x") is dskip, "only the skip output was used: its gradient is x's"
        assert all(g is None for g in got.values())
        return
    want, ones = _backward_ref(x.detach().float(), mods, None if T_k is None else T_k.float(), dqkv.float(),
                               None if dskip is None else dskip.float(), x_grad)
    _check(got, want, ones)


def _grads(out, dqkv):
    return [None if g is None else g.clone() for g in out.grad_fn.apply(dqkv)]


def _train_step(mods, seed):
    """change every trainable tensor the way the Adam kernel does (through raw pointers: torch's version counters do not
    see it), then announce the step"""
    from adapter4rec_b200 import functional as Fn
    with torch.no_grad():
        for i, p in enumerate(t for m in mods for t in m.parameters() if t.requires_grad):
            v = p._version
            p.data.add_(_rand(tuple(p.shape), 0.05, seed + i).float())
            assert p._version == v
    Fn.bump_param_epoch()


@pytest.mark.parametrize("case", ["lora_r8", "lora_r32", "full_ft"])
def test_qkv_cache_rebuilds(case):
    """after an optimizer step (and after an in-place change of a frozen weight), the next forward uses the new values:
    it matches the node run with a fresh cache bit for bit"""
    from adapter4rec_b200 import functional as Fn
    mods = CASES[case]()
    x = _rand((M, H), 1.0, 1).requires_grad_(True)
    dqkv = _rand((M, 3 * H), 1.0, 2)
    cache = Fn.QKVCache()
    before = Fn.qkv(x, mods, cache)
    _train_step(mods, 50)
    after = Fn.qkv(x, mods, cache)
    fresh = Fn.qkv(x, mods, Fn.QKVCache())
    assert torch.equal(after, fresh) and not torch.equal(after, before)
    for a, b in zip(_grads(after, dqkv), _grads(fresh, dqkv)):
        assert (a is None and b is None) or torch.equal(a, b)
    with torch.no_grad():
        mods[1].weight.mul_(0.5)                                        # bumps the version counter
    after = Fn.qkv(x, mods, cache)
    assert torch.equal(after, Fn.qkv(x, mods, Fn.QKVCache()))


def test_qkv_backward_of_an_earlier_forward():
    """two forwards with different parameters, then the backward of the FIRST: its gradients are those of the first
    forward's parameters"""
    from adapter4rec_b200 import functional as Fn
    mods = CASES["lora_r8"]()
    x = _rand((M, H), 1.0, 1).requires_grad_(True)
    dqkv = _rand((M, 3 * H), 1.0, 2)
    ref = _grads(Fn.qkv(x, mods, Fn.QKVCache()), dqkv)
    cache = Fn.QKVCache()
    first = Fn.qkv(x, mods, cache)
    _train_step(mods, 50)
    second = Fn.qkv(x, mods, cache)
    assert not torch.equal(first, second)
    for a, b in zip(_grads(first, dqkv), ref):
        assert (a is None and b is None) or torch.equal(a, b)
