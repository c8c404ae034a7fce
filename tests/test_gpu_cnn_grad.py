"""Backward of the stand-alone feature extractor (``VisionCnnModule.forward`` -> ``marlc_cnn_forward_save`` /
``marlc_cnn_backward``) and of ``aggregate_messages``.

* CPU: the new entry points are exported and declared; host-side argument errors; the workspace size of one net
  worked out by hand, with and without parameter gradients.
* The forward in grad mode has the bits of the forward under ``no_grad``.
* d windows (window by window) and every parameter gradient (norm-wise) against ``torch.autograd.grad`` of
  ``O.cnn_forward`` in fp64: every feature extractor of the package, window counts 1 / 7 / 129 / 4099 (ragged CTA
  tails of the layer kernel and of ``cnn_patch_grad``, weight-gradient reductions over more than 4096 rows), the
  golden MNIST checkpoint and initial weights with perturbed GroupNorm affines.
* A cotangent on the last window only; a frozen module (no weight-gradient GEMM runs); windows that do not require
  grad; a module inside a flattened ``ModelsWrapper`` (gradients in the flat bucket); double backward; a few Adam
  steps against torch's own modules in fp64.
* ``aggregate_messages`` against fp64 autograd of ``O.aggregate_messages``.
"""
import ctypes as C
import types

import pytest
import torch

from marlclassification_b200 import _lib
from oracle import marl_oracle as O
from tests.conftest import load_golden, rel_l2
from tests.test_gpu_regimes import row_err

DEV = "cuda"

# Bounds: about 10x the worst error measured on one NVIDIA B200 (1000 W power limit), never above 1e-3.
# d windows, worst window (row_err): measured 6.8e-6 (WorldStratCnn f = 16, N = 4099)
PATCH_BOUND = 7e-5
# parameter gradients, norm-wise per tensor: measured 3.0e-5 (AidCnn f = 24, N = 4099: split-K reductions)
PARAM_BOUND = 3e-4
# parameter gradients of the one-window cotangent: measured 2.0e-6 (Resisc45Cnn)
TAIL_BOUND = 2e-5
# parameters after five Adam steps, norm-wise per tensor: measured 8.2e-7
ADAM_BOUND = 1e-5
# aggregate_messages gradient, norm-wise: measured 9.7e-8 (Na = 40)
MSG_BOUND = 1e-6

# feature extractor, window, channels of the windows
NETS = {
    "mnist_f6_c1": ("MnistCnn", 6, 1),
    "mnist_f6_c3": ("MnistCnn", 6, 3),
    "mnist_f12": ("MnistCnn", 12, 1),
    "resisc45_f12": ("Resisc45Cnn", 12, 3),
    "aid_f24": ("AidCnn", 24, 3),
    "skin_cancer_f20": ("SkinCancerCnn", 20, 3),
    "worldstrat_f16": ("WorldStratCnn", 16, 3),
}
COUNTS = [1, 7, 129, 4099]


def _module(name, weights="init", seed=0):
    """A stand-alone feature extractor on the GPU: the golden MNIST checkpoint's CNN, or the package's initial
    weights (init_layers) with GroupNorm affines and conv biases perturbed."""
    from marlclassification_b200.networks import vision
    from marlclassification_b200.networks.blocks import init_layers

    cls, f, _ = NETS[name]
    m = getattr(vision, cls)(f)
    g = torch.Generator().manual_seed(seed)
    if weights == "ckpt":
        sd = load_golden("mnist_ckpt")["state_dict"]
        pre = "_ModelsWrapper__map_obs."
        m.load_state_dict({k[len(pre):]: v for k, v in sd.items() if k.startswith(pre)})
    else:
        m.apply(init_layers)
        with torch.no_grad():
            for mod in m.modules():
                if isinstance(mod, torch.nn.GroupNorm):
                    mod.weight.copy_(1 + 0.3 * torch.randn(mod.weight.shape, generator=g))
                    mod.bias.copy_(0.2 * torch.randn(mod.bias.shape, generator=g))
                elif isinstance(mod, torch.nn.Conv2d):
                    mod.bias.copy_(0.1 * torch.randn(mod.bias.shape, generator=g))
    return m.to(DEV)


def _oracle(m, x, d_out, need_x=True):
    """fp64 autograd of O.cnn_forward: (d x, [d param in module order])."""
    f, layers, groups, first_only = m.cnn_spec
    cfg = types.SimpleNamespace(cnn_groups=groups, ch0_only=first_only)
    names = [k for k, _ in m.named_parameters()]
    ps = [p.detach().double().cpu().requires_grad_() for p in m.parameters()]
    p = {O.CNN + k.split("__layers.")[1]: t for k, t in zip(names, ps)}
    x64 = x.detach().double().cpu().requires_grad_(need_x)
    out = O.cnn_forward(p, cfg, x64)
    g = torch.autograd.grad(out, ([x64] if need_x else []) + ps, d_out.double().cpu())
    return (g[0], list(g[1:])) if need_x else (None, list(g))


def _inputs(name, n, seed=0):
    _, f, c = NETS[name]
    g = torch.Generator().manual_seed(1000 + n + seed)
    return torch.rand(n, c, f, f, generator=g).to(DEV)


# ---------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------
def test_symbols_exported_and_declared():
    lib = _lib.lib()
    for name in ("marlc_cnn_forward_save", "marlc_cnn_backward_workspace_bytes", "marlc_cnn_backward"):
        assert hasattr(lib, name)
        assert name in _lib.exported_symbols()


def _ints(v):
    return (C.c_int * len(v))(*v)


def _ptrs(n, p=256):
    return (C.c_void_p * n)(*([p] * n))


def test_workspace_bytes_by_hand():
    """Resisc45Cnn at f = 12 on 7 windows: maps 6x6, 3x3, 2x2, so 252 / 63 / 28 rows.  Each section is rounded up to
    256 bytes: dY 252*16*4 = 16128 | 63*32*4 = 8064 -> 8192 | 28*64*4 = 7168; dCol (layers 1, 2) 63*144*4 = 36288 ->
    36352 | 28*288*4 = 32256; scratch 3*cout*4 = 192 -> 256 | 384 -> 512 | 768; and with parameter gradients the
    im2col rows 252*28*4 = 28224 -> 28416 (27 taps padded to 28) | 36352 | 32256."""
    L = _lib.lib()
    cin, cout = _ints([3, 16, 32]), _ints([16, 32, 64])
    frozen = 16128 + 256 + (8192 + 36352 + 512) + (7168 + 32256 + 768)
    assert frozen == 101632
    assert L.marlc_cnn_backward_workspace_bytes(3, cin, cout, 12, 7, 0) == frozen
    assert L.marlc_cnn_backward_workspace_bytes(3, cin, cout, 12, 7, 1) == frozen + 28416 + 36352 + 32256
    assert L.marlc_cnn_backward_workspace_bytes(3, cin, cout, 12, 0, 1) == 256 + 512 + 768  # scratch only
    assert L.marlc_cnn_backward_workspace_bytes(0, cin, cout, 12, 7, 1) == 0
    assert b"bad argument" in L.marlc_last_error()
    assert L.marlc_cnn_backward_workspace_bytes(3, cin, cout, 12, -1, 1) == 0
    assert L.marlc_cnn_backward_workspace_bytes(3, cin, _ints([16, 0, 64]), 12, 7, 1) == 0
    assert b"bad shape" in L.marlc_last_error()


def test_host_argument_errors():
    """Every call fails its host-side checks before anything is launched (the dummy pointers are never read)."""
    L = _lib.lib()
    d = C.c_void_p(256)
    P4 = [_ptrs(3)] * 4

    def bwd(layers=3, cin=(3, 16, 32), cout=(16, 32, 64), groups=(2, 4, 8), f=12, img_c=3, params=P4, patch=d,
            y_save=None, d_out=d, n=7, ws=d, ws_bytes=1 << 40, d_patch=d, grads=(None,) * 4):
        y_save = _ptrs(len(cin)) if y_save is None else y_save
        return L.marlc_cnn_backward(layers, _ints(cin), _ints(cout), _ints(groups), f, img_c, *params, patch, y_save,
                                    d_out, n, ws, ws_bytes, d_patch, *grads, None)

    def err(ret, text):
        assert ret != 0
        assert text in L.marlc_last_error(), L.marlc_last_error()

    err(bwd(layers=0), b"layers unsupported")
    err(bwd(layers=7, cin=(3,) + (16,) * 6, cout=(16,) * 7, groups=(2,) * 7), b"layers unsupported")
    err(bwd(params=[None] + P4[1:]), b"null pointer")
    err(bwd(y_save=C.cast(None, C.POINTER(C.c_void_p))), b"null pointer")
    err(bwd(ws=None), b"null pointer")
    err(bwd(patch=None), b"null pointer")
    err(bwd(d_out=None), b"null pointer")
    err(bwd(params=[(C.c_void_p * 3)(256, 256, None)] + P4[1:]), b"null pointer (layer 2)")
    err(bwd(y_save=(C.c_void_p * 3)(256, None, 256)), b"null pointer (layer 1)")
    err(bwd(cin=(3, 8, 32)), b"bad shape of layer 1")
    err(bwd(groups=(2, 4, 7)), b"bad shape of layer 2")
    err(bwd(img_c=2), b"the first layer reads 3")
    err(bwd(n=-1), b"windows unsupported")
    err(bwd(ws=C.c_void_p(384)), b"not 256-byte aligned")
    err(bwd(ws_bytes=101631), b"workspace of 101631 bytes, need 101632")
    err(bwd(ws_bytes=198655, grads=(_ptrs(3), None, None, None)), b"need 198656")
    # shapes the launchers refuse: a layer kernel beyond shared memory, a first layer cnn_patch_grad cannot take
    err(bwd(cin=(3, 256), cout=(256, 256), groups=(2, 2), layers=2, f=64), b"too large for shared memory")
    err(bwd(cin=(3,), cout=(6,), groups=(2,), layers=1), b"multiple of 4 output channels")
    # ... which is fine without d_patch, and N = 0 is a no-op whatever the data pointers
    assert bwd(cin=(3,), cout=(6,), groups=(2,), layers=1, n=0, d_patch=None, patch=None, d_out=None) == 0
    fwd = L.marlc_cnn_forward_save
    assert fwd(3, _ints([3, 16, 32]), _ints([16, 32, 64]), _ints([2, 4, 8]), 12, 3, *P4, None, _ptrs(3), d, 7,
               None) != 0
    assert b"null pointer" in L.marlc_last_error()
    assert fwd(0, _ints([3]), _ints([16]), _ints([2]), 12, 3, *P4, d, None, d, 7, None) != 0
    assert b"layers unsupported" in L.marlc_last_error()


# ---------------------------------------------------------------------------------------------------------------
# GPU: the feature extractor
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(NETS))
def test_forward_bits_unchanged(name):
    m = _module(name)
    x = _inputs(name, 129)
    with torch.no_grad():
        ref = m(x)
    out = m(x)  # the parameters require grad
    assert out.grad_fn is not None and torch.equal(out.detach(), ref)
    for p in m.parameters():
        p.requires_grad_(False)
    assert m(x).grad_fn is None
    out = m(x.clone().requires_grad_())  # only the windows require grad
    assert out.grad_fn is not None and torch.equal(out.detach(), ref)


def _cases():
    for name in NETS:
        for w in (("init", "ckpt") if NETS[name][0] == "MnistCnn" else ("init",)):
            for n in COUNTS:
                yield pytest.param(name, w, n, id=f"{name}-{w}-{n}")


@pytest.mark.gpu
@pytest.mark.parametrize("name,weights,n", list(_cases()))
def test_grad_vs_fp64(name, weights, n):
    m = _module(name, weights)
    x = _inputs(name, n).requires_grad_()
    out = m(x)
    d_out = torch.randn(out.shape, generator=torch.Generator().manual_seed(n)).to(DEV)
    grads = torch.autograd.grad(out, [x, *m.parameters()], d_out)
    ref_x, ref_p = _oracle(m, x, d_out)
    cin = m.cnn_spec[1][0][0]
    e, i = row_err(grads[0][:, :cin], ref_x[:, :cin])
    assert torch.count_nonzero(grads[0][:, cin:]) == 0  # channels the network does not read: exactly 0
    pe = [rel_l2(g.cpu(), r) for g, r in zip(grads[1:], ref_p)]
    print(f"measured {name} {weights} N={n}: d_patch {e:.2e} (window {i}), params {max(pe):.2e}")
    assert e < PATCH_BOUND, (e, i)
    for (k, _), v in zip(m.named_parameters(), pe):
        assert v < PARAM_BOUND, (k, v)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["resisc45_f12", "mnist_f6_c3"])
def test_tail_probe(name):
    """A cotangent on the last window only: every other window's gradient is exactly 0, and the parameter gradients
    are those of that one window."""
    n = 129
    m = _module(name)
    x = _inputs(name, n).requires_grad_()
    out = m(x)
    d_out = torch.zeros(out.shape, device=DEV)
    d_out[-1] = torch.randn(out.shape[1], generator=torch.Generator().manual_seed(3)).to(DEV)
    grads = torch.autograd.grad(out, [x, *m.parameters()], d_out)
    assert torch.count_nonzero(grads[0][:-1]) == 0
    assert torch.count_nonzero(grads[0][-1]) > 0
    ref_x, ref_p = _oracle(m, x[-1:], d_out[-1:])
    cin = m.cnn_spec[1][0][0]
    e = rel_l2(grads[0][-1:, :cin].cpu(), ref_x[:, :cin])
    pe = [rel_l2(g.cpu(), r) for g, r in zip(grads[1:], ref_p)]
    print(f"measured tail {name}: d_patch {e:.2e}, params {max(pe):.2e}")
    assert e < PATCH_BOUND
    assert max(pe) < TAIL_BOUND, pe


def _gemm_launches():
    L = _lib.lib()
    return L.marlc_gemm_launch_count(0) + L.marlc_gemm_launch_count(1)


@pytest.mark.gpu
def test_frozen_module():
    name, n = "aid_f24", 4099
    m = _module(name)
    x = _inputs(name, n).requires_grad_()
    d_out = torch.randn(n, m.out_size, generator=torch.Generator().manual_seed(5)).to(DEV)
    n_layers = len(m.cnn_spec[1])
    out = m(x)
    torch.cuda.synchronize()
    g0 = _gemm_launches()
    (d_train,) = torch.autograd.grad(out, [x], d_out)  # parameters require grad: all their gradients are computed
    torch.cuda.synchronize()
    trainable = _gemm_launches() - g0
    for p in m.parameters():
        p.requires_grad_(False)
    out = m(x)
    torch.cuda.synchronize()
    g0 = _gemm_launches()
    out.backward(d_out)
    torch.cuda.synchronize()
    frozen = _gemm_launches() - g0
    assert frozen == n_layers - 1  # the input-gradient GEMMs only
    assert trainable == frozen + n_layers  # + one weight-gradient GEMM per layer
    assert torch.equal(x.grad, d_train)
    assert all(p.grad is None for p in m.parameters())


@pytest.mark.gpu
def test_input_without_grad():
    name, n = "resisc45_f12", 4099
    m = _module(name)
    x = _inputs(name, n)
    d_out = torch.randn(n, m.out_size, generator=torch.Generator().manual_seed(6)).to(DEV)
    with_x = torch.autograd.grad(m(x.clone().requires_grad_()), list(m.parameters()), d_out)
    out = m(x)
    assert out.requires_grad
    without = torch.autograd.grad(out, list(m.parameters()), d_out)
    # the same products; only the order of the atomic / split-K reductions may differ
    for a, b in zip(with_x, without):
        assert rel_l2(b.cpu(), a.cpu()) < 1e-6


def _wrapper():
    from marlclassification_b200.config import ModelConfig

    mc = dict(ft_extr_str="resisc45", window_size=12, hidden_size_belief=64, hidden_size_action=64,
              hidden_size_msg=16, hidden_size_msg_output=24, hidden_size_state=8, state_dim=2,
              actions=[[1, 0], [-1, 0], [0, 1], [0, -1]], nb_class=45, hidden_size_linear_belief=96,
              hidden_size_linear_action=96)
    model = ModelConfig(**mc).build_networks().to(DEV)
    model.ensure_flat()
    return model


@pytest.mark.gpu
def test_inside_models_wrapper():
    model = _wrapper()
    fe = model.feature_extractor
    bucket = model.flat_grads
    x = torch.rand(129, 3, 12, 12, generator=torch.Generator().manual_seed(8)).to(DEV)
    d_out = torch.randn(129, fe.out_size, generator=torch.Generator().manual_seed(9)).to(DEV)
    _, ref = _oracle(fe, x, d_out, need_x=False)

    def in_bucket(p):
        return p.grad is not None and p.grad.untyped_storage().data_ptr() == bucket.untyped_storage().data_ptr()

    fe(x).backward(d_out)
    for p, r in zip(fe.parameters(), ref):
        assert in_bucket(p)
        assert rel_l2(p.grad.cpu(), r) < PARAM_BOUND
    others = [p for n, p in model.named_parameters() if "map_obs" not in n]
    assert all(torch.count_nonzero(p.grad) == 0 for p in others)
    first = [p.grad.clone() for p in fe.parameters()]
    fe(x).backward(d_out)  # accumulates
    for p, g in zip(fe.parameters(), first):
        assert in_bucket(p)
        assert rel_l2(p.grad.cpu(), 2 * g.cpu()) < 1e-6
    model.zero_grad(set_to_none=True)
    fe(x).backward(d_out)
    for p, r in zip(fe.parameters(), ref):
        assert in_bucket(p)
        assert rel_l2(p.grad.cpu(), r) < PARAM_BOUND
    assert torch.count_nonzero(bucket) > 0


@pytest.mark.gpu
def test_double_backward_raises():
    m = _module("resisc45_f12")
    x = _inputs("resisc45_f12", 7).requires_grad_()
    out = m(x)
    d = torch.randn(out.shape, device=DEV, requires_grad=True)
    (gx,) = torch.autograd.grad(out, [x], d, create_graph=True)
    with pytest.raises(RuntimeError, match="differentiate twice"):
        gx.sum().backward()


@pytest.mark.gpu
def test_adam_steps_track_torch_modules():
    """Resisc45Cnn + a linear head trained for a few Adam steps on the GPU, against the same steps of torch's own
    Conv2d / GroupNorm / SiLU modules in fp64 on the CPU."""
    torch.manual_seed(11)
    fe = _module("resisc45_f12", seed=11)
    head = torch.nn.Linear(fe.out_size, 45).to(DEV)
    ref_fe = torch.nn.Sequential(
        *[mod for conv, gn in zip([c for c in fe.modules() if isinstance(c, torch.nn.Conv2d)],
                                  [g for g in fe.modules() if isinstance(g, torch.nn.GroupNorm)])
          for mod in (torch.nn.Conv2d(conv.in_channels, conv.out_channels, 3, 2, 1),
                      torch.nn.GroupNorm(gn.num_groups, gn.num_channels), torch.nn.SiLU())],
        torch.nn.Flatten(1)).double()
    ref_head = torch.nn.Linear(fe.out_size, 45).double()
    with torch.no_grad():
        for a, b in zip(list(ref_fe.parameters()) + list(ref_head.parameters()),
                        list(fe.parameters()) + list(head.parameters())):
            a.copy_(b.detach().double().cpu())
    params = list(fe.parameters()) + list(head.parameters())
    ref_params = list(ref_fe.parameters()) + list(ref_head.parameters())
    opt = torch.optim.Adam(params, lr=1e-3)
    ref_opt = torch.optim.Adam(ref_params, lr=1e-3)
    g = torch.Generator().manual_seed(12)
    for step in range(5):
        x = torch.rand(257, 3, 12, 12, generator=g)
        y = torch.randint(45, (257,), generator=g)
        opt.zero_grad()
        loss = torch.nn.functional.cross_entropy(head(fe(x.to(DEV))), y.to(DEV))
        loss.backward()
        opt.step()
        ref_opt.zero_grad()
        ref_loss = torch.nn.functional.cross_entropy(ref_head(ref_fe(x.double())), y)
        ref_loss.backward()
        ref_opt.step()
        assert abs(loss.item() - ref_loss.item()) < 1e-4 * abs(ref_loss.item())
    errs = [rel_l2(p.detach().cpu(), r.detach()) for p, r in zip(params, ref_params)]
    print(f"measured adam: params {max(errs):.2e}")
    assert max(errs) < ADAM_BOUND, errs


# ---------------------------------------------------------------------------------------------------------------
# GPU: aggregate_messages
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("na", [1, 2, 5, 40])
def test_aggregate_messages_grad(na):
    from marlclassification_b200.networks.blocks import aggregate_messages

    nb, n = 3, 13
    g = torch.Generator().manual_seed(na)
    msg = torch.randn(na, nb, n, generator=g)
    d = torch.randn(na, nb, n, generator=g)
    m = msg.to(DEV).requires_grad_()
    out = aggregate_messages(m)
    assert out.requires_grad
    (gm,) = torch.autograd.grad(out, [m], d.to(DEV))
    if na == 1:
        assert torch.count_nonzero(gm) == 0
        return
    m64 = msg.double().requires_grad_()
    (ref,) = torch.autograd.grad(O.aggregate_messages(m64), [m64], d.double())
    e = rel_l2(gm.cpu(), ref)
    print(f"measured aggregate_messages na={na}: {e:.2e}")
    assert e < MSG_BOUND


@pytest.mark.gpu
def test_aggregate_messages_without_grad():
    from marlclassification_b200.networks.blocks import aggregate_messages

    msg = torch.randn(5, 3, 7, device=DEV)
    assert not aggregate_messages(msg).requires_grad
    with torch.no_grad():
        assert not aggregate_messages(msg.clone().requires_grad_()).requires_grad
