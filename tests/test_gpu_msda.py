"""Multi-scale deformable attention on the GPU: csrc/dcn_msda.cu against the msda_* fixtures and against Deformable
DETR's grid_sample composition evaluated live in float64 on the CPU (out <= 1e-4, each gradient <= 1e-3 of max |ref|),
the gradients one at a time, the determinism of the two coordinate-side gradients, the drop-in module against the
restated reference, CUDA-graph replay and the kernel names."""
import pytest
import torch

import jittor_dcn_b200 as dcn
from jittor_dcn_b200 import _lib
from oracle import msda_reference
from tests.util import golden, golden_names, rel_err

pytestmark = pytest.mark.gpu

GRAD_NAMES = ("grad_value", "grad_sampling_locations", "grad_attention_weights")


def _inputs(B, M, D, Q, levels, P, seed, spread=0.05):
    """value, shapes, start index, locations (reference points plus small offsets, some outside [0, 1]), softmax-free
    weights, grad_out — float32 on the CPU."""
    g = torch.Generator().manual_seed(seed)
    L = len(levels)
    S = sum(h * w for h, w in levels)
    ss = torch.tensor(levels, dtype=torch.int64)
    value = torch.randn(B, S, M, D, generator=g)
    ref = torch.rand(B, Q, 1, 1, 1, 2, generator=g) * 1.1 - 0.05
    loc = ref + spread * torch.randn(B, Q, M, L, P, 2, generator=g)
    aw = torch.randn(B, Q, M, L, P, generator=g)
    gout = torch.randn(B, Q, M * D, generator=g)
    return value, ss, msda_reference.level_start_index_of(ss), loc, aw, gout


def _engine(value, ss, lsi, loc, aw, gout, need=(True, True, True)):
    args = [t.cuda() for t in (value, ss, lsi, loc, aw)]
    out = dcn.dcn_msda_forward(*args)
    grads = dcn.dcn_msda_backward(*args, gout.cuda(), need=need)
    torch.cuda.synchronize()
    return out.cpu(), [None if t is None else t.cpu() for t in grads]


def _check(out, grads, ref):
    assert rel_err(out.numpy(), ref[0].numpy()) <= 1e-4
    for got, exp, name in zip(grads, ref[1:], GRAD_NAMES):
        assert rel_err(got.numpy(), exp.numpy()) <= 1e-3, name


@pytest.mark.parametrize("name", golden_names("msda_"))
def test_against_the_fixtures(name):
    g = golden(name)
    t = {k: torch.as_tensor(v) for k, v in g.items()}
    out, grads = _engine(t["value"], t["spatial_shapes"], t["level_start_index"], t["sampling_locations"],
                         t["attention_weights"], t["grad_out"])
    _check(out, grads, [t[k] for k in ("out",) + GRAD_NAMES])


LIVE = {
    #  name        B  M  D    Q    levels                                   P
    "d16":        (2, 4, 16,  20, ((7, 9), (4, 5)), 4),
    "d128":       (1, 2, 128, 12, ((6, 8), (3, 4)), 2),
    "d256":       (1, 1, 256, 8,  ((5, 6),), 3),
    "l5_p8":      (1, 8, 32,  16, ((16, 20), (8, 10), (4, 5), (2, 3), (1, 2)), 8),
    "l1_p1_d64":  (3, 2, 64,  9,  ((5, 11),), 1),
}


@pytest.mark.parametrize("name", list(LIVE))
def test_against_the_live_float64_composition(name):
    B, M, D, Q, levels, P = LIVE[name]
    value, ss, lsi, loc, aw, gout = _inputs(B, M, D, Q, levels, P, seed=list(LIVE).index(name), spread=0.3)
    out, grads = _engine(value, ss, lsi, loc, aw, gout)
    _check(out, grads, msda_reference.reference(value, ss, loc, aw, gout))


@pytest.mark.parametrize("Q", ["S", 300])
def test_realistic_multi_level_shape(Q):
    """2 images, levels 32x48 / 16x24 / 8x12 / 4x6, 8 heads of 32 channels, 4 points."""
    levels = ((32, 48), (16, 24), (8, 12), (4, 6))
    S = sum(h * w for h, w in levels)
    value, ss, lsi, loc, aw, gout = _inputs(2, 8, 32, S if Q == "S" else Q, levels, 4, seed=3)
    aw = aw.softmax(-1)
    out, grads = _engine(value, ss, lsi, loc, aw, gout)
    _check(out, grads, msda_reference.reference(value, ss, loc, aw, gout))


def test_gradients_one_at_a_time():
    value, ss, lsi, loc, aw, gout = _inputs(2, 4, 32, 24, ((9, 7), (5, 4)), 4, seed=5, spread=0.2)
    ref = msda_reference.reference(value, ss, loc, aw, gout)
    _, full = _engine(value, ss, lsi, loc, aw, gout)
    for i in range(3):
        need = tuple(k == i for k in range(3))
        _, grads = _engine(value, ss, lsi, loc, aw, gout, need=need)
        for k, got in enumerate(grads):
            if k != i:
                assert got is None
        assert rel_err(grads[i].numpy(), ref[1 + i].numpy()) <= 1e-3, GRAD_NAMES[i]
        if i > 0:                                   # plain stores: the same bits with or without the other gradients
            assert torch.equal(grads[i], full[i])


def test_coordinate_side_gradients_are_deterministic():
    levels = ((32, 48), (16, 24), (8, 12), (4, 6))
    value, ss, lsi, loc, aw, gout = _inputs(2, 8, 32, 500, levels, 4, seed=11)
    _, a = _engine(value, ss, lsi, loc, aw, gout)
    _, b = _engine(value, ss, lsi, loc, aw, gout)
    assert torch.equal(a[1], b[1]) and torch.equal(a[2], b[2])


def test_inconsistent_device_shapes_stay_in_bounds():
    """spatial_shapes / level_start_index are never read by the host: levels that overrun value, negative or huge
    start indices are treated as empty in the kernels, and nothing outside value is addressed."""
    value, ss, lsi, loc, aw, gout = _inputs(1, 2, 32, 10, ((6, 8), (3, 4)), 4, seed=13, spread=0.3)
    big = torch.tensor([[600, 800], [300, 400]])                # far larger than S
    neg = torch.tensor([-5, 1 << 40])
    for s, l in ((big, lsi), (ss, neg)):
        out, grads = _engine(value, s, l, loc, aw, gout)
        assert torch.isfinite(out).all() and all(torch.isfinite(g).all() for g in grads)


@pytest.mark.parametrize("form", [2, 4])
@pytest.mark.parametrize("padding", [False, True])
def test_module_against_the_restated_reference(form, padding):
    torch.manual_seed(0)
    m = dcn.MSDeformAttn(d_model=64, n_levels=3, n_heads=2, n_points=4)
    torch.manual_seed(0)
    ref = msda_reference.MSDeformAttnRef(d_model=64, n_levels=3, n_heads=2, n_points=4).double()
    with torch.no_grad():                                   # trained-looking parameters, identical in both
        for (_, p), (_, q) in zip(m.named_parameters(), ref.named_parameters()):
            p.add_(0.05 * torch.randn_like(p))
            q.copy_(p.double())
    levels = ((10, 14), (5, 7), (3, 4))
    ss = torch.tensor(levels, dtype=torch.int64)
    lsi = msda_reference.level_start_index_of(ss)
    S = int(ss.prod(1).sum())
    B, Q = 2, 30
    query, src = torch.randn(B, Q, 64), torch.randn(B, S, 64)
    rp = torch.rand(B, Q, 3, form)
    if form == 4:
        rp[..., 2:] = rp[..., 2:] * 0.5 + 0.05
    mask = (torch.rand(B, S) < 0.2) if padding else None
    gout = torch.randn(B, Q, 64)
    # ours on the GPU in float32
    m = m.cuda()
    qd, sd, rd = (t.cuda().requires_grad_(True) for t in (query, src, rp))
    out = m(qd, rd, sd, ss.cuda(), lsi.cuda(), None if mask is None else mask.cuda())
    out.backward(gout.cuda())
    # the reference on the CPU in float64
    qr, sr, rr = (t.double().requires_grad_(True) for t in (query, src, rp))
    exp = ref(qr, rr, sr, ss, lsi, mask)
    exp.backward(gout.double())
    assert rel_err(out.detach().cpu().numpy(), exp.detach().numpy()) <= 1e-4
    for got, want, name in ((qd.grad, qr.grad, "query"), (sd.grad, sr.grad, "input_flatten"),
                            (rd.grad, rr.grad, "reference_points")):
        assert rel_err(got.cpu().numpy(), want.numpy()) <= 1e-3, name
    for (name, p), (_, q) in zip(m.named_parameters(), ref.named_parameters()):
        assert rel_err(p.grad.cpu().numpy(), q.grad.numpy()) <= 1e-3, name


def test_cuda_graph_capture_and_replay():
    levels = ((12, 16), (6, 8), (3, 4))
    value, ss, lsi, loc, aw, gout = _inputs(2, 4, 32, 50, levels, 4, seed=17)
    sv, sl, sa = (t.cuda().requires_grad_(True) for t in (value, loc, aw))
    sss, slsi, sg = ss.cuda(), lsi.cuda(), gout.cuda()

    def step():
        out = dcn.ms_deform_attn(sv, sss, slsi, sl, sa)
        return (out,) + torch.autograd.grad(out, [sv, sl, sa], sg)

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            step()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static = step()
    for seed in (21, 22):
        value, ss2, lsi2, loc, aw, gout = _inputs(2, 4, 32, 50, levels, 4, seed=seed)
        with torch.no_grad():
            sv.copy_(value.cuda())
            sl.copy_(loc.cuda())
            sa.copy_(aw.cuda())
            sg.copy_(gout.cuda())
        graph.replay()
        torch.cuda.synchronize()
        ref = msda_reference.reference(value, ss, loc, aw, gout)
        _check(static[0].detach().cpu(), [t.cpu() for t in static[1:]], ref)
    dcn.clear_workspaces()


def test_kernel_names_through_the_profiler():
    value, ss, lsi, loc, aw, gout = _inputs(1, 2, 32, 8, ((4, 6),), 2, seed=23)
    _lib.profile_begin()
    before = dcn.load().dcn_launch_count()
    _engine(value, ss, lsi, loc, aw, gout)
    launched = dcn.load().dcn_launch_count() - before
    prof = _lib.profile_end()
    assert prof["msda_fwd_kernel"][0] == 1 and prof["msda_bwd_kernel"][0] == 1
    assert launched == 2
