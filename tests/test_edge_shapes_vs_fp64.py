"""Kernels against an exact (fp64, autograd, on the device) evaluation of the oracle at the shapes where hand-written
kernels go wrong: ragged row counts (a partial last 128-row tile, S not a multiple of 32, one-row batches), backward
batches that span several chunks and end in a chunk of one ray or in a partial tile, and the edges of the stand-alone
kernels (S = 2 and S > 1536 in compositing, idle warps of the last block, a resampling merge padded up to 4096, the
Huber loss's grid-stride loop).  The documented accumulate (+=) contract of every *_backward entry point is checked
through the C ABI with prefilled gradient buffers, as sparf_b200.distributed uses it.

Yardstick (as in test_tc_engine.py / test_cuda_parity.py): a kernel is compared with the fp64 truth and gated against
the distance of a plain fp32 computation of the same operation from that truth (the SIMT engine for the MLP, the fp32
oracle for the stand-alone kernels), with a floor.  Errors are max-normalised per tensor (max|a - b| / max|b|) unless
stated; ray gradients use relative L2.
"""
import ctypes
import math

import numpy as np
import pytest
import torch

import common

pytestmark = pytest.mark.gpu

KEYS = sum([["mlp_feat.%d.weight" % i, "mlp_feat.%d.bias" % i] for i in range(8)], []) + \
    ["mlp_rgb.0.weight", "mlp_rgb.0.bias", "mlp_rgb.1.weight", "mlp_rgb.1.bias"]
C2F = (0.4, 0.7)
TILE = 128          # rows per tcgen05 tile
CHUNK_TILES = 1024  # row tiles per tcgen05 backward chunk


def _maxnorm(a, b, floor=1e-30):
    """max|a - b| / max(max|b|, floor) in float64."""
    a, b = a.double(), b.double()
    return ((a - b).abs().max() / b.abs().max().clamp_min(floor)).item()


def _rel_l2(a, b):
    a, b = a.double(), b.double()
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


def _tc_available():
    from sparf_b200 import _lib
    return bool(_lib.lib().sparf_engine_available(_lib.ENGINE_TC_3X))


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


# ================================================================================================ A. MLP engines
def _chunk_rays(R, S):
    """Rays per tcgen05 backward chunk: whole 128-row tiles, <= 1024 tiles (mirrors bwd_chunk_rays in mlp_tc.cu)."""
    unit = TILE // math.gcd(S, TILE)
    n = CHUNK_TILES * TILE // S
    return min(R, max(unit, n - n % unit))


def _tail_rows(R, S):
    """[R, S] bool: the rows the backward handles last and separately -- the partial last tile and, for a batch of
    several chunks, the whole last chunk."""
    M = R * S
    row = torch.arange(M, device="cuda").reshape(R, S)
    tail = row >= (M // TILE) * TILE if M % TILE else torch.zeros(R, S, dtype=torch.bool, device="cuda")
    nrc = _chunk_rays(R, S)
    if nrc < R:
        tail = tail | (row >= ((R - 1) // nrc) * nrc * S)
    return tail


def _mlp_problem(R, S, c2f, seed):
    opt = common.make_opt(S=S, barf_c2f=c2f)
    sd = common.det_weights(opt, seed, peaky=True, sigma_bias=-3.0, progress=0.6 if c2f else None)
    params = [sd[k].cuda() for k in KEYS]
    g = torch.Generator(device="cpu").manual_seed(seed)
    o = (torch.randn(R, 3, generator=g) * 0.5).cuda()
    d = torch.randn(R, 3, generator=g)
    d = (d / d.norm(dim=-1, keepdim=True) * (1 + 0.2 * torch.rand(R, 1, generator=g))).cuda()
    t = torch.sort(torch.rand(R, S, generator=g) * 4 + 1.2, dim=1).values.cuda()
    noise = (torch.randn(R, S, generator=g) * 0.3).cuda()
    return params, o, d, t, noise, sd["progress"].cuda()


def _upstream(R, S, seed):
    """Fixed upstream gradients on sigma and rgb, the tail rows scaled up so that they carry about a third of each
    gradient's energy (a kernel that drops or double-counts them then moves every gradient by far more than the gate);
    returns (g_sigma, g_rgb, tail mask)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    gs = torch.randn(R, S, device="cuda", generator=g) * 1e-3
    gc = torch.randn(R, S, 3, device="cuda", generator=g) * 1e-3
    tail = _tail_rows(R, S)
    n_tail = int(tail.sum())
    n_head = R * S - n_tail
    f = max(1.0, math.sqrt(n_head / (3.0 * n_tail))) if n_tail and n_head else 1.0
    w = torch.where(tail, torch.full_like(gs, f), torch.ones_like(gs))
    return gs * w, gc * w[..., None], tail


def _fp64_mlp(params, o, d, t, noise, prog, c2f, gs, gc, tail):
    """Exact outputs and gradients.  The sample points carry the fp32 value the kernels compute (x = o + d t, rounded
    twice) and the exact derivative w.r.t. o and d.  Gradients are returned for the full upstream gradient and for the
    upstream gradient with its tail rows set to zero (the negative control)."""
    from oracle import sparf_oracle as O
    p64 = {k: p.double().requires_grad_(True) for k, p in zip(KEYS, params)}
    p64["progress"] = prog.double()
    o64, d64, t64 = o.double().requires_grad_(True), d.double().requires_grad_(True), t.double()
    pts32 = o[:, None] + d[:, None] * t[..., None]
    pts = pts32.double() + (o64 - o64.detach())[:, None] + (d64 - d64.detach())[:, None] * t64[..., None]
    dens, rgb = O.mlp_forward(p64, pts[None], d64[None], barf_c2f=c2f, noise=noise.double()[None])
    dens, rgb = dens[0], rgb[0]
    inputs = [p64[k] for k in KEYS] + [o64, d64]
    keep = (~tail).double()
    gs64, gc64 = gs.double(), gc.double()
    head = torch.autograd.grad((dens * gs64 * keep).sum() + (rgb * gc64 * keep[..., None]).sum(), inputs, retain_graph=True)
    tl = torch.autograd.grad((dens * gs64 * (1 - keep)).sum() + (rgb * gc64 * (1 - keep)[..., None]).sum(), inputs)
    full = [a + b for a, b in zip(head, tl)]
    return dens.detach(), rgb.detach(), full, list(head)


def _run_engine(eng, tape, rays, params, o, d, t, noise, prog, c2f, gs, gc):
    """One forward + backward through ops (autograd); rays: request d_origins / d_dirs."""
    from sparf_b200 import ops
    spec = ops.MLPSpec(barf_c2f=c2f)
    ops.USE_TAPE[0] = tape
    try:
        ps = [p.clone().requires_grad_(True) for p in params]
        oo, dd = o.clone().requires_grad_(rays), d.clone().requires_grad_(rays)
        s, c = ops.mlp_forward(spec, oo, dd, t, ps, noise=noise, progress=prog, engine=eng)
        ((s * gs).sum() + (c * gc).sum()).backward()
        torch.cuda.synchronize()
    finally:
        ops.USE_TAPE[0] = True
    return s.detach(), c.detach(), [p.grad for p in ps], ((oo.grad, dd.grad) if rays else None)


MLP_SHAPES = [(1, 1, None), (3, 33, None), (77, 65, None), (129, 200, C2F), (1025, 128, None), (2000, 65, None),
              (700, 200, C2F)]


@pytest.mark.parametrize("R,S,c2f", MLP_SHAPES)
def test_mlp_engines_vs_fp64_ragged(R, S, c2f):
    """SIMT fp32, TC_3X (taped and recompute) and TC_3X_W1 vs fp64 at ragged shapes, sigma noise on:
      (1,1) one row; (3,33) one partial tile, rays straddle warps; (77,65) partial last tile of 13 rows;
      (129,200,c2f) rays span tiles unaligned; (1025,128) second backward chunk of ONE ray; (2000,65) chunks of
      1920 + 80 rays, the last ending in a partial tile; (700,200,c2f) chunks of 640 + 60 rays (unit 16).
    Gates (the yardstick of test_tc_engine.py::test_tc_backward_matches_simt), measured worst on a B200 in brackets:
      * forward sigma / rgb: every engine within 1e-3 of fp64 (SIMT 1.2e-5 .. 1.9e-4: the fp32 encoding of the
        2^9 pi band), tcgen05 within max(5e-5, 4x SIMT) (1.0x .. 1.4x);
      * taped forward outputs bit-identical to the plain forward (sparf_b200.h: "identical to sparf_mlp_forward");
      * every parameter gradient: TC_3X taped within max(2e-3, 4x SIMT's distance from fp64) (worst tensor 6.9e-5 ..
        4.4e-2, SIMT 6.1e-5 .. 4.4e-2), the recompute path within max(2e-3, 6x SIMT) (4.1x, see below);
        TC_3X_W1 within 3e-2 of TC_3X (3.5e-3 .. 5.4e-3);
      * backward with and without ray gradients (different side-stream topology): parameter gradients agree to 1e-5
        (<= 1.3e-6);
      * d_origins / d_dirs (relative L2): tcgen05 within max(1e-3, 4x SIMT) (SIMT 1.3e-4 .. 1.5e-2, tcgen05 <= 2x);
      * negative control: the fp64 gradient with the tail's upstream gradient zeroed is >= 3x the TC_3X gate away
        from the full one in every tensor (measured 3.4x .. 16x; 500x and 2.4x for the one-tile batches).
    """
    from sparf_b200 import _lib, ops
    if not _tc_available():
        pytest.skip("tcgen05 engine not available")
    params, o, d, t, noise, prog = _mlp_problem(R, S, c2f, seed=R + S)
    gs, gc, tail = _upstream(R, S, seed=R * 7 + S)
    runs = {"simt": (_lib.ENGINE_SIMT_FP32, True), "tc": (_lib.ENGINE_TC_3X, True),
            "tc_recompute": (_lib.ENGINE_TC_3X, False), "tc_w1": (_lib.ENGINE_TC_3X_W1, True)}
    res = {}
    for name, (eng, tape) in runs.items():
        with_rays = _run_engine(eng, tape, True, params, o, d, t, noise, prog, c2f, gs, gc)
        no_rays = _run_engine(eng, tape, False, params, o, d, t, noise, prog, c2f, gs, gc)
        res[name] = (with_rays, no_rays)
    s64, c64, truth, control = _fp64_mlp(params, o, d, t, noise, prog, c2f, gs, gc, tail)
    report = []

    # forward vs fp64, and the taped forward == the plain forward
    spec = ops.MLPSpec(barf_c2f=c2f)
    e_fwd = {}
    for name, (eng, tape) in runs.items():
        s, c = res[name][0][0], res[name][0][1]
        e_fwd[name] = max(_maxnorm(s, s64), _maxnorm(c, c64))
        assert e_fwd[name] < 1e-3, (name, "forward", e_fwd[name])
        if eng != _lib.ENGINE_SIMT_FP32 and tape:
            with torch.no_grad():
                s_plain, c_plain = ops.mlp_forward(spec, o, d, t, params, noise=noise, progress=prog, engine=eng)
            assert torch.equal(s, s_plain) and torch.equal(c, c_plain), (name, "taped forward differs from the plain one")
    for name in ("tc", "tc_recompute", "tc_w1"):
        assert e_fwd[name] < max(5e-5, 4 * e_fwd["simt"]), (name, e_fwd[name], e_fwd["simt"])
    report.append("fwd " + " ".join("%s %.1e" % kv for kv in e_fwd.items()))

    # parameter gradients vs fp64
    n_par = len(KEYS)
    worst = {k: 0.0 for k in runs}
    worst_w1_vs_tc = 0.0
    margin, margin_at = float("inf"), None
    for i in range(n_par):
        tr = truth[i]
        e = {name: _maxnorm(res[name][0][2][i], tr) for name in runs}
        for k in runs:
            worst[k] = max(worst[k], e[k])
        gate = max(2e-3, 4 * e["simt"])
        assert e["tc"] < gate, (KEYS[i], "tc taped", e["tc"], e["simt"])
        # the recompute path re-runs the forward with bf16 halves (the taped forward keeps fp16 halves): measured 4.1x
        # SIMT on mlp_feat.7.bias at (700, 200, c2f), where the taped path with the same backward kernels is within 4x
        assert e["tc_recompute"] < max(2e-3, 6 * e["simt"]), (KEYS[i], "tc recompute", e["tc_recompute"], e["simt"])
        w1 = _maxnorm(res["tc_w1"][0][2][i], res["tc"][0][2][i])
        worst_w1_vs_tc = max(worst_w1_vs_tc, w1)
        assert w1 < 3e-2, (KEYS[i], "tc_w1 vs tc", w1)
        ctrl = _maxnorm(control[i], tr)
        if ctrl / gate < margin:
            margin, margin_at = ctrl / gate, KEYS[i]
    # a batch inside one partial tile is all tail: its control is the zero gradient (distance 1), so the margin is
    # 1 / gate, and at 99 rows the SIMT engine itself sits 0.1 from fp64 on mlp_feat.1.weight (measured margin 2.4)
    assert margin > (2.0 if R * S < TILE else 3.0), ("negative control too close to the gate", margin_at, margin)
    report.append("grad worst " + " ".join("%s %.1e" % kv for kv in worst.items()) +
                  " | w1 vs tc %.1e | control / gate >= %.1f (%s)" % (worst_w1_vs_tc, margin, margin_at))

    # the two stream topologies (with / without ray gradients) give the same parameter gradients
    worst_topo = 0.0
    for name in runs:
        for a, b in zip(res[name][0][2], res[name][1][2]):
            worst_topo = max(worst_topo, _maxnorm(b, a))
    assert worst_topo < 1e-5, ("parameter gradients depend on whether ray gradients were requested", worst_topo)
    report.append("with/without ray grads %.1e" % worst_topo)

    # ray gradients vs fp64
    e_ray = {}
    for name in runs:
        e_ray[name] = max(_rel_l2(res[name][0][3][0], truth[n_par]), _rel_l2(res[name][0][3][1], truth[n_par + 1]))
    for name in ("tc", "tc_recompute", "tc_w1"):
        assert e_ray[name] < max(1e-3, 4 * e_ray["simt"]), (name, "ray grads", e_ray[name], e_ray["simt"])
    report.append("ray grads " + " ".join("%s %.1e" % kv for kv in e_ray.items()))
    print("R=%d S=%d: %s" % (R, S, "; ".join(report)))


# ================================================================================================ B. accumulate (+=)
def _abi_mlp_backward(eng, tape, params, prog, c2f, o, d, t, noise, gs, gc, grads, d_o, d_d):
    """sparf_mlp_backward[_tape] straight through the C ABI into the given (possibly prefilled) buffers."""
    from sparf_b200 import _lib, ops
    L = _lib.lib()
    spec = ops.MLPSpec(barf_c2f=c2f)
    m, keep = spec.fill(params, prog)
    gstruct = spec.grad_struct(grads)
    R, S = t.shape
    P = ops._ptr
    nb = max(L.sparf_mlp_workspace_bytes(ctypes.byref(m), R, S, k, eng) for k in (0, 2 if tape else 1))
    ws = torch.empty(max(nb, 1), dtype=torch.uint8, device="cuda")
    if tape:
        tb = L.sparf_mlp_tape_bytes(ctypes.byref(m), eng, R, S)
        assert tb > 0
        tp = torch.empty(tb, dtype=torch.uint8, device="cuda")
        sigma, rgb = torch.empty(R, S, device="cuda"), torch.empty(R, S, 3, device="cuda")
        _lib.check(L.sparf_mlp_forward_tape(ctypes.byref(m), eng, R, S, P(o), P(d), P(t), P(noise), P(sigma), P(rgb), P(tp),
                                            tb, P(ws), ws.numel(), _stream()), "mlp_forward_tape")
        _lib.check(L.sparf_mlp_backward_tape(ctypes.byref(m), eng, R, S, P(o), P(d), P(t), P(sigma), P(rgb), P(gs), P(gc),
                                             ctypes.byref(gstruct), P(d_o), P(d_d), P(tp), tb, P(ws), ws.numel(), _stream()),
                   "mlp_backward_tape")
    else:
        _lib.check(L.sparf_mlp_backward(ctypes.byref(m), eng, R, S, P(o), P(d), P(t), P(noise), P(gs), P(gc),
                                        ctypes.byref(gstruct), P(d_o), P(d_d), P(ws), ws.numel(), _stream()), "mlp_backward")
    torch.cuda.synchronize()
    del keep


def _prefill_like(ref, g):
    """Seeded random values at the scale of `ref`: (x + p) - p then stays within a few ulps of max|ref|."""
    return torch.randn(ref.shape, device="cuda", generator=g) * ref.abs().max().clamp_min(1e-30)


def _assert_accumulated(out, prefill, zero_start, what):
    # the sums are fp32 atomics (not bitwise reproducible): 1e-5 of the tensor's largest entry
    e = _maxnorm(out - prefill, zero_start)
    assert e < 1e-5, (what, "not accumulated (+=)", e)
    return e


@pytest.mark.parametrize("R,S", [(77, 65), (2000, 65)])
@pytest.mark.parametrize("engine", ["simt_fp32", "tc_3x_tape", "tc_3x_recompute"])
def test_mlp_backward_accumulates(engine, R, S):
    """Every gradient output of sparf_mlp_backward / _backward_tape is accumulated (+=): the output minus a seeded random
    prefill equals the zero-start result, for each parameter gradient and d_origins / d_dirs, single-chunk (77x65) and
    multi-chunk (2000x65) batches.  Then the in-place autograd path (p._sparf_inplace_grad, sparf_b200.distributed)
    accumulates into the existing p.grad storage.  (Measured out - prefill vs zero start <= 3.7e-6 of the largest
    entry; a kernel that wrote instead of adding would be off by ~1.)"""
    from sparf_b200 import _lib, ops
    eng = _lib.ENGINE_SIMT_FP32 if engine == "simt_fp32" else _lib.ENGINE_TC_3X
    if eng == _lib.ENGINE_TC_3X and not _tc_available():
        pytest.skip("tcgen05 engine not available")
    tape = engine == "tc_3x_tape"
    params, o, d, t, noise, prog = _mlp_problem(R, S, None, seed=3 * R + S)
    gs, gc, _ = _upstream(R, S, seed=R + 1)
    zeros = lambda: ([torch.zeros_like(p) for p in params], torch.zeros_like(o), torch.zeros_like(d))
    g0, do0, dd0 = zeros()
    _abi_mlp_backward(eng, tape, params, prog, None, o, d, t, noise, gs, gc, g0, do0, dd0)
    gen = torch.Generator(device="cuda").manual_seed(R + S)
    pre = [_prefill_like(x, gen) for x in g0 + [do0, dd0]]
    out = [x.clone() for x in pre]
    _abi_mlp_backward(eng, tape, params, prog, None, o, d, t, noise, gs, gc, out[:-2], out[-2], out[-1])
    names = KEYS + ["d_origins", "d_dirs"]
    worst = 0.0
    for x, p, z, nm in zip(out, pre, g0 + [do0, dd0], names):
        worst = max(worst, _assert_accumulated(x, p, z, nm))

    # autograd with p._sparf_inplace_grad: the backward adds into p.grad where it is
    spec = ops.MLPSpec()
    ops.USE_TAPE[0] = tape
    try:
        ps = [p.clone().requires_grad_(True) for p in params]
        for p, q in zip(ps, pre):
            p.grad = q.clone()
            p._sparf_inplace_grad = True
        ptrs = [p.grad.data_ptr() for p in ps]
        s, c = ops.mlp_forward(spec, o, d, t, ps, noise=noise, progress=prog, engine=eng)
        ((s * gs).sum() + (c * gc).sum()).backward()
        torch.cuda.synchronize()
    finally:
        ops.USE_TAPE[0] = True
    assert [p.grad.data_ptr() for p in ps] == ptrs, "the in-place path did not run"
    for p, q, z, nm in zip(ps, pre, g0, KEYS):
        worst = max(worst, _assert_accumulated(p.grad, q, z, nm + " (autograd in place)"))
    print("%s R=%d S=%d: out - prefill vs zero start %.1e" % (engine, R, S, worst))


# ================================================================================================ C. compositing
def _composite_inputs(R, S, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    sigma = torch.rand(R, S, device="cuda", generator=g) * 3
    rgb = torch.rand(R, S, 3, device="cuda", generator=g)
    t = torch.sort(torch.rand(R, S, device="cuda", generator=g) * 4 + 1, dim=1).values
    dirs = torch.randn(R, 3, device="cuda", generator=g)
    if R >= 2:
        sigma[0] = 0.0          # a ray through empty space
        sigma[-1, 0] = 1e6      # a ray that is opaque at its first sample
    up = (torch.randn(R, 3, device="cuda", generator=g), torch.randn(R, device="cuda", generator=g),
          torch.randn(R, device="cuda", generator=g), torch.randn(R, S, device="cuda", generator=g) * 0.1)
    return sigma, rgb, t, dirs, up


def _composite_oracle(sigma, rgb, t, dirs, white_bg, need_dirs, up, use_w, dtype):
    from oracle import sparf_oracle as O
    s = sigma.detach().to(dtype).clone().requires_grad_(True)
    c = rgb.detach().to(dtype).clone().requires_grad_(True)
    dr = dirs.detach().to(dtype).clone().requires_grad_(need_dirs)
    out = O.composite(dr[None], s[None], c[None], t.to(dtype)[None], white_bg=white_bg)
    vals = [out["rgb"][0], out["depth"][0, :, 0], out["opacity"][0, :, 0], out["weights"][0, :, :, 0],
            out["depth_var"][0, :, 0], out["rgb_var"][0, :, 0], out["all_cumulated"][0]]
    loss = (vals[0] * up[0].to(dtype)).sum() + (vals[1] * up[1].to(dtype)).sum() + (vals[2] * up[2].to(dtype)).sum()
    if use_w:
        loss = loss + (vals[3] * up[3].to(dtype)).sum()
    loss.backward()
    grads = [s.grad, c.grad] + ([dr.grad] if need_dirs else [])
    return [v.detach() for v in vals], grads


@pytest.mark.parametrize("R", [1, 5, 4099])
@pytest.mark.parametrize("S", [2, 3, 31, 33, 1537, 2048, 4096])
def test_composite_vs_fp64(S, R):
    """ops.composite forward (all seven outputs) and backward (d_sigma, d_rgb, d_dirs) vs fp64 autograd through
    O.composite, with white_bg on / off, with / without g_weights and with / without a dirs gradient.  S = 2, S not a
    multiple of 32, S > 1536 (the backward's opt-in shared-memory branch), R not a multiple of 4 (idle warps in the
    last block); a ray with zero density everywhere and a ray opaque at its first sample.
    Gate: within max(2e-5, 4x the fp32 oracle's own distance from fp64) per tensor (measured worst 1.3e-7 .. 1.3e-6
    for S <= 33, up to 5.7e-5 at S = 4096, R = 4099, where the fp32 oracle is as far)."""
    from sparf_b200 import ops
    sigma, rgb, t, dirs, up = _composite_inputs(R, S, seed=S * 10 + R)
    names = ("rgb", "depth", "opacity", "weights", "depth_var", "rgb_var", "all_cumulated", "d_sigma", "d_rgb", "d_dirs")
    worst = 0.0
    for white_bg in (False, True):
        for use_w in (False, True):
            for need_dirs in (False, True):
                s = sigma.clone().requires_grad_(True)
                c = rgb.clone().requires_grad_(True)
                dr = dirs.clone().requires_grad_(need_dirs)
                out = ops.composite(s, c, t, dr, white_bg)
                loss = (out[0] * up[0]).sum() + (out[1] * up[1]).sum() + (out[2] * up[2]).sum()
                if use_w:
                    loss = loss + (out[3] * up[3]).sum()
                loss.backward()
                torch.cuda.synchronize()
                ours = [x.detach() for x in out] + [s.grad, c.grad] + ([dr.grad] if need_dirs else [])
                v64, g64 = _composite_oracle(sigma, rgb, t, dirs, white_bg, need_dirs, up, use_w, torch.float64)
                v32, g32 = _composite_oracle(sigma, rgb, t, dirs, white_bg, need_dirs, up, use_w, torch.float32)
                for nm, a, b32, b64 in zip(names, ours, v32 + g32, v64 + g64):
                    # rgb_var is a signed sum that can vanish (one ray): measured on the scale of the colours, 1
                    fl = 1.0 if nm == "rgb_var" else 1e-30
                    e, e32 = _maxnorm(a, b64, fl), _maxnorm(b32, b64, fl)
                    assert e < max(2e-5, 4 * e32), (nm, white_bg, use_w, need_dirs, e, e32)
                    worst = max(worst, e)
    print("composite R=%d S=%d: worst vs fp64 %.1e" % (R, S, worst))


def test_composite_backward_abi_writes_and_accumulates():
    """sparf_composite_backward writes d_sigma / d_rgb (a prefill is overwritten) and accumulates d_dirs (+=), at S = 33
    and at S = 2048 (opt-in shared memory); S = 4097 is rejected with SPARF_ERR_INVALID."""
    from sparf_b200 import _lib, ops
    L = _lib.lib()
    P = ops._ptr
    for R, S in ((5, 33), (7, 2048)):
        sigma, rgb, t, dirs, up = _composite_inputs(R, S, seed=S)
        gen = torch.Generator(device="cuda").manual_seed(S + 1)

        def call(ds, dc, dd):
            _lib.check(L.sparf_composite_backward(R, S, P(sigma), P(rgb), P(t), P(dirs), 1, P(up[0]), P(up[1]), P(up[2]),
                                                  P(up[3]), P(ds), P(dc), P(dd), _stream()), "composite_backward")
            torch.cuda.synchronize()
        z = (torch.zeros(R, S, device="cuda"), torch.zeros(R, S, 3, device="cuda"), torch.zeros(R, 3, device="cuda"))
        call(*z)
        pre = [_prefill_like(x, gen) for x in z]
        out = [x.clone() for x in pre]
        call(*out)
        assert torch.equal(out[0], z[0]) and torch.equal(out[1], z[1]), "d_sigma / d_rgb must be written, not added"
        _assert_accumulated(out[2], pre[2], z[2], "composite d_dirs")
    R, S = 1, 4097
    buf = torch.zeros(R * S * 3 + 16, device="cuda")
    rc = L.sparf_composite_backward(R, S, P(buf), P(buf), P(buf), P(buf), 0, P(buf), P(buf), P(buf), None, P(buf), P(buf),
                                    None, _stream())
    assert rc == 1, rc   # SPARF_ERR_INVALID


def test_composite_properties_s4096():
    """The size-independent properties of test_cuda_parity.py::test_composite_properties_full_size at the largest S the
    backward accepts (4096 samples, 1027 rays): weights >= 0, opacity = sum(weights) <= 1, depth within the samples,
    all_cumulated = 1 - the sum of all weights but the last two, rgb in [0, 1]."""
    from sparf_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(2)
    R, S = 1027, 4096
    sigma = torch.rand(R, S, device="cuda", generator=g) * 3
    rgb = torch.rand(R, S, 3, device="cuda", generator=g)
    t = torch.sort(torch.rand(R, S, device="cuda", generator=g) * 4 + 1, dim=1).values
    dirs = torch.randn(R, 3, device="cuda", generator=g)
    rgb_map, depth, opacity, weights, depth_var, rgb_var, all_cum = ops.composite(sigma, rgb, t, dirs)
    assert (weights >= 0).all()
    assert torch.allclose(opacity, weights.sum(1), atol=1e-5)
    assert (opacity <= 1 + 1e-5).all()
    assert ((depth >= t[:, 0] * opacity - 1e-4) & (depth <= t[:, -1] + 1e-4)).all()
    # all_cumulated = T_{S-2} vs 1 - sum of 4094 weights: each w = T (1 - e^-sd) with sd ~ 3e-3 carries the fp32
    # cancellation of 1 - e^-sd, which the reference's formula shares, so the identity is held to the fp32 oracle's own
    # residual (4x, floor 2e-5) rather than to the 2e-5 of the 384-sample test
    from oracle import sparf_oracle as O
    ref = O.composite(dirs[None], sigma[None], rgb[None], t[None])
    res32 = (ref["all_cumulated"][0] - (1 - ref["weights"][0, :, :-2, 0].sum(1))).abs().max().item()
    res = (all_cum - (1 - weights[:, :-2].sum(1))).abs().max().item()
    assert res < max(2e-5, 4 * res32), (res, res32)
    assert (rgb_map >= -1e-6).all() and (rgb_map <= 1 + 1e-5).all()
    print("composite S=4096: all_cumulated identity residual %.1e (fp32 oracle %.1e)" % (res, res32))


# ================================================================================================ C. ray generation
H_IMG, W_IMG = 60, 100


def _camera(B, seed):
    from oracle import sparf_oracle as O
    g = torch.Generator(device="cpu").manual_seed(seed)
    d9 = torch.randn(B, 9, generator=g, dtype=torch.float64)
    pose = O.d9_to_pose(d9).float().cuda()
    intr = torch.tensor([[120.0, 0.0, 50.0], [0.0, 110.0, 30.0], [0.0, 0.0, 1.0]]).repeat(B, 1, 1)
    intr[:, 0, 0] += torch.rand(B, generator=g) * 10
    return pose, intr.cuda()


@pytest.mark.parametrize("n", [1, 255, 256, 257, 5000])
@pytest.mark.parametrize("B", [1, 3])
def test_raygen_backward_vs_fp64(B, n):
    """ops.raygen backward (d_pose, and d_pixels on the float-pixel path) vs fp64 autograd through
    O.rays_from_ray_idx / O.rays_at_pixels, for shared and per-image ray_idx and shared and per-image pixels (a shared
    pixel list sums the images' gradients with atomics).  n = 255 / 256 / 257 straddle the 256-thread block.
    Gate: within max(1e-5, 4x the fp32 oracle's own distance from fp64) per tensor (measured worst 2.8e-7)."""
    from oracle import sparf_oracle as O
    from sparf_b200 import ops
    pose, intr = _camera(B, seed=B * 1000 + n)
    g = torch.Generator(device="cuda").manual_seed(n)
    go = torch.randn(B, n, 3, device="cuda", generator=g)
    gd = torch.randn(B, n, 3, device="cuda", generator=g)
    modes = {
        "idx_shared": torch.randint(0, H_IMG * W_IMG, (n,), device="cuda", generator=g),
        "idx_per_image": torch.randint(0, H_IMG * W_IMG, (B, n), device="cuda", generator=g),
        "px_shared": torch.rand(n, 2, device="cuda", generator=g) * torch.tensor([W_IMG, H_IMG], device="cuda"),
        "px_per_image": torch.rand(B, n, 2, device="cuda", generator=g) * torch.tensor([W_IMG, H_IMG], device="cuda"),
    }
    worst = 0.0
    for mode, src in modes.items():
        is_px = mode.startswith("px")
        p = pose.clone().requires_grad_(True)
        px = src.clone().requires_grad_(True) if is_px else None
        o, d = ops.raygen(p, intr, W_IMG, **({"pixels": px} if is_px else {"ray_idx": src}))
        ((o * go).sum() + (d * gd).sum()).backward()
        torch.cuda.synchronize()
        ours = [p.grad] + ([px.grad] if is_px else [])
        ref = {}
        for dt in (torch.float64, torch.float32):
            p_r = pose.to(dt).clone().requires_grad_(True)
            px_r = src.to(dt).clone().requires_grad_(True) if is_px else None
            if is_px:
                o_r, d_r = O.rays_at_pixels(p_r, intr.to(dt), px_r)
            else:
                o_r, d_r = O.rays_from_ray_idx(p_r, intr.to(dt), H_IMG, W_IMG, src)
            ((o_r * go.to(dt)).sum() + (d_r * gd.to(dt)).sum()).backward()
            ref[dt] = [p_r.grad] + ([px_r.grad] if is_px else [])
        for nm, a, b32, b64 in zip(("d_pose", "d_pixels"), ours, ref[torch.float32], ref[torch.float64]):
            e, e32 = _maxnorm(a, b64), _maxnorm(b32, b64)
            assert e < max(1e-5, 4 * e32), (mode, nm, e, e32)
            worst = max(worst, e)
    print("raygen B=%d n=%d: worst vs fp64 %.1e" % (B, n, worst))


def test_raygen_backward_abi_accumulates():
    """sparf_raygen_backward accumulates d_pose (+=) and, for a shared pixel list, d_pixels (+=); per-image d_pixels
    are written (a prefill is overwritten)."""
    from sparf_b200 import _lib, ops
    L = _lib.lib()
    P = ops._ptr
    B, n = 3, 1000
    pose, intr = _camera(B, seed=5)
    kinv = torch.linalg.inv(intr)
    g = torch.Generator(device="cuda").manual_seed(6)
    go = torch.randn(B, n, 3, device="cuda", generator=g)
    gd = torch.randn(B, n, 3, device="cuda", generator=g)
    for per_image in (0, 1):
        px = torch.rand(*((B, n, 2) if per_image else (n, 2)), device="cuda", generator=g) * 50

        def call(dp, dpx):
            _lib.check(L.sparf_raygen_backward(B, n, W_IMG, P(pose), P(kinv), None, P(px), per_image, P(go), P(gd), P(dp),
                                               P(dpx), _stream()), "raygen_backward")
            torch.cuda.synchronize()
        z = (torch.zeros_like(pose), torch.zeros_like(px))
        call(*z)
        pre = [_prefill_like(x, g) for x in z]
        out = [x.clone() for x in pre]
        call(*out)
        _assert_accumulated(out[0], pre[0], z[0], "d_pose")
        if per_image:
            assert torch.equal(out[1], z[1]), "per-image d_pixels must be written, not added"
        else:
            _assert_accumulated(out[1], pre[1], z[1], "shared d_pixels")


# ================================================================================================ C. resampling
@pytest.mark.parametrize("S,Sf", [(1, 1), (2, 63), (63, 129), (128, 128), (1000, 3000), (2048, 2048)])
def test_sample_pdf_merge_edges(S, Sf):
    """ops.sample_pdf_merge vs O.sample_pdf (fp32) with rays whose weights are all zero, one non-zero bin, mass only in
    the first or only in the last bin, and random.  t_fine within the existing 5e-6 (test_cuda_parity.py); t_all
    bit-identical to torch.sort(cat([t_coarse, t_fine])): an exact check of the bitonic merge including its +inf
    padding up to the next power of two (S + S_fine = 4096 at the largest case).  Measured t_fine error <= 1.5e-6."""
    from oracle import sparf_oracle as O
    from sparf_b200 import ops
    near, far = 1.2, 5.2
    R = 9
    g = torch.Generator(device="cuda").manual_seed(S + Sf)
    w = torch.rand(R, S, device="cuda", generator=g) + 0.05
    w[0] = 0.0
    w[1] = 0.0
    w[1, S // 2] = 0.7
    w[2] = 0.0
    w[2, 0] = 0.3
    w[3] = 0.0
    w[3, -1] = 2.0
    t_c = torch.sort(torch.rand(R, S, device="cuda", generator=g) * (far - near) + near, dim=1).values
    grid = torch.linspace(0, 1, Sf + 1, device="cuda")
    u_mid = 0.5 * (grid[:-1] + grid[1:])
    t_fine, t_all = ops.sample_pdf_merge(w, t_c, u_mid, near, far)
    torch.cuda.synchronize()
    ref = O.sample_pdf(w[None], S, Sf, (near, far))[0]
    e = _maxnorm(t_fine, ref)
    assert e < 5e-6, e
    assert torch.equal(t_all, torch.sort(torch.cat([t_c, t_fine], dim=1), dim=1).values)
    print("sample_pdf S=%d Sf=%d: t_fine vs fp32 oracle %.1e" % (S, Sf, e))


# ================================================================================================ C. Huber
@pytest.mark.parametrize("n", [1, 257, 262145, 3_000_001])
def test_huber2_vs_fp64(n):
    """ops.huber2 (2 x mean Huber, delta 0.5) vs an fp64 evaluation, with residuals exactly at |z| = 0.5 and one ulp on
    either side of it; n = 262145 is the first size whose grid-stride loop (1024 blocks x 256 threads) iterates twice.
    Loss within 1e-5 relative (fp32 partial sums; measured <= 6.9e-8), d_pred within 1e-6 of its largest entry
    (measured <= 8.3e-8)."""
    from sparf_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(n)
    target = torch.randn(n, device="cuda", generator=g) * 0.4
    pred = target + torch.randn(n, device="cuda", generator=g) * 0.5
    edge = torch.tensor([0.5, -0.5, np.nextafter(np.float32(0.5), np.float32(0)), np.nextafter(np.float32(0.5), np.float32(1)),
                         -np.nextafter(np.float32(0.5), np.float32(0)), -np.nextafter(np.float32(0.5), np.float32(1))],
                        device="cuda", dtype=torch.float32)
    k = min(n, edge.numel())
    idx = torch.randperm(n, device="cuda", generator=g)[:k]
    target[idx] = 0.0
    pred[idx] = edge[:k]
    p = pred.clone().requires_grad_(True)
    loss = ops.huber2(p, target)
    loss.backward()
    torch.cuda.synchronize()
    z = pred.double() - target.double()
    az = z.abs()
    ref = 2 * torch.where(az < 0.5, 0.5 * z * z, 0.5 * (az - 0.25)).mean()
    ref_d = 2.0 / n * torch.where(az < 0.5, z, 0.5 * torch.sign(z))
    el = abs(loss.item() - ref.item()) / abs(ref.item())
    ed = _maxnorm(p.grad, ref_d)
    assert el < 1e-5, el
    assert ed < 1e-6, ed
    print("huber2 n=%d: loss rel %.1e, d_pred %.1e" % (n, el, ed))
