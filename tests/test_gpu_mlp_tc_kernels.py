"""The bf16 tcgen05 MLP kernels of csrc/mlp_tc.cu one entry point at a time, each against an fp64 reference of the same
operation: dX (ep_tc_linear_dx_bf16), dW / db (ep_tc_linear_dw_bf16, both orientations), the output layer
(ep_tc_linear_final_bf16), the hidden forward (ep_tc_linear_fwd_bf16) and the packing kernels.

Every kernel input is taken from the bytes the kernel reads: packed tiles through mlp_tc.unpack_rows, weights rounded to
bf16.  Those values are exact in fp64, so the only error left is the fp32 accumulation of the tensor cores, plus one final
rounding of the output.  With u = 2^-24, uB = 2^-8, gamma_m = m u / (1 - m u) and E = gamma_K (|A| |B|) (elementwise,
fp64), each comparison is either exact (one-hot probes, packing, masks, padding, determinism) or the a-priori bound

    |got - ref| <= u_out (|ref| + E) + E                                                  (assert_bound)

  dX, hidden forward   u_out = uB (bf16 output)    K = out_padded; in_padded + 1 with the bias as one more term
  dW, db               u_out = 0                   K = n + grid + 4 (per-CTA sums, then a fixed-order reduction)
  output layer         u_out = u (fp32 output)     K = in_padded, E + gamma_1 |b|

An entry whose reference and E are both 0 (masked, padded, or a row >= n of the last tile) must therefore be exactly 0.
The rounding of the fp64 reference itself (about 2^-29 of E) is not counted.  Output buffers are 0xFF- or NaN-filled
and followed by a guard region, so a value the kernel fails to write, or writes past the end, shows."""
import math
from ctypes import c_void_p as P

import numpy as np
import pytest
import torch

from gpu_util import pkg, dev

pytestmark = pytest.mark.gpu

U32, UB = 2.0 ** -24, 2.0 ** -8
GUARD = 4096                        # bytes checked after every output region
MANY = "many_tiles"                 # n with more 128-row tiles than 2 * sm_count, resolved on the device
N_SET = [1, 127, 128, 129, 40001, MANY]
TRUE_WIDTH = {32: 26, 64: 50, 96: 82, 128: 100, 160: 146, 256: 256}     # padded width -> unpadded width used with it


# ------------------------------------------------------------------------------------------------ bound
def gamma(m):
    return m * U32 / (1.0 - m * U32)


def assert_bound(got, ref, E, u_out, what):
    """|got - ref| <= u_out (|ref| + E) + E elementwise in fp64; NaN fails."""
    got = got.double()
    bound = u_out * (ref.abs() + E) + E
    bad = ~((got - ref).abs() <= bound)
    if bad.any():
        i = tuple(int(v) for v in bad.nonzero()[0])
        raise AssertionError("%s: %d of %d entries out of bound, first at %s: got %r ref %r bound %r" % (
            what, int(bad.sum()), bad.numel(), i, got[i].item(), ref[i].item(), bound[i].item()))


# ------------------------------------------------------------------------------------------------ library access
def _call(name, *a):
    pkg("_cabi").call(name, *a)


def _q(name, *a):
    return pkg("_cabi").query(name, *a)


def _p(t):
    return P(t.data_ptr()) if t is not None else None


def _st():
    return P(torch.cuda.current_stream().cuda_stream)


def _sm():
    return torch.cuda.get_device_properties(dev()).multi_processor_count


def _n(n):
    return 128 * 3 * _sm() + 77 if n == MANY else n


def _tiles(n):
    return (n + 127) // 128


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def guarded_u8(nbytes):
    """(region, whole buffer): nbytes of 0xFF followed by GUARD more."""
    buf = torch.full((nbytes + GUARD,), 0xFF, dtype=torch.uint8, device=dev())
    return buf[:nbytes], buf


def guarded_f32(count):
    buf = torch.full((count + GUARD // 4,), float("nan"), device=dev())
    return buf[:count], buf


def assert_guard(buf, used):
    tail = buf[used:]
    ok = torch.isnan(tail).all() if tail.dtype == torch.float32 else (tail == 0xFF).all()
    assert ok, "written past the end of the output"


# ------------------------------------------------------------------------------------------------ packed operands
def pack_ref(X, dp):
    """fp32 (n, d) -> bytes of the packed tiles [tile][dp/8][128][8] bf16 (torch rounding: nearest even), zero padded."""
    n, d = X.shape
    Z = torch.zeros(_tiles(n) * 128, dp, dtype=torch.bfloat16, device=X.device)
    Z[:n, :d] = X.to(torch.bfloat16)
    return Z.view(-1, 128, dp // 8, 8).permute(0, 2, 1, 3).contiguous().view(-1).view(torch.uint8)


def unpack_all(packed, n, dp):
    """What the kernel reads / wrote: every row of every tile (rows >= n of the last tile included), fp64."""
    return pkg("mlp_tc").unpack_rows(packed, _tiles(n) * 128, dp).double()


def rand_packed(n, d, dp, g):
    """Random operand, mixed signs, zero padded: (packed bytes, its values (tiles * 128, dp) fp64)."""
    packed = pack_ref(torch.randn(n, d, device=dev(), generator=g), dp)
    return packed, unpack_all(packed, n, dp)


def one_hot_packed(n, dp, r, f):
    """Packed tiles of the (n, dp) matrix e(r, f): bf16 1.0 at row r, feature f."""
    t = torch.zeros(_q("ep_tc_packed_rows_bytes", n, dp) // 2, dtype=torch.int16, device=dev())
    t[((r // 128 * (dp // 8) + f // 8) * 128 + r % 128) * 8 + f % 8] = 0x3F80
    return t.view(torch.uint8)


def weight_layouts(Wb, pair=True):
    """Bytes of the layouts ep_tc_pack_weight_bf16 writes for the padded bf16 matrix Wb [outp x inp] (header;
    pack_weight_kernel): Wp = [inp/8][outp][8] then its CTA-pair copy [inp/32][2][4][outp/2][8] (K = in, N = out);
    WTp = [outp/8][inp][8] then [outp/32][2][4][inp/2][8] (K = out, N = in)."""
    op, ip = Wb.shape
    wp = [Wb.view(op, ip // 8, 8).permute(1, 0, 2)]
    wt = [Wb.view(op // 8, 8, ip).permute(0, 2, 1)]
    if pair:
        wp.append(Wb.view(2, op // 2, ip // 32, 4, 8).permute(2, 0, 3, 1, 4))
        wt.append(Wb.view(op // 32, 4, 8, 2, ip // 2).permute(0, 3, 1, 4, 2))
    flat = lambda ts: torch.cat([t.reshape(-1) for t in ts]).view(torch.uint8)
    return flat(wp), flat(wt)


def rand_weights(out, inn, op, ip, g):
    """Random nn.Linear weight [out x in]: (Wp bytes, WTp bytes, padded bf16 values (op, ip) fp64)."""
    W = torch.randn(out, inn, device=dev(), generator=g) / math.sqrt(inn)
    Wb = torch.zeros(op, ip, dtype=torch.bfloat16, device=dev())
    Wb[:out, :inn] = W.to(torch.bfloat16)
    Wp, WTp = weight_layouts(Wb)
    return Wp, WTp, Wb.double()


def rand_mask(n, dp, g):
    """Random ReLU bit masks, one int32 word per (row, 32 features), for every row of every tile."""
    return torch.randint(-2 ** 31, 2 ** 31, (_tiles(n) * 128, dp // 32), dtype=torch.int32, device=dev(), generator=g)


def mask_bits(words, dp):
    """Mask words -> bool (rows, dp) in the header's order: bit i of word w = feature 32w + 2i, bit 16 + i = 32w + 2i + 1."""
    pos = torch.arange(32, device=words.device)
    pos = (pos % 2) * 16 + pos // 2
    return ((words.view(-1, dp // 32).unsqueeze(-1) >> pos) & 1).reshape(-1, dp).bool()


# ------------------------------------------------------------------------------------------------ kernel calls
def run_dx(n, op, ip, dZp, WTp, words, max_ctas=0):
    """ep_tc_linear_dx_bf16 into a 0xFF-filled buffer; returns the packed output bytes."""
    nbytes = _q("ep_tc_packed_rows_bytes", n, ip)
    out, buf = guarded_u8(nbytes)
    _call("ep_tc_linear_dx_bf16", n, op, ip, _p(dZp), _p(WTp), _p(words), _p(out), max_ctas, _st())
    torch.cuda.synchronize()
    assert_guard(buf, nbytes)
    return out


def dw_grid(n, max_ctas):
    grid = min(_sm(), max_ctas) if max_ctas > 0 else _sm()
    return min(grid, _tiles(n))


def run_dw(n, out, inn, op, ip, dZp, actp, max_ctas=0):
    """ep_tc_linear_dw_bf16 into NaN-filled dW / db and a 0xFF-filled workspace (a partial the kernel did not write
    reads as NaN); returns (dW [out x in], db [out])."""
    dW, dW_buf = guarded_f32(out * inn)
    db, db_buf = guarded_f32(out)
    ws = torch.full((_q("ep_tc_dw_workspace_bytes"),), 0xFF, dtype=torch.uint8, device=dev())
    _call("ep_tc_linear_dw_bf16", n, out, inn, op, ip, _p(dZp), _p(actp), _p(dW), _p(db), _p(ws), ws.numel(), max_ctas,
          _st())
    torch.cuda.synchronize()
    assert_guard(dW_buf, out * inn)
    assert_guard(db_buf, out)
    return dW.view(out, inn), db


# ------------------------------------------------------------------------------------------------ random cases
# Each returns [(what, got, ref, E, u_out)] for assert_bound, plus what the exact checks need.
def dx_case(n, op, ip, seed, max_ctas=0):
    g = _gen(seed)
    out, inn = TRUE_WIDTH[op], TRUE_WIDTH[ip]
    dZp, dZ = rand_packed(n, out, op, g)
    _, WTp, W = rand_weights(out, inn, op, ip, g)
    words = rand_mask(n, ip, g)
    m = mask_bits(words, ip).double()
    raw = run_dx(n, op, ip, dZp, WTp, words, max_ctas)
    got = unpack_all(raw, n, ip)
    ref = (dZ @ W) * m
    E = gamma(op) * (dZ.abs() @ W.abs()) * m
    return [("dX", got, ref, E, UB)], dict(raw=raw, got=got, m=m, inn=inn)


def dw_case(n, out, op, inn, ip, seed, max_ctas=0):
    g = _gen(seed)
    dZp, dZ = rand_packed(n, out, op, g)
    actp, act = rand_packed(n, inn, ip, g)
    dW, db = run_dw(n, out, inn, op, ip, dZp, actp, max_ctas)
    Z, A = dZ[:, :out], act[:, :inn]
    K = n + dw_grid(n, max_ctas) + 4
    return [("dW", dW, Z.t() @ A, gamma(K) * (Z.abs().t() @ A.abs()), 0.0),
            ("db", db, Z.sum(0), gamma(K) * Z.abs().sum(0), 0.0)], dict(dW=dW, db=db)


def final_case(n, out, seed, variant="plain"):
    g = _gen(seed)
    inn, ip = 250, 256
    op = _q("ep_tc_pad_features", out, 0)
    actp, act = rand_packed(n, inn, ip, g)
    Wp, _, W = rand_weights(out, inn, op, ip, g)
    b = torch.randn(out, device=dev(), generator=g)
    ldc, ldu = (out + 5, out + 3) if variant == "strided" else (out, out)
    corr, corr_buf = guarded_f32(n * ldc)
    U_base = U_pred = up_buf = scale_dev = None
    scale = 0.75
    if variant != "U_base_null":
        U_base = torch.randn(n * ldu, device=dev(), generator=g)
        U_pred, up_buf = guarded_f32(n * ldu)
    if variant == "scale_dev":
        scale_dev = torch.tensor([-0.375], device=dev())
    _call("ep_tc_linear_final_bf16", n, ip, out, op, _p(actp), _p(Wp), _p(b), _p(corr), ldc, _p(U_base),
          scale if scale_dev is None else 3.0, _p(scale_dev), _p(U_pred), ldu, _st())
    torch.cuda.synchronize()
    c = corr.view(n, ldc)
    A, Wo, bd = act[:n], W[:out], b.double()
    E = gamma(ip) * (A.abs() @ Wo.abs().t()) + gamma(1) * bd.abs()
    extra = dict(c=c, corr_buf=corr_buf, ldc=ldc, ldu=ldu, U_base=U_base, U_pred=U_pred, up_buf=up_buf,
                 scale=-0.375 if scale_dev is not None else scale)
    return [("corr", c[:, :out], A @ Wo.t() + bd, E, U32)], extra


def hidden_case(n, inn, ip, out, op, seed):
    g = _gen(seed)
    actp, act = rand_packed(n, inn, ip, g)
    Wp, _, W = rand_weights(out, inn, op, ip, g)
    b = torch.randn(out, device=dev(), generator=g)
    bpad = torch.zeros(op, dtype=torch.float64, device=dev())
    bpad[:out] = b.double()
    nbytes, mbytes = _q("ep_tc_packed_rows_bytes", n, op), _q("ep_tc_relu_mask_bytes", n, op)
    outp, out_buf = guarded_u8(nbytes)
    mask, mask_buf = guarded_u8(mbytes)
    _call("ep_tc_linear_fwd_bf16", n, ip, out, op, _p(actp), _p(Wp), _p(b), 1, _p(outp), _p(mask), _st())
    torch.cuda.synchronize()
    assert_guard(out_buf, nbytes)
    assert_guard(mask_buf, mbytes)
    got = unpack_all(outp, n, op)[:n]
    A = act[:n]
    ref = torch.relu(A @ W.t() + bpad)
    E = gamma(ip + 1) * (A.abs() @ W.abs().t() + bpad.abs())
    return [("hidden", got, ref, E, UB)], dict(got=got, bits=mask_bits(mask.view(torch.int32), op)[:n])


# ------------------------------------------------------------------------------------------------ dX
@pytest.mark.parametrize("ip", [128, 256], ids=lambda v: "in%d" % v)
@pytest.mark.parametrize("op", [32, 64, 96, 128, 256], ids=lambda v: "K%d" % v)
@pytest.mark.parametrize("n", N_SET, ids=str)
def test_dx_random(n, op, ip):
    """dZ_prev = (dZ W) * mask with a random mask (not from a forward pass, so a bit-order error shows).  The bound also
    demands exact zeros where the mask bit is 0, in padded features and in rows >= n of the last tile."""
    n = _n(n)
    checks, x = dx_case(n, op, ip, seed=n * 31 + op + ip)
    for c in checks:
        assert_bound(*c[1:], what=c[0])
    got = x["got"]
    assert (got[x["m"] == 0] == 0).all()
    assert (got[:, x["inn"]:] == 0).all()
    assert (got[n:] == 0).all()


DX_PROBES = [(256, 256, 256, 256), (82, 96, 100, 128), (10, 32, 256, 256)]        # (out, out_padded, in, in_padded)


def _probe_rows(n):
    return sorted({r for r in (0, 127, 128, n - 1) if 0 <= r < n})


def _probe_cols(k):
    return sorted({o for o in (0, 127, 128, k - 1) if o < k})


@pytest.mark.parametrize("shape", DX_PROBES, ids=lambda s: "K%d-in%d" % (s[1], s[3]))
@pytest.mark.parametrize("n", [129, 40001], ids=str)
def test_dx_one_hot_probes(n, shape):
    """dZ = e(r, o): row r of dX must be W[o, :] * mask[r] exactly and every other row exactly 0 (tile, chunk and
    M-half indexing)."""
    out, op, inn, ip = shape
    g = _gen(n + op)
    _, WTp, W = rand_weights(out, inn, op, ip, g)
    words = rand_mask(n, ip, g)
    m = mask_bits(words, ip).double()
    for r in _probe_rows(n):
        for o in _probe_cols(out):
            got = unpack_all(run_dx(n, op, ip, one_hot_packed(n, op, r, o), WTp, words), n, ip)
            want = torch.zeros_like(got)
            want[r] = W[o] * m[r]
            assert torch.equal(got, want), (r, o)


# ------------------------------------------------------------------------------------------------ dW / db
# (out, out_padded, in, in_padded).  Orientation (a): out_padded 128 / 256, db summed from the X operand (dZ).
# Orientation (b): out_padded 32..96 (the output layer), operands swapped, db from the Y operand, reduced transposed.
DW_SHAPES = [(TRUE_WIDTH[op], op, TRUE_WIDTH[ip], ip) for op in (128, 256) for ip in (32, 96, 160, 256)] + \
            [(k, 32, TRUE_WIDTH[ip], ip) for k in (10, 16, 32) for ip in (128, 256)] + \
            [(TRUE_WIDTH[op], op, TRUE_WIDTH[ip], ip) for op in (64, 96) for ip in (128, 256)]


def _dw_id(s):
    out, op, inn, ip = s
    return ("a_dbX-o%d" % op if op % 128 == 0 else "b_dbY-o%dk%d" % (op, out)) + "-i%d" % ip


@pytest.mark.parametrize("shape", DW_SHAPES, ids=_dw_id)
@pytest.mark.parametrize("n", N_SET, ids=str)
def test_dw_random(n, shape):
    out, op, inn, ip = shape
    n = _n(n)
    checks, _ = dw_case(n, out, op, inn, ip, seed=n * 17 + op * 3 + ip + out)
    for c in checks:
        assert_bound(*c[1:], what=c[0])


DW_PROBES = [(256, 256, 146, 160), (100, 128, 82, 96), (10, 32, 256, 256), (82, 96, 100, 128)]


@pytest.mark.parametrize("shape", DW_PROBES, ids=_dw_id)
@pytest.mark.parametrize("n", [129, 40001], ids=str)
def test_dw_one_hot_probes(n, shape):
    """dZ = e(r, o): dW must be act[r] in row o and 0 elsewhere, db must be e_o, exactly."""
    out, op, inn, ip = shape
    actp, act = rand_packed(n, inn, ip, _gen(n + ip))
    for r in _probe_rows(n):
        for o in _probe_cols(out):
            dW, db = run_dw(n, out, inn, op, ip, one_hot_packed(n, op, r, o), actp)
            want = torch.zeros(out, inn, dtype=torch.float64, device=dev())
            want[o] = act[r, :inn]
            assert torch.equal(dW.double(), want), (r, o)
            e = torch.zeros(out, dtype=torch.float64, device=dev())
            e[o] = 1.0
            assert torch.equal(db.double(), e), (r, o)


# ------------------------------------------------------------------------------------------------ grid size
MAX_CTAS = [0, 1, 2, 65, "sm-1", "gt_tiles"]


def _max_ctas(v, n):
    return _sm() - 1 if v == "sm-1" else _tiles(n) + 7 if v == "gt_tiles" else v


@pytest.mark.parametrize("max_ctas", MAX_CTAS, ids=lambda v: "ctas_%s" % v)
def test_dx_independent_of_grid(max_ctas):
    """Each output tile is computed by one CTA whatever the grid: dX is bit-identical to the default grid's."""
    n = 40001
    mc = _max_ctas(max_ctas, n)
    checks, x = dx_case(n, 256, 256, seed=5, max_ctas=mc)
    for c in checks:
        assert_bound(*c[1:], what=c[0])
    _, x0 = dx_case(n, 256, 256, seed=5, max_ctas=0)
    assert torch.equal(x["raw"], x0["raw"])


@pytest.mark.parametrize("max_ctas", MAX_CTAS, ids=lambda v: "ctas_%s" % v)
@pytest.mark.parametrize("shape", [(256, 256, 256, 256), (10, 32, 256, 256)], ids=_dw_id)
def test_dw_grid_bound_and_determinism(shape, max_ctas):
    """dW / db are within the bound of their own grid (K = n + grid + 4) and bit-identical when run twice."""
    out, op, inn, ip = shape
    n = 40001
    mc = _max_ctas(max_ctas, n)
    checks, x = dw_case(n, out, op, inn, ip, seed=9, max_ctas=mc)
    for c in checks:
        assert_bound(*c[1:], what=c[0])
    _, y = dw_case(n, out, op, inn, ip, seed=9, max_ctas=mc)
    assert torch.equal(x["dW"].view(torch.int32), y["dW"].view(torch.int32))
    assert torch.equal(x["db"].view(torch.int32), y["db"].view(torch.int32))


# ------------------------------------------------------------------------------------------------ concurrent backward
@pytest.mark.parametrize("n,dims", [(40001, [82, 256, 256, 32]), (777, [50, 128, 256, 10])], ids=["n40001", "n777"])
def test_concurrent_backward_equals_serial(n, dims):
    """TcMlp.backward runs dW (side stream) and dX (main stream) of a layer concurrently on their SM shares.  Its
    gradient must be bit-identical to the same calls issued one after another on one stream with the same max_ctas."""
    engine, tcm = pkg("engine"), pkg("mlp_tc")
    g = torch.Generator().manual_seed(n)
    Ws = [torch.randn(dims[i + 1], dims[i], generator=g) / np.sqrt(dims[i]) for i in range(len(dims) - 1)]
    bs = [0.1 * torch.randn(dims[i + 1], generator=g) for i in range(len(dims) - 1)]
    h = torch.randn(n, dims[0], generator=g).to(dev())
    d_out = (torch.randn(n, dims[-1], generator=g) / n).to(dev())
    p = engine.FlatParams(Ws, bs, dev())
    m = tcm.TcMlp(n, p, dev(), h)
    m.forward(h)
    m.backward(h, d_out)
    torch.cuda.synchronize()
    concurrent = p.grad.clone()
    p.grad.fill_(float("nan"))
    # the loop of TcMlp.backward, serially
    n_dx = min(m.sm_count - 1, max(1, int(round(m.sm_count * m.dx_share))))
    n_dw = m.sm_count - n_dx
    tcm.pack_rows(d_out, m.pd[-1], out=m.dz_out)
    dz, dz_w = m.dz_out, m.pd[-1]
    for l in range(m.L - 1, -1, -1):
        act = m.acts[l - 1] if l > 0 else m.x0
        _call("ep_tc_linear_dw_bf16", n, dims[l + 1], dims[l], dz_w, m.pd[l], _p(dz), _p(act), _p(p.dW[l]), _p(p.db[l]),
              _p(m.ws), m.ws_bytes, n_dw if l > 0 else 0, _st())
        if l > 0:
            nxt = m.dz[l & 1]
            _call("ep_tc_linear_dx_bf16", n, dz_w, m.pd[l], _p(dz), _p(m.WTp[l]), _p(m.masks[l - 1]), _p(nxt), n_dx,
                  _st())
            dz, dz_w = nxt, m.pd[l]
    torch.cuda.synchronize()
    assert torch.isfinite(concurrent).all()
    assert torch.equal(p.grad.view(torch.int32), concurrent.view(torch.int32))


# ------------------------------------------------------------------------------------------------ output layer
FINAL_OUT = [1, 10, 16, 32, 50, 64, 128]
FINAL_CASES = [(n, "plain") for n in N_SET] + [(n, v) for n in (129, 40001) for v in ("scale_dev", "U_base_null", "strided")]


@pytest.mark.parametrize("out", FINAL_OUT, ids=lambda v: "out%d" % v)
@pytest.mark.parametrize("n,variant", FINAL_CASES, ids=["%s-%s" % c for c in FINAL_CASES])
def test_final_layer(n, variant, out):
    """corr = act W^T + b within the bound; U_pred = fl(U_base + fl(scale * corr)) bit for bit, with the scale from
    scale_dev when given (the scalar argument is then ignored); columns >= out of strided rows, and everything after
    the last row, untouched.  U_base_null: U_base = U_pred = NULL, corr only."""
    n = _n(n)
    checks, x = final_case(n, out, seed=n * 13 + out, variant=variant)
    for c in checks:
        assert_bound(*c[1:], what=c[0])
    c, ldc, ldu = x["c"], x["ldc"], x["ldu"]
    assert torch.isnan(c[:, out:]).all()
    assert_guard(x["corr_buf"], n * ldc)
    if x["U_pred"] is None:
        return
    ub = x["U_base"].view(n, ldu)[:, :out].cpu().numpy()
    want = ub + np.float32(x["scale"]) * c[:, :out].cpu().numpy()       # float32: product rounded, then the sum
    up = x["U_pred"].view(n, ldu)
    assert np.array_equal(up[:, :out].cpu().numpy().view(np.int32), want.view(np.int32))
    assert torch.isnan(up[:, out:]).all()
    assert_guard(x["up_buf"], n * ldu)


# ------------------------------------------------------------------------------------------------ hidden forward
HID_IN = [(3, 32), (82, 96), (146, 160), (256, 256)]
HID_OUT = [(50, 64), (100, 128), (256, 256)]


@pytest.mark.parametrize("out,op", HID_OUT, ids=["o%d" % op for _, op in HID_OUT])
@pytest.mark.parametrize("inn,ip", HID_IN, ids=["i%d" % ip for _, ip in HID_IN])
@pytest.mark.parametrize("n", [1, 129, 40001], ids=str)
def test_hidden_forward(n, inn, ip, out, op):
    """relu(act W^T + b) within the bound, padded features exactly 0, and every mask bit equal to (stored > 0) in the
    header's bit order."""
    checks, x = hidden_case(n, inn, ip, out, op, seed=n + 7 * ip + op)
    for c in checks:
        assert_bound(*c[1:], what=c[0])
    assert (x["got"][:, out:] == 0).all()
    assert torch.equal(x["bits"], x["got"] > 0)


# ------------------------------------------------------------------------------------------------ the comparator
def _ulp_bf16(v):
    return 2.0 ** (math.frexp(v)[1] - 8)


@pytest.mark.parametrize("kind", ["dX", "dW", "db", "corr", "hidden"])
def test_bound_rejects_two_ulp_error(kind):
    """The bound is not vacuous: the reference moved by 2 bf16 ulps at its largest entry fails assert_bound."""
    n = 129
    if kind == "dX":
        checks, _ = dx_case(n, 256, 256, seed=1)
    elif kind in ("dW", "db"):
        checks, _ = dw_case(n, 10, 32, 256, 256, seed=2)
    elif kind == "corr":
        checks, _ = final_case(n, 32, seed=3)
    else:
        checks, _ = hidden_case(n, 82, 96, 256, 256, seed=4)
    what, got, ref, E, u_out = next(c for c in checks if c[0] == kind)
    assert_bound(got, ref, E, u_out, what)
    i = int(ref.abs().argmax())
    moved = ref.clone()
    v = moved.view(-1)[i].item()
    moved.view(-1)[i] = v + 2 * _ulp_bf16(v)
    with pytest.raises(AssertionError):
        assert_bound(got, moved, E, u_out, what)


# ------------------------------------------------------------------------------------------------ packing
def special_bits(shape, g):
    """fp32 bit patterns (int64, CPU) with moderate exponents: many exactly halfway between two bf16 values (low half
    0x8000), others one below / above halfway, exact bf16 values, random low halves, and some +-0."""
    sign = torch.randint(0, 2, shape, generator=g) << 31
    hi = torch.randint(0x3000, 0x4F00, shape, generator=g) << 16
    lo = torch.tensor([0x8000, 0x8000, 0x7FFF, 0x8001, 0x0000])[torch.randint(0, 5, shape, generator=g)]
    lo = torch.where(torch.rand(shape, generator=g) < 0.3, torch.randint(0, 0x10000, shape, generator=g), lo)
    bits = sign | hi | lo
    return torch.where(torch.rand(shape, generator=g) < 0.02, sign, bits)


def as_f32(bits):
    return torch.where(bits >= 2 ** 31, bits - 2 ** 32, bits).to(torch.int32).view(torch.float32)


def rne_bf16(bits):
    """bf16 bit patterns (as int16) of fp32 bit patterns, round to nearest even (finite values)."""
    r = ((bits + 0x7FFF + ((bits >> 16) & 1)) >> 16) & 0xFFFF
    return torch.where(r >= 0x8000, r - 0x10000, r).to(torch.int16)


@pytest.mark.parametrize("n,d,dp,ldx,off", [(1, 3, 32, 8, 3), (127, 82, 96, 90, 5), (128, 32, 32, 40, 1),
                                            (129, 146, 160, 151, 2), (40001, 256, 256, 260, 4)])
def test_pack_rows(n, d, dp, ldx, off):
    """ep_tc_pack_rows_bf16 from a strided view at an offset (ldx > d): round to nearest even, ties included; padded
    rows and features written as zero; nothing written past the buffer."""
    g = torch.Generator().manual_seed(n + d)
    bits = special_bits((n + 1, ldx), g)
    X = as_f32(bits).to(dev())[1:, off:off + d]
    nbytes = _q("ep_tc_packed_rows_bytes", n, dp)
    out, buf = guarded_u8(nbytes)
    _call("ep_tc_pack_rows_bf16", n, d, dp, _p(X), ldx, _p(out), _st())
    torch.cuda.synchronize()
    assert_guard(buf, nbytes)
    Z = torch.zeros(_tiles(n) * 128, dp, dtype=torch.int16)
    Z[:n, :d] = rne_bf16(bits[1:, off:off + d])
    want = Z.view(-1, 128, dp // 8, 8).permute(0, 2, 1, 3).reshape(-1)
    assert torch.equal(out.cpu().view(torch.int16), want)


@pytest.mark.parametrize("with_wt", [True, False], ids=["WTp", "no_WTp"])
@pytest.mark.parametrize("out,inn,op,ip", [(256, 82, 256, 96), (10, 256, 32, 256), (100, 146, 128, 160), (3, 5, 32, 32),
                                           (256, 256, 256, 256), (20, 12, 24, 16)],
                         ids=["o256-i96", "o32-i256", "o128-i160", "o32-i32", "o256-i256", "o24-i16_no_pair"])
def test_pack_weight(out, inn, op, ip, with_wt):
    """ep_tc_pack_weight_bf16: Wp, WTp and both CTA-pair copies byte for byte against the index formulas, padding
    included.  Widths that are not multiples of 32 have no pair copy: the second half of each buffer stays as it was.
    Without WTp that buffer is untouched."""
    g = torch.Generator().manual_seed(out * 1000 + inn)
    bits = special_bits((out, inn), g)
    W = as_f32(bits).to(dev())
    Z = torch.zeros(op, ip, dtype=torch.int16)
    Z[:out, :inn] = rne_bf16(bits)
    want_wp, want_wt = weight_layouts(Z.view(torch.bfloat16), pair=op % 32 == 0 and ip % 32 == 0)
    nbytes = _q("ep_tc_packed_weight_bytes", op, ip)
    assert nbytes == 2 * op * ip * 2
    Wp, wp_buf = guarded_u8(nbytes)
    WTp, wt_buf = guarded_u8(nbytes)
    _call("ep_tc_pack_weight_bf16", out, inn, op, ip, _p(W), _p(Wp), _p(WTp) if with_wt else None, _st())
    torch.cuda.synchronize()
    assert torch.equal(wp_buf[:want_wp.numel()].cpu(), want_wp)
    assert_guard(wp_buf, want_wp.numel())
    if with_wt:
        assert torch.equal(wt_buf[:want_wt.numel()].cpu(), want_wt)
        assert_guard(wt_buf, want_wt.numel())
    else:
        assert_guard(wt_buf, 0)


# ------------------------------------------------------------------------------------------------ argument errors
ARG_ERRORS = ["dw_workspace_too_small", "dw_o32_i32", "dw_n0", "dx_in288", "dx_out288", "final_in288", "final_out288",
              "fwd_relu0", "final_U_base_null_U_pred_set"]


@pytest.mark.parametrize("case", ARG_ERRORS)
def test_argument_errors(case):
    """Host-side checks: each call raises EpError and launches nothing.  Buffers are sized for the request anyway."""
    EpError = pkg("_cabi").EpError
    u8 = lambda nbytes: torch.zeros(nbytes, dtype=torch.uint8, device=dev())
    rows = lambda n, dp: u8(128 * _tiles(max(n, 1)) * dp * 2)
    wts = lambda op, ip: u8(2 * op * ip * 2)
    f32 = lambda count: torch.zeros(count, device=dev())
    ws_bytes = _q("ep_tc_dw_workspace_bytes")
    ws = u8(ws_bytes)
    st = _st()
    with pytest.raises(EpError):
        if case == "dw_workspace_too_small":
            _call("ep_tc_linear_dw_bf16", 300, 256, 82, 256, 96, _p(rows(300, 256)), _p(rows(300, 96)), _p(f32(256 * 82)),
                  _p(f32(256)), _p(ws), ws_bytes - 1, 0, st)
        elif case == "dw_o32_i32":
            _call("ep_tc_linear_dw_bf16", 300, 32, 32, 32, 32, _p(rows(300, 32)), _p(rows(300, 32)), _p(f32(32 * 32)),
                  _p(f32(32)), _p(ws), ws_bytes, 0, st)
        elif case == "dw_n0":
            _call("ep_tc_linear_dw_bf16", 0, 256, 256, 256, 256, _p(rows(1, 256)), _p(rows(1, 256)), _p(f32(256 * 256)),
                  _p(f32(256)), _p(ws), ws_bytes, 0, st)
        elif case in ("dx_in288", "dx_out288"):
            op, ip = (256, 288) if case == "dx_in288" else (288, 256)
            _call("ep_tc_linear_dx_bf16", 1, op, ip, _p(rows(1, op)), _p(wts(op, ip)), _p(u8(128 * ip // 8)),
                  _p(rows(1, ip)), 0, st)
        elif case in ("final_in288", "final_out288"):
            ip, out, op = (288, 32, 32) if case == "final_in288" else (256, 260, 288)
            _call("ep_tc_linear_final_bf16", 1, ip, out, op, _p(rows(1, ip)), _p(wts(op, ip)), _p(f32(out)),
                  _p(f32(out)), out, None, 1.0, None, None, 0, st)
        elif case == "fwd_relu0":
            _call("ep_tc_linear_fwd_bf16", 1, 256, 256, 256, _p(rows(1, 256)), _p(wts(256, 256)), _p(f32(256)), 0,
                  _p(rows(1, 256)), _p(u8(128 * 32)), st)
        else:
            _call("ep_tc_linear_final_bf16", 1, 256, 32, 32, _p(rows(1, 256)), _p(wts(32, 256)), _p(f32(32)),
                  _p(f32(32)), 32, None, 1.0, None, _p(f32(32)), 32, st)
    torch.cuda.synchronize()
