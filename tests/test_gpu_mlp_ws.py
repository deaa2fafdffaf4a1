"""GPU: the warp-specialised fused MLP kernels (mlp_ws.cuh: k_mlp_fwd_ws, the nine k_mlp_bwd_ws<NG, NA, MODE>,
k_dw_planes, k_dw0_planes, k_bias_finish, k_planes_build and k_adam's plane emission) element by element against
float64, driven through the library's real pass dispatch (saceo.cu mlp_forward / mlp_backward, reached through
saceo_test_mlp_ws).  Each case states its route - fused or GEMM chain, the backward instantiation, dW1 / dW0 from the
plane images or the chain, biases from the column sums or the ones row - and asserts it from the route report.

The reference is layer-local: every stage is recomputed in float64 from the kernel's own fp32 inputs to that stage
(h2 from the kernel's h1, dH1 from the kernel's dH2, dW1 from the decoded h1 / dH2 images, ...), so errors do not
compound and a ReLU pre-activation within the bar of zero may take either branch.  Where a stage input is not
observable (dH1 of an input-gradient-only pass) the reference value stands in and its bar is carried through the
stage (|error| <= sum_k bar_k |b_k|).  Every element must satisfy |y - y64| <= bar, with the bar of each stage derived
in _fwd_bar / _bwd_bar / _dw_bar.  Every buffer is NaN-filled: padding words, rows >= rows and the activation buffers
a route does not write must stay bit-for-bit NaN."""
import ctypes as C
import zlib
from collections import defaultdict

import numpy as np
import pytest
import torch

from sac_expert_b200 import lib as L

pytestmark = pytest.mark.gpu

RELU, TANH, ELU = 0, 1, 2
H = 256
U = 2.0 ** -24                    # fp32 unit roundoff
F16_REL, F16_ABS = 2.0 ** -22, 2.0 ** -25       # fp16 hi/lo residual: relative, and absolute below 2^-3 (subnormal lo)
BF16_REL = 2.0 ** -16             # bf16 hi/lo residual
STAGE = 32768

COVERAGE = defaultdict(lambda: [0, 0.0])        # route -> [cases, largest err / bar]
VARIANTS = set()


@pytest.fixture(scope="module", autouse=True)
def _coverage_table():
    yield
    if COVERAGE:
        print("\nroute | cases | max err/bar")
        for k in sorted(COVERAGE):
            print("%s | %d | %.3g" % (k, COVERAGE[k][0], COVERAGE[k][1]))
        print("k_mlp_bwd_ws instantiations launched:", sorted(VARIANTS))


def rup(x, m):
    return (x + m - 1) // m * m


def _act64(act, v):
    if act == RELU:
        return np.maximum(v, 0.0)
    if act == TANH:
        return np.tanh(v)
    return np.where(v > 0, v, np.expm1(np.minimum(v, 0.0)))


def _dact64(act, h):             # dact_from_out: the derivative from the post-activation value
    if act == RELU:
        return (h > 0).astype(np.float64)
    if act == TANH:
        return 1.0 - h * h
    return np.where(h > 0, 1.0, h + 1.0)


def _offsets(inp, nout, hid=H):
    o = {"W0": 0, "b0": inp * hid}
    o["W1"] = o["b0"] + hid
    o["b1"] = o["W1"] + hid * hid
    o["W2"] = o["b1"] + hid
    o["b2"] = o["W2"] + hid * nout
    o["n"] = o["b2"] + nout
    return o


# ------------------------------------------------------------------------------------------
# plane image decoders (planes.cuh: ws_image_off / ws_w2_off; mlp_ws.cuh: ws_store_planes_p)
# ------------------------------------------------------------------------------------------
def _image_offsets(rows, cols=H):
    """Byte offset (hi plane; lo = +16384) of element (row, col) of a [rows x 256] image."""
    r = np.arange(rows)[:, None]
    c = np.arange(cols)[None, :]
    c8 = c >> 3
    return (r >> 5) * STAGE + (c8 >> 3) * 4096 + (r & 31) * 128 + (((c8 & 7) ^ (r & 7)) << 4) + (c & 7) * 2


def _u16(img, off):
    return img.view(np.uint8)[off[..., None] + np.arange(2)].view(np.uint16)[..., 0]


def decode_bf16(img, rows):
    off = _image_offsets(rows)
    hi = (_u16(img, off).astype(np.uint32) << 16).view(np.float32)
    lo = (_u16(img, off + 16384).astype(np.uint32) << 16).view(np.float32)
    return hi.astype(np.float64) + lo.astype(np.float64)


def _f16(u):
    return u.view(np.float16).astype(np.float64)


def decode_weights(img, inp, nout):
    """-> (W0 rows padded to 32, W1, W2^T section [N2 x 256] divided by the 2^8 scale or None)."""
    n0 = (inp + 31) // 32
    off = _image_offsets(n0 * 32 + H)
    w = _f16(_u16(img, off)) + _f16(_u16(img, off + 16384))
    w2 = None
    if nout > 1:
        N2 = rup(nout, 16)
        n = np.arange(N2)[:, None]
        j = np.arange(H)[None, :]
        c8 = j >> 3
        o = (n0 + 8) * STAGE + (c8 >> 3) * (N2 * 256) + n * 128 + (((c8 & 7) ^ (n & 7)) << 4) + (j & 7) * 2
        w2 = (_f16(_u16(img, o)) + _f16(_u16(img, o + N2 * 128))) / 256.0
    return w[:n0 * 32], w[n0 * 32:], w2


def check_weight_image(img, th, inp, nout):
    """hi + lo reconstructs every weight to 2^-22 relative, plus 2^-25 where the lo half is an fp16 subnormal (|w| <
    2^-3; the W2 section holds 256 W2, so 2^-33 there); rows >= in and W2 rows n >= nout are zero."""
    o = _offsets(inp, nout)
    W0 = th[o["W0"]:o["b0"]].reshape(inp, H).astype(np.float64)
    W1 = th[o["W1"]:o["b1"]].reshape(H, H).astype(np.float64)
    d0, d1, d2 = decode_weights(img, inp, nout)
    assert np.all(np.abs(d0[:inp] - W0) <= F16_REL * np.abs(W0) + F16_ABS)
    assert np.all(d0[inp:] == 0)
    assert np.all(np.abs(d1 - W1) <= F16_REL * np.abs(W1) + F16_ABS)
    if nout > 1:
        W2 = th[o["W2"]:o["b2"]].reshape(H, nout).astype(np.float64).T
        assert np.all(np.abs(d2[:nout] - W2) <= F16_REL * np.abs(W2) + F16_ABS / 256)
        assert np.all(d2[nout:] == 0)


# ------------------------------------------------------------------------------------------
# bars
# ------------------------------------------------------------------------------------------
def _fwd_bar(K, tc):
    """Relative part of a forward layer's bar, per element, T = sum_k |a_k||b_k| + |bias|.

    Tensor core, fp16 hi/lo operands (tc_gemm.cuh split8<true>, the forward error model): x = hi + lo + r with
    |x - hi| <= 2^-11 |x|, |r| <= 2^-22 |x| + 2^-25 (below |x| = 2^-3 the lo half is an fp16 subnormal of spacing 2^-24;
    X down to 1e-6 and small weights land there).  a.b - (ha.hb + ha.lb + la.hb) = la.lb + a.rb + ra.b, so each
    product is off by <= 3 * 2^-22 |a||b| + 2^-25 (|a| + |b|) (the absolute part is the floor, _floor).  The three
    products of every k go into the fp32 TMEM accumulator, one rounding each at <= 2^-23 (truncation allowed):
    3 K 2^-23.  Epilogue: + bias and the activation (tanhf / expm1f within 2 ulp, 1-Lipschitz): 6 * 2^-24.  The
    output layer of multi-output nets runs on the W2 section, which holds 256 W2: the power of two is removed
    exactly, the floor of its W2 operand is 2^-25 / 256.
    CUDA cores (single-output layer): an fp32 FMA chain of K products plus the fixed-order sum of four column groups
    and b2: (K + 6) 2^-24."""
    if not tc:
        return (K + 6) * U
    return 3 * F16_REL + 3 * K * 2 * U + 6 * U


def _bwd_bar(K):
    """Relative part of a backward-chain step's bar (dH2 = (dOut W2^T) act1'(h2) for NG > 0, dH1 = (dH2 W1^T)
    act0'(h1)).  The gradient operand goes in as fp16 hi/lo after a per-row power-of-two scale (ws_row_scale) that
    puts the row bound into [512, 1024): 22 significant bits relative to the row bound, not to the element - an
    element far below the bound lands in the fp16 subnormals with absolute residual 2^-25 / scale <= 2^-34 bound (a
    row-relative floor, added in verify).  The weight operand: fp16 hi/lo as in _fwd_bar.  The scale is removed exactly
    (power of two); act' is evaluated in fp32 from the saved post-activation (2 ulp) and multiplied (1 rounding),
    |act'| <= 1: 3 * 2^-22 + 3 K 2^-23 + 6 * 2^-24.  NG = 0 (single output): dH2 = d0 w2_j act1'(h2) in fp32, no
    accumulation: 6 * 2^-24."""
    if K == 0:
        return 6 * U
    return 3 * F16_REL + 3 * K * 2 * U + 6 * U


def _dw_bar(rows):
    """Relative part of a weight-gradient bar, T = sum_b |a_b||g_b| (+ the bias row).  k_dw_planes / k_dw0_planes and
    the chain's tensor-core GEMM use bf16 hi/lo operands (|r| <= 2^-16 |x|, full fp32 exponent range): 3 * 2^-16 per
    product, then 3 rows fp32 accumulations at <= 2^-23, and one rounding on the way out.  The CUDA-core GEMMs of the
    chain (row tails, skinny shapes) are fp32 FMA chains, well inside this bar.
    The bias gradients from the kernel's column sums (ws_store_planes_cs / ws_store_rows -> dbpart -> k_bias_finish)
    are fp32 sums in a fixed order: rows + 8 roundings, also inside it."""
    return 3 * BF16_REL + 3 * rows * 2 * U + 2 * U


def _image_bar(bar, ref):
    """Bar of a bf16 hi/lo activation image against the reference of the fp32 value v it was split from:
    |dec - v| <= 2^-16 |v| (hi = rn_bf16(v) within 2^-8 |v|, lo = rn_bf16(v - hi) within 2^-8 of that) and
    |v - ref| <= bar, so |dec - ref| <= bar + 2^-16 (|ref| + bar)."""
    return bar + BF16_REL * (np.abs(ref) + bar)


def _floor(A, B):
    """sum_k 2^-25 (|a_rk| + |b_kj|): the absolute fp16 residual of both operands of a tensor-core product."""
    return F16_ABS * (np.abs(A).sum(1)[:, None] + np.abs(B).sum(0)[None, :])


def _check(name, got, ref, bar, route, seed):
    assert np.all(np.isfinite(got)), (name, route, "seed %d" % seed, int((~np.isfinite(got)).sum()))
    err = np.abs(got.astype(np.float64) - ref)
    ratio = err / np.maximum(bar, 1e-300)
    worst = float(ratio.max()) if ratio.size else 0.0
    if worst > 1:
        i = np.unravel_index(int(ratio.argmax()), ratio.shape)
        raise AssertionError("%s (%s, seed %d): %d elements over the bar, worst at %s: got %r ref %r bar %r" % (
            name, route, seed, int((ratio > 1).sum()), i, got[i], ref[i], bar[i]))
    k = "%s %s" % (route, name)
    COVERAGE[k][0] += 1
    COVERAGE[k][1] = max(COVERAGE[k][1], worst)


# ------------------------------------------------------------------------------------------
# one pass through saceo_test_mlp_ws
# ------------------------------------------------------------------------------------------
class Buf:
    """A NaN-filled device buffer of fp32 blocks [agent][net] (rows x cols, leading dimension ld) at off + a sa + n sn."""

    def __init__(self, na, nn, rows, cols, ld, sa, sn, off=4):
        self.na, self.nn, self.rows, self.cols, self.ld, self.sa, self.sn, self.off = na, nn, rows, cols, ld, sa, sn, off
        self.size = off + (na - 1) * sa + (nn - 1) * sn + rows * ld + 9
        self.host = np.full(self.size, np.nan, np.float32)
        self.mask = np.zeros(self.size, bool)

    def idx(self, a, n, rows=None):
        base = self.off + a * self.sa + n * self.sn
        return base + np.arange(self.rows if rows is None else rows)[:, None] * self.ld + np.arange(self.cols)[None, :]

    def put(self, a, n, x):
        i = self.idx(a, n)
        self.host[i] = x
        self.mask[i] = True

    def upload(self):
        self.dev = torch.from_numpy(self.host.copy()).cuda()
        return self

    def ptr(self):
        return self.dev.data_ptr() + 4 * self.off

    def get(self, a, n, rows=None):
        return self.res[self.idx(a, n, rows)]

    def fetch(self):
        self.res = self.dev.cpu().numpy()
        return self.res


def _theta(rng, inp, nout, w2_scale, onehot, hid=H):
    o = _offsets(inp, nout, hid)
    th = np.zeros(o["n"], np.float32)
    lim0 = np.sqrt(6.0 / (inp + hid))
    if onehot:      # W0[k, perm(k)] only: h1 rows of one-hot inputs have one nonzero, layer 1 sums a single product
        W0 = np.zeros((inp, hid))
        W0[np.arange(inp), rng.permutation(hid)[:inp]] = rng.uniform(0.5, 1.5, inp)
        b0 = np.zeros(hid)
    else:
        W0 = rng.uniform(-lim0, lim0, (inp, hid))
        b0 = rng.standard_normal(hid) * 0.1
    th[o["W0"]:o["b0"]] = W0.ravel()
    th[o["b0"]:o["W1"]] = b0
    th[o["W1"]:o["b1"]] = rng.uniform(-np.sqrt(3.0 / hid), np.sqrt(3.0 / hid), hid * hid)
    th[o["b1"]:o["W2"]] = rng.standard_normal(hid) * 0.1
    th[o["W2"]:o["b2"]] = (rng.uniform(-1, 1, hid * nout) * w2_scale)
    th[o["b2"]:o["n"]] = rng.standard_normal(nout) * 0.1
    return th


def _x(rng, rows, inp, kind):
    if kind == "onehot":
        x = np.zeros((rows, inp))
        x[np.arange(rows), rng.integers(0, inp, rows)] = rng.uniform(0.5, 2.0, rows) * rng.choice([-1, 1], rows)
        return x.astype(np.float32)
    x = rng.standard_normal((rows, inp))
    if kind == "range":      # 1e-6 ... 1e3 within every row
        x = x * 10.0 ** rng.uniform(-6, 3, (rows, inp))
    return x.astype(np.float32)


def _dout(rng, rows, k, kind):
    d = rng.standard_normal((rows, k))
    if kind == "edges":     # row magnitudes 2^-60 .. 2^60, a zero row, a one-nonzero row, one element 2^20 above its row
        d *= 2.0 ** rng.integers(-60, 61, (rows, 1))
        d[0] = 0
        if rows > 1:
            d[1] = 0
            d[1, k - 1] = 3.0
        if rows > 2:
            d[2, 0] *= 2.0 ** 20
    return d.astype(np.float32)


def run_pass(c, seed, save_h=True):
    """Runs one case; returns (route report, dict of fetched results and inputs)."""
    lib = L.load()
    rng = np.random.default_rng(seed)
    na, nn, rows, inp, nout = c["agents"], c["nnet"], c["rows"], c["in"], c["nout"]
    hid = c.get("hidden", H)
    acts = c["acts"]
    nparams = _offsets(inp, nout, hid)["n"]
    sTn = rup(nparams, 4) + 8 if nn > 1 else 0
    sTa = nn * sTn if nn > 1 else rup(nparams, 4) + 12
    mis = 1 if c.get("misalign") else 0
    ldx = c.get("ldx", rup(inp, 4) + 4)
    rowsH = rup(rows, 32) + 3
    hn = nn + 1
    A_cols, grads, dxa = c.get("A_cols"), c.get("grads", True), c.get("A_cols") is not None
    bwd = grads or dxa
    # agent 2 repeats agent 0: two CTAs that carry the same problem must give bit-identical results
    pick = lambda a: 0 if a == 2 else a
    th, X, D = {}, {}, {}
    for a in range(na):
        for n in range(nn):
            if pick(a) != a:
                th[a, n], X[a, n], D[a, n] = th[pick(a), n], X[pick(a), n], D[pick(a), n]
                continue
            th[a, n] = _theta(rng, inp, nout, c.get("w2", 0.05), c.get("x") == "onehot", hid)
            X[a, n] = _x(rng, rows, inp, c.get("x", "normal"))
            D[a, n] = _dout(rng, rows, nout, c.get("dout", "normal"))
    Tb = Buf(na, nn, 1, nparams, nparams, sTa, sTn, off=4 + mis)
    Xb = Buf(na, nn, rows, inp, ldx, nn * (rows * ldx + 4 * (nn > 1)) + 8, rows * ldx + 4 if nn > 1 else 0)
    Ob = Buf(na, nn, rows, nout, nout + 3, nn * (rows * (nout + 3) + 5) + 7, rows * (nout + 3) + 5)
    Db = Buf(na, nn, rows, nout, nout + 2, nn * (rows * (nout + 2) + 3) + 6, rows * (nout + 2) + 3)
    Hb = [Buf(na, nn, rowsH, hid, hid, hn * rowsH * hid, rowsH * hid, off=0) for _ in range(2)]
    dHb = [Buf(na, nn, rowsH, hid, hid, hn * rowsH * hid, rowsH * hid, off=0) for _ in range(2)]
    Gb = Buf(na, nn, 1, nparams, nparams, sTa, sTn, off=4 + mis)
    Ab = Buf(na, nn, rows, A_cols, A_cols, nn * (rows * A_cols + 3) + 5, rows * A_cols + 3) if dxa else None
    for a in range(na):
        for n in range(nn):
            Tb.put(a, n, th[a, n][None])
            Xb.put(a, n, X[a, n])
            Db.put(a, n, D[a, n])
    for b in [Tb, Xb, Ob, Db, Gb] + Hb + dHb + ([Ab] if Ab else []):
        b.upload()
    # weight-plane image (bytes 0xFF until built) and bf16 activation images: rows < rows NaN, pad rows zero
    img_bytes = ((inp + 31) // 32 + 8) * STAGE + (rup(nout, 16) * 1024 if nout > 1 else 0)
    planes = torch.full((na * nn * img_bytes + 64,), 0xFF, dtype=torch.uint8, device="cuda")
    q_img = rup(rows, 32) * 1024
    sQn, sQa = q_img + 2048, nn * (q_img + 2048) + 4096
    act_imgs = []
    for _ in range(3):
        t = np.full(na * sQa + 64, 0xFF, np.uint8)
        for a in range(na):
            for n in range(nn):
                base = a * sQa + n * sQn
                view = t[base:base + q_img]
                pad = _image_offsets(rup(rows, 32))[rows:].ravel()
                for p in (pad, pad + 16384):
                    view[p] = 0
                    view[p + 1] = 0
        act_imgs.append(torch.from_numpy(t).cuda())
    tiles = -(-rows // 128)
    need = na * nn * tiles * 2 * H
    dbpart = torch.full((need + 64,), float("nan"), device="cuda")
    use_img = c.get("act_images", True)
    args = L.MlpWsArgs(n_agents=na, nnet=nn, hnets=hn, in_=inp, nout=nout, kout=nout, rows=rows, rowsAllocH=rowsH,
                       theta=Tb.ptr(), sTa=sTa, sTn=sTn, X=Xb.ptr(), ldx=ldx, sXa=Xb.sa, sXn=Xb.sn,
                       out=Ob.ptr(), ldo=Ob.ld, sOa=Ob.sa, sOn=Ob.sn,
                       dout=Db.ptr() if bwd else None, ldd=Db.ld, sDa=Db.sa, sDn=Db.sn,
                       planes=planes.data_ptr() if c.get("planes", True) else None,
                       H1p=act_imgs[0].data_ptr() if use_img else None,
                       dH2p=act_imgs[1].data_ptr() if use_img else None,
                       dH1p=act_imgs[2].data_ptr() if use_img else None, sQa=sQa, sQn=sQn,
                       dbpart=dbpart.data_ptr(), dbpart_cap=need - 1 if c.get("dbpart_small") else need,
                       grads=Gb.ptr() if grads else None, dXa=Ab.ptr() if Ab else None, A_cols=A_cols or 0,
                       sXaA=Ab.sa if Ab else 0, sXaN=Ab.sn if Ab else 0, save_h=int(save_h))
    args.hidden[0] = args.hidden[1] = hid
    args.act[0], args.act[1] = acts
    args.H[0], args.H[1] = Hb[0].ptr(), Hb[1].ptr()
    args.dH[0], args.dH[1] = dHb[0].ptr(), dHb[1].ptr()
    rep = L.MlpWsRoute()
    L.check(lib.saceo_test_mlp_ws(C.byref(args), C.byref(rep), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    for b in [Tb, Xb, Ob, Db, Gb] + Hb + dHb + ([Ab] if Ab else []):
        b.fetch()
    res = dict(T=Tb, X=Xb, O=Ob, D=Db, G=Gb, H=Hb, dH=dHb, A=Ab, planes=planes.cpu().numpy(), img_bytes=img_bytes,
               act_imgs=[t.cpu().numpy() for t in act_imgs], sQa=sQa, sQn=sQn, q_img=q_img, th=th, Xh=X, Dh=D,
               rowsH=rowsH, pick=pick)
    return rep, res


def _route_of(rep):
    r = {"fwd": "ws" if rep.n_fwd_ws else "chain",
         "bwd": (rep.bwd_ng, rep.bwd_na, rep.bwd_mode) if rep.n_bwd_ws else None,
         "dw1": "planes" if rep.n_dw_planes else "chain",
         "dw0": "planes" if rep.n_dw0_planes else "chain",
         "bias": "colsum" if rep.n_bias_finish else "ones",
         "plane_path": bool(rep.plane_path)}
    return r


def _unchanged_nan(buf, written):
    """Every word outside the blocks `written` (a list of index arrays) is still NaN."""
    keep = np.ones(buf.size, bool)
    for i in written:
        keep[i.ravel()] = False
    assert np.all(np.isnan(buf.res[keep])), int((~np.isnan(buf.res[keep])).sum())


def verify(c, rep, res, route, seed):
    na, nn, rows, inp, nout = c["agents"], c["nnet"], c["rows"], c["in"], c["nout"]
    hid = c.get("hidden", H)
    a0, a1 = c["acts"]
    A_cols, grads = c.get("A_cols"), c.get("grads", True)
    o = _offsets(inp, nout, hid)
    r = _route_of(rep)
    _chk = lambda name, got, ref, bar: _check(name, got, ref, bar, route, seed)
    # the output layer on the tensor core: the fused kernel's W2 section (nout > 1) or the chain's GEMM (which sends
    # 128-row tiles there); the fused kernel's single-output layer is an fp32 FMA chain on CUDA cores
    tc_out = nout > 1 or r["fwd"] == "chain"
    if c.get("planes", True) and r["fwd"] == "chain":     # no image is built for a net the fused kernels refuse
        assert np.all(res["planes"] == 0xFF)
    Ob, Hb, dHb, Gb, Ab = res["O"], res["H"], res["dH"], res["G"], res["A"]
    wH1, wH2, wdH1, wdH2, wO, wG, wA = [], [], [], [], [], [], []
    for a in range(na):
        for n in range(nn):
            th = res["th"][a, n].astype(np.float64)
            W0 = th[o["W0"]:o["b0"]].reshape(inp, hid); b0 = th[o["b0"]:o["W1"]]
            W1 = th[o["W1"]:o["b1"]].reshape(hid, hid); b1 = th[o["b1"]:o["W2"]]
            W2 = th[o["W2"]:o["b2"]].reshape(hid, nout); b2 = th[o["b2"]:o["n"]]
            X = res["Xh"][a, n].astype(np.float64)
            Dout = res["Dh"][a, n].astype(np.float64)
            if c.get("planes", True) and r["fwd"] == "ws" and a == 0:
                base = (a * nn + n) * res["img_bytes"]
                check_weight_image(res["planes"][base:base + res["img_bytes"]], res["th"][a, n], inp, nout)
            q0 = a * res["sQa"] + n * res["sQn"]
            img = lambda i: res["act_imgs"][i][q0:q0 + res["q_img"]]
            # ---- h1: the fp32 H1 or the bf16 plane image (decoded value within 2^-16 of the kernel's fp32 h1)
            ref1 = _act64(a0, X @ W0 + b0)
            bar1 = _fwd_bar(inp, True) * (np.abs(X) @ np.abs(W0) + np.abs(b0)) + _floor(X, W0)
            if r["plane_path"]:
                h1 = decode_bf16(img(0), rup(rows, 32))
                assert np.all(h1[rows:] == 0), "pad rows of the h1 image written"
                h1 = h1[:rows]
                _chk("h1 image", h1, ref1, _image_bar(bar1, ref1))
            else:
                h1 = Hb[0].get(a, n, rows).astype(np.float64)
                wH1.append(Hb[0].idx(a, n, rows))
                _chk("h1", h1, ref1, bar1)
            # ---- h2 from the kernel's h1
            ref2 = _act64(a1, h1 @ W1 + b1)
            bar2 = _fwd_bar(hid, True) * (np.abs(h1) @ np.abs(W1) + np.abs(b1)) + _floor(h1, W1)
            h2 = Hb[1].get(a, n, rows).astype(np.float64)
            wH2.append(Hb[1].idx(a, n, rows))
            _chk("h2", h2, ref2, bar2)
            # ---- out from the kernel's h2
            refo = h2 @ W2 + b2
            baro = _fwd_bar(hid, tc_out) * (np.abs(h2) @ np.abs(W2) + np.abs(b2))
            if r["fwd"] == "chain":
                baro = baro + _floor(h2, W2)
            elif tc_out:
                baro = baro + F16_ABS * (np.abs(W2).sum(0)[None, :] + np.abs(h2).sum(1)[:, None] / 256)
            _chk("out", Ob.get(a, n).astype(np.float64), refo, baro)
            wO.append(Ob.idx(a, n))
            if not (grads or A_cols):
                continue
            # ---- dH2 = (dOut W2^T) act1'(h2)
            fused = r["bwd"] is not None
            D2 = Dout @ W2.T
            absD2 = np.abs(Dout) @ np.abs(W2.T)
            if not fused:                 # the chain: a bf16x3 GEMM with the dact epilogue
                bar_d2 = (_dw_bar(nout) + 4 * U) * absD2
            elif nout == 1:
                bar_d2 = _bwd_bar(0) * absD2
            else:
                dmax = np.abs(Dout).max(1, keepdims=True)
                bar_d2 = _bwd_bar(rup(nout, 16)) * absD2 + 2.0 ** -34 * dmax * np.abs(W2).sum(1)[None, :] + \
                    2.0 ** -33 * np.abs(Dout).sum(1, keepdims=True)
            refd2 = D2 * _dact64(a1, h2)
            dh2, dh2_bar = None, None
            if r["dw1"] == "planes":
                dimg = decode_bf16(img(1), rup(rows, 32))
                assert np.all(dimg[rows:] == 0), "pad rows of the dH2 image written"
                dh2 = dimg[:rows]
                _chk("dH2 image", dh2, refd2, _image_bar(bar_d2, refd2))
                dh2_bar = BF16_REL / (1 - BF16_REL) * np.abs(dh2)       # the kernel's fp32 dH2 behind the decoded value
            elif grads or not fused:          # kept in fp32: MODE 0 with weight gradients, or the chain
                dh2 = dHb[1].get(a, n, rows).astype(np.float64)
                wdH2.append(dHb[1].idx(a, n, rows))
                _chk("dH2", dh2, refd2, bar_d2)
                dh2_bar = 0 * dh2
            else:       # input gradient only: dH2 is not kept, its reference and bar stand in
                dh2, dh2_bar = refd2, bar_d2
            # ---- dH1 = (dH2 W1^T) act0'(h1), act' from the h1 the kernel read (fp32 H1 or the decoded image)
            bound = (np.abs(Dout).sum(1, keepdims=True) * np.abs(W2).max()) if nout > 1 else \
                np.abs(Dout[:, :1]) * np.abs(W2[:, 0]).max()
            refd1 = (dh2 @ W1.T) * _dact64(a0, h1)
            bar_d1 = (_bwd_bar(H) if fused else _fwd_bar(hid, True) + 3 * BF16_REL) * (np.abs(dh2) @ np.abs(W1.T)) + \
                (2.0 ** -34 * bound * np.abs(W1).sum(1)[None, :] + F16_ABS * np.abs(dh2).sum(1, keepdims=True)) + \
                dh2_bar @ np.abs(W1.T)
            dh1, dh1_bar = None, None
            if r["dw0"] == "planes":
                dimg = decode_bf16(img(2), rup(rows, 32))
                assert np.all(dimg[rows:] == 0), "pad rows of the dH1 image written"
                dh1 = dimg[:rows]
                _chk("dH1 image", dh1, refd1, _image_bar(bar_d1, refd1))
                dh1_bar = BF16_REL / (1 - BF16_REL) * np.abs(dh1)
            elif grads or not fused:
                dh1 = dHb[0].get(a, n, rows).astype(np.float64)
                wdH1.append(dHb[0].idx(a, n, rows))
                _chk("dH1", dh1, refd1, bar_d1)
                dh1_bar = 0 * dh1
            else:
                dh1, dh1_bar = refd1, bar_d1
            if A_cols:
                W0a = W0[inp - A_cols:]
                refa = dh1 @ W0a.T
                bara = ((hid + 6) * U if fused else _dw_bar(hid)) * (np.abs(dh1) @ np.abs(W0a.T)) + dh1_bar @ np.abs(W0a.T)
                _chk("dXa", Ab.get(a, n).astype(np.float64), refa, bara)
                wA.append(Ab.idx(a, n))
            if not grads:
                continue
            # ---- weight and bias gradients from the stage inputs the kernels read
            G = Gb.get(a, n)[0].astype(np.float64)
            wG.append(Gb.idx(a, n))
            ebar = _dw_bar(rows)
            for name, A_, D_, Dbar, lo, hi_, bo in (("dW2", h2, Dout, 0 * Dout, o["W2"], o["b2"], o["b2"]),
                                                    ("dW1", h1, dh2, dh2_bar, o["W1"], o["b1"], o["b1"]),
                                                    ("dW0", X, dh1, dh1_bar, o["W0"], o["b0"], o["b0"])):
                refw = A_.T @ D_
                barw = ebar * (np.abs(A_.T) @ np.abs(D_)) + np.abs(A_.T) @ Dbar
                _chk(name, G[lo:hi_].reshape(refw.shape), refw, barw)
                nb = D_.shape[1]
                refb = D_.sum(0)
                barb = ebar * np.abs(D_).sum(0) + Dbar.sum(0)
                _chk("d" + name[1:].replace("W", "b"), G[bo:bo + nb], refb, barb)
    # padding, rows >= rows and the buffers this route does not write stay NaN
    _unchanged_nan(Ob, wO)
    _unchanged_nan(Hb[0], wH1)
    _unchanged_nan(Hb[1], wH2)
    _unchanged_nan(dHb[0], wdH1)
    _unchanged_nan(dHb[1], wdH2)
    _unchanged_nan(Gb, wG)
    if Ab:
        _unchanged_nan(Ab, wA)
    # agent 2 carries agent 0's problem: bit-identical
    if na > 2:
        for b in [Ob, Gb] + Hb + dHb + ([Ab] if Ab else []):
            for n in range(nn):
                assert np.array_equal(b.get(2, n), b.get(0, n), equal_nan=True)
        for t in res["act_imgs"]:
            for n in range(nn):
                s0, s2 = n * res["sQn"], 2 * res["sQa"] + n * res["sQn"]
                assert np.array_equal(t[s0:s0 + res["q_img"]], t[s2:s2 + res["q_img"]])


# ------------------------------------------------------------------------------------------
# cases: each states the route the dispatch must take
# ------------------------------------------------------------------------------------------
def R(fwd="ws", bwd=None, dw1="planes", dw0="planes", bias="colsum", pp=True):
    return {"fwd": fwd, "bwd": bwd, "dw1": dw1, "dw0": dw0, "bias": bias, "plane_path": pp}


CHAIN = R("chain", None, "chain", "chain", "ones", False)
CASES = [
    # plane path, MODE 1 (the SAC / SAC-EO training forms)
    dict(id="critic_mode1", agents=3, nnet=2, in_=11, nout=1, rows=276, acts=(RELU, RELU), route=R(bwd=(0, 0, 1))),
    dict(id="critic_mode1_r1", agents=3, nnet=2, in_=1, nout=1, rows=1, acts=(TANH, ELU), route=R(bwd=(0, 0, 1))),
    dict(id="critic_mode1_r31_in33", agents=3, nnet=1, in_=33, nout=1, rows=31, acts=(ELU, TANH), route=R(bwd=(0, 0, 1))),
    dict(id="actor_mode1_o6", agents=3, nnet=1, in_=17, nout=6, rows=448, acts=(RELU, TANH), route=R(bwd=(1, 0, 1)),
         dout="edges"),
    dict(id="actor_mode1_o16", agents=3, nnet=2, in_=64, nout=16, rows=129, acts=(TANH, TANH), route=R(bwd=(1, 0, 1)),
         w2=1e-3),
    dict(id="actor_mode1_o2_onehot", agents=3, nnet=1, in_=32, nout=2, rows=127, acts=(RELU, ELU), x="onehot",
         route=R(bwd=(1, 0, 1))),
    dict(id="actor_mode1_o15_w2big", agents=3, nnet=1, in_=3, nout=15, rows=128, acts=(ELU, RELU), w2=200.0,
         x="range", route=R(bwd=(1, 0, 1))),
    # plane path without weight gradients: the input gradient only (MODE 2), h1 read back from its image
    dict(id="critic_dxa_mode2", agents=3, nnet=2, in_=31, nout=1, rows=449, acts=(RELU, TANH), grads=False, A_cols=8,
         route=R(bwd=(0, 1, 2), dw1="chain", dw0="chain", bias="ones")),
    dict(id="critic_dxa_mode2_a1", agents=3, nnet=2, in_=45, nout=1, rows=1024, acts=(ELU, ELU), grads=False, A_cols=1,
         route=R(bwd=(0, 1, 2), dw1="chain", dw0="chain", bias="ones")),
    # plane path with dW0 on the chain (in > 64, rows > 448, ldx % 4 != 0): MODE 0 with h1 / dH2 images
    dict(id="actor_o17_in376", agents=3, nnet=1, in_=376, nout=17, rows=276, acts=(RELU, RELU), route=R(bwd=(2, 0, 0), dw0="chain")),
    dict(id="actor_o34_in65", agents=3, nnet=1, in_=65, nout=34, rows=128, acts=(TANH, RELU), route=R(bwd=(3, 0, 0), dw0="chain"),
         dout="edges"),
    dict(id="actor_o36_in393", agents=3, nnet=1, in_=393, nout=36, rows=31, acts=(ELU, TANH), route=R(bwd=(3, 0, 0), dw0="chain")),
    dict(id="actor_o32_rows449", agents=3, nnet=2, in_=11, nout=32, rows=449, acts=(RELU, TANH), route=R(bwd=(2, 0, 0), dw0="chain")),
    dict(id="actor_o33_ldx", agents=3, nnet=1, in_=17, nout=33, rows=129, acts=(TANH, ELU), ldx=19, route=R(bwd=(3, 0, 0), dw0="chain")),
    dict(id="critic_in65", agents=3, nnet=2, in_=65, nout=1, rows=276, acts=(RELU, RELU), route=R(bwd=(0, 0, 0), dw0="chain")),
    # no activation images: fused chain, MODE 0, fp32 dH; db from the column sums, dW on the GEMM chain
    dict(id="critic_noimg", agents=3, nnet=2, in_=17, nout=1, rows=127, acts=(TANH, RELU), act_images=False,
         route=R(bwd=(0, 0, 0), dw1="chain", dw0="chain", pp=False)),
    dict(id="actor_noimg_o16", agents=3, nnet=1, in_=45, nout=16, rows=1024, acts=(RELU, ELU), act_images=False,
         route=R(bwd=(1, 0, 0), dw1="chain", dw0="chain", pp=False), x="range", w2=0.1),
    dict(id="critic_dxa16", agents=3, nnet=2, in_=33, nout=1, rows=129, acts=(ELU, RELU), act_images=False, A_cols=16,
         grads=False, route=R(bwd=(0, 1, 0), dw1="chain", dw0="chain", bias="ones", pp=False)),
    dict(id="critic_dxa17", agents=3, nnet=2, in_=45, nout=1, rows=276, acts=(TANH, TANH), act_images=False, A_cols=17,
         grads=False, route=R(bwd=(0, 2, 0), dw1="chain", dw0="chain", bias="ones", pp=False)),
    dict(id="critic_dxa32_grads", agents=3, nnet=2, in_=64, nout=1, rows=31, acts=(RELU, ELU), act_images=False, A_cols=32,
         route=R(bwd=(0, 2, 0), dw1="chain", dw0="chain", pp=False)),
    dict(id="critic_dxa3_grads", agents=3, nnet=1, in_=11, nout=1, rows=448, acts=(RELU, TANH), act_images=False, A_cols=3,
         route=R(bwd=(0, 1, 0), dw1="chain", dw0="chain", pp=False)),
    # refusals: the GEMM chain takes the pass (or its backward) and meets the same element bars
    dict(id="refuse_nout37", agents=3, nnet=1, in_=17, nout=37, rows=129, acts=(RELU, TANH), route=CHAIN),
    dict(id="refuse_acols33", agents=3, nnet=2, in_=45, nout=1, rows=128, acts=(TANH, RELU), A_cols=33, grads=False,
         act_images=False, route=R("ws", None, "chain", "chain", "ones", False)),
    dict(id="refuse_hidden128", agents=3, nnet=2, in_=11, nout=1, rows=129, acts=(ELU, RELU), hidden=128, route=CHAIN),
    dict(id="refuse_misaligned", agents=3, nnet=1, in_=17, nout=6, rows=276, acts=(RELU, RELU), misalign=True, route=CHAIN),
    dict(id="refuse_dbpart", agents=3, nnet=2, in_=11, nout=1, rows=449, acts=(TANH, ELU), dbpart_small=True,
         route=R(bwd=(0, 0, 0), dw1="chain", dw0="chain", bias="ones", pp=False)),
    dict(id="refuse_noplanes", agents=3, nnet=2, in_=11, nout=1, rows=128, acts=(RELU, RELU), planes=False, route=CHAIN),
]
for _c in CASES:
    _c["in"] = _c.pop("in_")


@pytest.mark.parametrize("c", CASES, ids=[c["id"] for c in CASES])
def test_mlp_ws_pass(c):
    seed = zlib.crc32(c["id"].encode())
    rep, res = run_pass(c, seed)
    got = _route_of(rep)
    assert got == c["route"], (got, c["route"])
    if c["route"]["fwd"] == "chain" or c["route"]["bwd"] is None:
        assert rep.n_tc + rep.n_skinny + rep.n_simt > 0
    if rep.n_bwd_ws:
        VARIANTS.add(got["bwd"])
    verify(c, rep, res, c["id"].split("_")[0] + " " + str(got["bwd"]), seed)
    # a second launch gives bit-identical results
    rep2, res2 = run_pass(c, seed)
    for k in ("O", "G", "A"):
        if res[k] is not None:
            assert np.array_equal(res[k].res, res2[k].res, equal_nan=True), (k, "seed %d" % seed)
    for i in range(2):
        assert np.array_equal(res["H"][i].res, res2["H"][i].res, equal_nan=True), ("H", i, "seed %d" % seed)
        assert np.array_equal(res["dH"][i].res, res2["dH"][i].res, equal_nan=True), ("dH", i, "seed %d" % seed)
    for t1, t2 in zip(res["act_imgs"], res2["act_imgs"]):
        assert np.array_equal(t1, t2), "seed %d" % seed


def test_plane_path_refuses_a_chain_backward():
    """A pass on the plane path keeps h1 only as its image, which the GEMM chain cannot read: a backward the fused
    kernel does not take (here dXa over 33 columns) is refused instead of reading an fp32 h1 nobody wrote."""
    c = dict(CASES[[x["id"] for x in CASES].index("refuse_acols33")], act_images=True)
    with pytest.raises(L.SaceoError, match="plane path"):
        run_pass(c, seed=1)


def test_save_h_false_writes_no_activation():
    """The forward without save_h gives bit-identical outputs and writes neither H nor the h1 image."""
    c = dict(CASES[3], grads=False)
    rep1, r1 = run_pass(c, seed=3, save_h=True)
    rep2, r2 = run_pass(c, seed=3, save_h=False)
    assert rep1.n_fwd_ws == rep2.n_fwd_ws == 1 and rep1.plane_path and rep2.plane_path
    assert np.array_equal(r1["O"].res, r2["O"].res, equal_nan=True)
    assert not np.all(np.isnan(r1["H"][1].res))
    for b in r2["H"]:
        assert np.all(np.isnan(b.res))
    assert np.all((r2["act_imgs"][0] == 0xFF) | (r2["act_imgs"][0] == 0))
    assert not np.all((r1["act_imgs"][0] == 0xFF) | (r1["act_imgs"][0] == 0))


# ------------------------------------------------------------------------------------------
# plane maintenance: k_adam's emission (and its Polyak line) against a fresh k_planes_build
# ------------------------------------------------------------------------------------------
def _images(pop):
    return {k: pop.debug(k, torch.int32).clone() for k in ("pl_actor", "pl_q", "pl_qt")}


@pytest.mark.parametrize("A,per_state_std,tui", [(3, True, 1), (8, False, 2), (17, True, 1000), (17, False, 1)])
def test_planes_after_updates_match_a_fresh_build(A, per_state_std, tui):
    from sac_expert_b200.population import Population, PopulationSpec
    from sac_expert_b200.synth import fill_synthetic
    S, n = 11, 3
    pop = Population(PopulationSpec(n_agents=n, S=S, A=A, B=256, E=20, replay_capacity=600, per_state_std=per_state_std,
                                    target_update_int=tui, gemm_mode=L.GEMM_TCGEN05_BF16X3, use_graph=True))
    try:
        fill_synthetic(pop, seed=4, replay_rows=500)
        obs = torch.randn(n, 40, S, device="cuda", generator=torch.Generator("cuda").manual_seed(1))
        pop.actor_forward(obs)
        pop.update(5, num_timesteps=0, use_device_rng=True, seed=9)
        torch.cuda.synchronize()
        kept = _images(pop)
        L.check(pop.lib.saceo_weights_changed(pop.ctx))
        pop.actor_forward(obs)                  # ensure_planes rebuilds every image from the fp32 tables
        torch.cuda.synchronize()
        fresh = _images(pop)
        for k in kept:
            assert torch.equal(kept[k], fresh[k]), k
        # the images decode to the tables
        Ao = 2 * A if per_state_std else A
        for k, tab, inp, nout, nets in (("pl_actor", "actor", S, Ao, n), ("pl_q", "q", S + A, 1, 2 * n),
                                        ("pl_qt", "qt", S + A, 1, 2 * n)):
            img = fresh[k].cpu().numpy().view(np.uint8)
            ths = pop.t[tab].reshape(nets, -1).cpu().numpy()
            nb = img.size // nets
            for z in (0, nets - 1):
                check_weight_image(img[z * nb:(z + 1) * nb], ths[z], inp, nout)
        # saceo_actor_step alone marks the actor image stale: the forward after it rebuilds the image, which then is
        # what a fresh build gives (the forward before the step clears the tables' handed-out mark)
        ref = pop.t["actor"].clone()
        d = torch.randn_like(ref) * 1e-3
        pop.actor_forward(obs)
        torch.cuda.synchronize()
        before = _images(pop)["pl_actor"]
        assert not pop.t.dirty
        pop.actor_step(ref + d, d, torch.ones(n, device="cuda"))
        pop.actor_forward(obs)
        torch.cuda.synchronize()
        stepped = _images(pop)["pl_actor"]
        assert not torch.equal(stepped, before)
        L.check(pop.lib.saceo_weights_changed(pop.ctx))
        pop.actor_forward(obs)
        torch.cuda.synchronize()
        assert torch.equal(stepped, _images(pop)["pl_actor"])
    finally:
        pop.close()
