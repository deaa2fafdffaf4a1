"""GPU: the library's GEMM dispatch (saceo.cu gemm(), reached through saceo_test_gemm_ex) element by element against
float64, on every route one call can take: the tcgen05 streaming and register-staged kernels with the CUDA-core row
tail, the skinny kernel on rows (one or two passes) and role-swapped on columns, and the tiled SIMT kernel.  Each case
states the route it is meant to take and asserts it from the route report, so the coverage is proved by the run.

The reference is epi(op(A) . op(B) [+ ones row] + bias + addend) in float64 from the same fp32 inputs, for every
(agent, net).  Every element must satisfy |C - C64| <= eps * T with T = sum_k |a_ik||b_kj| + |bias_j| + |addend_ij|
(see _eps for the derivation of eps per engine and plane format); padding words of C and the operands hold NaN and
must stay bit-for-bit untouched or unread.  The last test runs depth-3 dynamics models through the real per-layer
chain at the same thresholds."""
import ctypes as C
import zlib
from collections import defaultdict

import numpy as np
import pytest
import torch

import oracle.sac_eo_oracle as O
from oracle.sac_eo_oracle import NetCfg, model_sample, to_torch_state
from sac_expert_b200 import lib as L
from tests.helpers import build, rel
from tests.test_gpu_model_depth import GRAD_TOL, init_net_any_depth
from tests.test_gpu_model_fit import _run, _setup

pytestmark = pytest.mark.gpu

SIMT, TC = L.GEMM_FP32_SIMT, L.GEMM_TCGEN05_BF16X3
RELU, TANH, ELU = 0, 1, 2
EPI_NONE, EPI_ACT, EPI_MUL_DACT = 0, 1, 2
U = 2.0 ** -24           # fp32 unit roundoff
NAN_BITS = np.float32(np.nan).view(np.uint32)

# route -> [cases, largest err / bound], printed at the end of the module (pytest -s)
COVERAGE = defaultdict(lambda: [0, 0.0])


@pytest.fixture(scope="module", autouse=True)
def _coverage_table():
    yield
    if COVERAGE:
        print("\nroute | cases | max err/bound")
        for k in sorted(COVERAGE):
            print("%s | %d | %.3g" % (k, COVERAGE[k][0], COVERAGE[k][1]))


def _eps(engine, f16, nnz, epi):
    """Relative part of the bar, per element (nnz: nonzero products op(A)_ik op(B)_kj of the element; a zero product
    adds exactly and costs no rounding).

    fp32 FMA chain (skinny, SIMT, every row tail): one rounding per nonzero product, two for bias and addend:
        (nnz + 2) * 2^-24.
    tcgen05 bf16x3: x = hi + lo + r with hi = rn_bf16(x), |x - hi| <= 2^-8 |x|, lo = rn_bf16(x - hi), |r| <= 2^-16 |x|;
        a.b - (ha.hb + ha.lb + la.hb) = la.lb + a.rb + ra.b + O(2^-24) <= 3 * 2^-16 |a||b|.  The three products of every
        k are added into the fp32 TMEM accumulator, one rounding each at <= 2^-23 (the tensor core may truncate):
        3 * 2^-16 + 3 nnz * 2^-23, then the fp32 bias / addend adds.
    tcgen05 fp16x3 (GemmP::f16): the same with 11-bit halves, |x - hi| <= 2^-11 |x|, |r| <= 2^-22 |x|: 3 * 2^-22 + ...;
        below 2^-14 the halves are subnormal with spacing 2^-24, so each operand also carries an absolute residual of
        2^-25 (the floor term in run_case).
    Epilogue: tanhf / expm1f are within 2 ulp of |act(v)| <= |v| <= T, and 1 - h^2 / h + 1 of the derivative within
        2 ulp of 1 while |act'| <= 1: 4 * 2^-24 more when an activation or derivative is applied."""
    e_epi = (2 + (4 if epi else 0)) * U
    if engine == "fp32":
        return nnz * U + e_epi
    split = 3 * 2.0 ** -22 if f16 else 3 * 2.0 ** -16
    return split + 3 * nnz * 2 * U + e_epi


def _act64(act, v):
    if act == RELU:
        return np.maximum(v, 0.0)
    if act == TANH:
        return np.tanh(v)
    return np.where(v > 0, v, np.expm1(np.minimum(v, 0.0)))


def _dact64(act, h):          # gemm_simt.cuh dact_from_out, from the fp32 post-activation value
    h = h.astype(np.float64)
    if act == RELU:
        return (h > 0).astype(np.float64)
    if act == TANH:
        return 1.0 - h * h
    return np.where(h > 0, 1.0, h + 1.0)


def _values(rng, shape, kind, scale):
    x = rng.standard_normal(shape)
    if kind == "f16mix":     # fp16-plane range: near the fp16 maximum, O(1) and deep in the fp16 subnormals
        pick = rng.integers(0, 3, shape)
        x = np.where(pick == 0, np.sign(x) * rng.uniform(3e4, 6e4, shape), np.where(pick == 1, x, x * 1e-6))
    return (x * scale).astype(np.float32)


def _aux(rng, shape, act):
    """Saved post-activations with the values where derivatives switch or vanish: exact zeros, tanh near +-1, elu
    near -1."""
    x = rng.standard_normal(shape)
    if act == RELU:
        h = np.maximum(x, 0.0)
    elif act == TANH:
        h = np.tanh(2 * x)
        h.flat[1::7] = np.sign(x.flat[1::7]) * (1 - 2.0 ** -20)
        h.flat[3::11] = np.sign(x.flat[3::11]) * (1 - 2.0 ** -11)
    else:
        h = np.where(x > 0, x, np.expm1(4 * x))
        h.flat[2::9] = -1 + 2.0 ** -20
        h.flat[5::13] = -0.9999
    h.flat[::5] = 0.0
    return h.astype(np.float32)


class Operand:
    """A population operand in one NaN-filled device buffer: block (agent a, net n) of `rows` x `cols` with leading
    dimension ld starts at off + a * sa + n * sn.  Everything outside the blocks stays NaN."""

    def __init__(self, blocks, rows, cols, ld, sa, sn, off):
        na, nn = len(blocks), len(blocks[0])
        self.rows, self.cols, self.ld, self.sa, self.sn, self.off = rows, cols, ld, sa, sn, off
        size = off + (na - 1) * sa + (nn - 1) * sn + rows * ld + 67
        host = np.full(size, np.nan, np.float32)
        self.mask = np.zeros(size, bool)
        for a in range(na):
            for n in range(nn):
                idx = self.index(a, n)
                host[idx] = blocks[a][n]
                self.mask[idx] = True
        self.host = host
        self.dev = torch.from_numpy(host).cuda()

    def index(self, a, n):
        base = self.off + a * self.sa + n * self.sn
        return base + np.arange(self.rows)[:, None] * self.ld + np.arange(self.cols)[None, :]

    def ptr(self):
        return self.dev.data_ptr() + 4 * self.off


def _strides(rows, ld, nnet, pad_n, pad_a, zero_net=False):
    sn = 0 if zero_net else rows * ld + pad_n
    sa = nnet * max(sn, rows * ld) + pad_a
    return sa, sn


def _route_key(rep, c):
    """Human-readable kernels of the tensor-core part and of the rest, from the route report (plus the shape, which
    names the skinny kernel's template bound MS and its BT variant)."""
    M, N = c["M"], c["N"]
    tc = None
    if rep.n_tc:
        tc = ("tc stream<%d,%d>" % (rep.tc_akc, rep.tc_bkc) if rep.tc_stream else
              "tc staged<%d,%d,%d>" % (rep.tc_bn, rep.tc_stages, rep.tc_threads))
    rest = M - rep.tc_rows
    ms = lambda m: next(b for b in (1, 4, 8, 16, 32) if m <= b)
    ldb = c["ldb"]
    tail = None
    if rep.n_simt:
        tail = "simt<%d,%d,%d>" % (c["ta"], c["tb"], c["ones"])
    elif rep.n_skinny == 2:
        tail = "skinny 2-pass MS32+MS%d BT%d" % (ms(rest - 32), int(c["tb"] and ldb != 1))
    elif rep.n_skinny == 1 and rest > 32:
        tail = "skinny cols MS%d BT%d" % (ms(N), int(not c["ta"] and c["lda"] != 1))
    elif rep.n_skinny == 1:
        tail = "skinny rows MS%d BT%d" % (ms(rest), int(c["tb"] and ldb != 1))
    return tc, tail


def run_case(c, seed):
    """Runs one gemm() call described by the case dict c and checks every element, every padding word and the route.
    Returns the route report."""
    lib = L.load()
    rng = np.random.default_rng(seed)
    M, N, K, ta, tb, ones = c["M"], c["N"], c["K"], c["ta"], c["tb"], c["ones"]
    na, nnet = c["agents"], c["nnet"]
    Mx = M - ones                                   # rows of X when op(A) = [X^T; 1]
    a_rows, a_cols = (K, Mx) if ta else (M, K)
    b_rows, b_cols = (N, K) if tb else (K, N)
    c["lda"] = lda = a_cols + c["lda_pad"]
    c["ldb"] = ldb = b_cols + c["ldb_pad"]
    ldc = N + c["ldc_pad"]
    sAa, sAn = _strides(a_rows, lda, nnet, *c["a_pad"], zero_net=c["zero_net_a"])
    sBa, sBn = _strides(b_rows, ldb, nnet, *c["b_pad"])
    sCa, sCn = _strides(M, ldc, nnet, *c["c_pad"])
    sa_, sb_ = c["scale"]

    opA, opB, bias, addend, aux, blkA, blkB = [], [], [], [], [], [], []
    for a in range(na):
        rowA, rowB = [], []
        shared = None
        for n in range(nnet):
            if c["zero_net_a"] and shared is not None:
                x = shared
            else:
                x = _values(rng, (Mx, K), c["kind"], sa_)
                # single-product rows: the bar there is one product's rounding, so a plane format or a k slab that
                # is off shows at full size instead of being averaged over K terms
                for i in range(2, Mx, 5):
                    v = x[i, (7 * i + a + n) % K]
                    x[i] = 0
                    x[i, (7 * i + a + n) % K] = v
                shared = x
            w = _values(rng, (K, N), c["kind"], sb_)
            full = np.concatenate([x, np.ones((1, K), np.float32)]) if ones else x
            opA.append(full.astype(np.float64)); opB.append(w.astype(np.float64))
            rowA.append(x.T if ta else x); rowB.append(w.T if tb else w)
            bias.append(_values(rng, (N,), "normal", sa_ * sb_ * 2) if c["bias"] else np.zeros(N, np.float32))
            addend.append(_values(rng, (M, N), "normal", sa_ * sb_ * 2) if c["addend"] else np.zeros((M, N), np.float32))
            aux.append(_aux(rng, (M, N), c["act"]) if c["epi"] == EPI_MUL_DACT else None)
        blkA.append(rowA); blkB.append(rowB)
    per = lambda lst: [lst[a * nnet:(a + 1) * nnet] for a in range(na)]
    Ad = Operand(blkA, a_rows, a_cols, lda, sAa, sAn, 16 + c["a_off"])
    Bd = Operand(blkB, b_rows, b_cols, ldb, sBa, sBn, 16 + c["b_off"])
    Cd = Operand([[np.full((M, N), np.nan, np.float32)] * nnet] * na, M, N, ldc, sCa, sCn, 16 + c["c_off"])
    Dd = Operand(per(addend), M, N, ldc, sCa, sCn, 16 + c["c_off"]) if c["addend"] else None
    Xd = Operand(per(aux), M, N, ldc, sCa, sCn, 16 + c["c_off"]) if c["epi"] == EPI_MUL_DACT else None
    # bias at the offset of a flat Keras [W | b] layout: after the K x N kernel, odd agent / net strides
    sbn, sba = K * N + N + 3, nnet * (K * N + N + 3) + 5
    bias_host = np.full(c["bias_off"] + (na - 1) * sba + (nnet - 1) * sbn + N + 9, np.nan, np.float32)
    for a in range(na):
        for n in range(nnet):
            o = c["bias_off"] + a * sba + n * sbn
            bias_host[o:o + N] = bias[a * nnet + n]
    bias_dev = torch.from_numpy(bias_host).cuda()

    g = L.GemmArgs(gemm_mode=c["mode"] | (c["variant"] << 8), n_agents=na, nnet=nnet, transA=ta, transB=tb, ones=ones,
                   M=M, N=N, K=K, lda=lda, ldb=ldb, ldc=ldc, sAa=sAa, sAn=sAn, sBa=sBa, sBn=sBn, sCa=sCa, sCn=sCn,
                   sba=sba, sbn=sbn, A=Ad.ptr(), B=Bd.ptr(), C=Cd.ptr(),
                   bias=bias_dev.data_ptr() + 4 * c["bias_off"] if c["bias"] else None,
                   addend=Dd.ptr() if Dd else None, aux=Xd.ptr() if Xd else None,
                   epi=c["epi"], act=c["act"], f16=c["f16"])
    rep = L.GemmRoute()
    L.check(lib.saceo_test_gemm_ex(C.byref(g), C.byref(rep), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()

    # route: the kinds of both parts, the tensor-core template and tc_rows where the case names them
    tc, tail = _route_key(rep, c)
    want = c["route"]
    got_kind = ("stream" if rep.tc_stream else "staged") if rep.n_tc else None
    got_tail = None if tail is None else "simt" if tail.startswith("simt") else " ".join(tail.split(" ")[:2])
    assert (got_kind, got_tail) == tuple(want[:2]), (tc, tail, want)
    if tc:
        assert tc == "tc " + want[2], (tc, want)
        if len(want) > 3:
            assert rep.tc_rows == want[3], (rep.tc_rows, want)
    else:
        assert rep.tc_rows == 0

    # a kernel that read an operand's NaN padding into a result shows as a non-finite element; C's padding must be
    # untouched
    out = Cd.dev.cpu().numpy()
    assert np.all(out[~Cd.mask].view(np.uint32) == NAN_BITS), "a padding word of C was written"
    worst = {"tc": 0.0, "rest": 0.0}
    amb = 0
    for a in range(na):
        for n in range(nnet):
            z = a * nnet + n
            A64, B64 = opA[z], opB[z]
            acc = A64 @ B64
            b64, d64 = bias[z].astype(np.float64), addend[z].astype(np.float64)
            pre = acc + b64[None, :] + d64
            T = np.abs(A64) @ np.abs(B64) + np.abs(b64)[None, :] + np.abs(d64)
            nnz = (A64 != 0).astype(np.float64) @ (B64 != 0).astype(np.float64)
            if c["epi"] == EPI_ACT:
                ref = _act64(c["act"], pre)
            elif c["epi"] == EPI_MUL_DACT:
                ref = pre * _dact64(c["act"], aux[z])
            else:
                ref = pre
            bound = _eps("fp32", 0, nnz, c["epi"]) * T
            r0 = rep.tc_rows
            if r0:
                btc = _eps("tc", c["f16"], nnz[:r0], c["epi"]) * T[:r0]
                if c["f16"]:     # fp16 subnormal halves: 2^-25 absolute per operand
                    btc += 2.0 ** -25 * ((np.abs(A64) @ (B64 != 0)) + ((A64 != 0) @ np.abs(B64)))[:r0]
                bound[:r0] = btc
            got_c = out[Cd.index(a, n)].astype(np.float64)
            assert np.all(np.isfinite(got_c)), "non-finite output in (agent %d, net %d)" % (a, n)
            err = np.abs(got_c - ref)
            ratio = np.divide(err, bound, out=np.where(err > 0, np.inf, 0.0), where=bound > 0)
            if c["epi"] == EPI_ACT and c["act"] in (RELU, ELU):
                # relu / elu are 1-Lipschitz, so an element whose pre-activation lies within the bar of 0 may take either
                # branch and still land inside the bar; count them so that the bar is not met by such luck alone
                amb += int(np.sum(np.abs(pre) <= bound))
            bad = np.argwhere(ratio > 1)
            assert bad.size == 0, ("(agent %d, net %d): %d elements outside the bar, max err/bound %.3g at %s "
                                   "(tc_rows %d): got %r want %r" % (a, n, len(bad), ratio.max(), tuple(bad[0]), r0,
                                                                     got_c[tuple(bad[0])], ref[tuple(bad[0])]))
            if r0:
                worst["tc"] = max(worst["tc"], float(ratio[:r0].max()))
            if r0 < M:
                worst["rest"] = max(worst["rest"], float(ratio[r0:].max()))
    assert amb <= max(4, M * N * na * nnet // 500), "%d elements within the bar of a relu / elu branch point" % amb
    if tc:
        key = tc + (" f16" if c["f16"] else "")
        COVERAGE[key][0] += 1
        COVERAGE[key][1] = max(COVERAGE[key][1], worst["tc"])
    if tail:
        COVERAGE[tail][0] += 1
        COVERAGE[tail][1] = max(COVERAGE[tail][1], worst["rest"])
    return rep, worst


def G(name, route, M, N, K, mode=TC, ta=0, tb=0, ones=0, **kw):
    """One case.  route = (tensor-core kernel, rest, tc kernel template[, tc_rows]): tensor-core kernel "stream",
    "staged" or None; rest "skinny rows", "skinny 2-pass", "skinny cols", "simt" or None."""
    c = dict(M=M, N=N, K=K, mode=mode, ta=ta, tb=tb, ones=ones, agents=2, nnet=1, variant=0, f16=0, epi=EPI_NONE,
             act=RELU, bias=True, addend=False, kind="normal", scale=(1.0, 1.0), lda_pad=0, ldb_pad=0, ldc_pad=0,
             a_pad=(4, 8), b_pad=(4, 8), c_pad=(4, 8), a_off=0, b_off=0, c_off=0, zero_net_a=False, route=route)
    c["bias_off"] = K * N
    for k, v in kw.items():
        assert k in c, k
        c[k] = v
    return pytest.param(c, id=name)


ST10, ST00, ST01 = ("stream", None, "stream<1,0>"), ("stream", None, "stream<0,0>"), ("stream", None, "stream<0,1>")
R256, R128, R64 = ("staged", None, "staged<256,2,512>"), ("staged", None, "staged<128,3,512>"), ("staged", None, "staged<64,4,512>")
V128, V64 = ("staged", None, "staged<128,1,256>"), ("staged", None, "staged<64,1,256>")


def r(base, rest=None, rows=None):
    t = (base[0], rest, base[2])
    return t + (rows,) if rows is not None else t


ROWS, TWO, COLS, SIMT_ = "skinny rows", "skinny 2-pass", "skinny cols", "simt"
FWD = dict(f16=1, epi=EPI_ACT, act=TANH)            # a hidden layer of a forward pass

CASES = [
    # ---- tcgen05 streaming: all three instantiations; NT goes to the staged kernel by design
    G("stream-NN-fwd", r(ST10, rows=256), 256, 256, 64, **FWD),
    G("stream-NN-K32", r(ST10, rows=128), 128, 256, 32, f16=1),
    G("stream-NN-K96-tail3", r(ST10, ROWS, 128), 131, 512, 96, f16=1, epi=EPI_ACT, act=RELU),
    G("stream-NN-bf16", r(ST10, rows=256), 256, 256, 128),
    G("stream-TN-ones-dW", r(ST00, ROWS, 256), 257, 256, 64, ta=1, ones=1),
    G("stream-TN-ones-partial", r(ST00, ROWS, 200), 201, 256, 96, ta=1, ones=1),
    G("stream-TN", r(ST00, rows=384), 384, 256, 32, ta=1),
    G("stream-TT", r(ST01, rows=128), 128, 256, 32, ta=1, tb=1),
    G("stream-TT-partial", r(ST01, rows=200), 200, 512, 64, ta=1, tb=1),
    G("stream-NN-f16-partial", r(ST10, rows=20), 20, 256, 64, f16=1),
    G("NT-staged-by-design", r(R256, rows=256), 256, 256, 64, tb=1),
    G("NT-staged-by-design-f16", r(R256, rows=256), 256, 512, 128, tb=1, f16=1),
    # ---- register-staged tile widths, variant 1 and the forced variant 2
    G("staged-N200", r(R256, rows=128), 128, 200, 64, **FWD),
    G("staged-N129", r(R256, rows=256), 256, 129, 64),
    G("staged-N128", r(R128, rows=256), 256, 128, 64, **FWD),
    G("staged-N65", r(R128, rows=128), 128, 65, 40),
    G("staged-N64", r(R64, rows=256), 256, 64, 64),
    G("staged-N33", r(R64, rows=128), 128, 33, 70, f16=1),
    G("staged-N384-K200", r(R256, rows=140), 140, 384, 200, ta=1),
    G("v1-stream-still", r(ST10, rows=256), 256, 256, 64, variant=1),
    G("v1-N200", r(V128, rows=256), 256, 200, 64, variant=1),
    G("v1-N65", r(V128, rows=128), 128, 65, 64, variant=1, tb=1),
    G("v1-N64", r(V64, rows=256), 256, 64, 64, variant=1, f16=1),
    G("v1-N40-TN-ones", r(V64, ROWS, 128), 129, 40, 64, variant=1, ta=1, ones=1),
    G("v2-forced-NN", r(R256, rows=256), 256, 256, 64, variant=2, **FWD),
    G("v2-forced-TN-ones", r(R256, ROWS, 256), 257, 256, 64, variant=2, ta=1, ones=1),
    G("v2-forced-TT", r(R256, rows=128), 128, 512, 32, variant=2, ta=1, tb=1),
    # ---- streaming refused, one reason each
    G("refuse-A-base", r(R256, rows=256), 256, 256, 64, a_off=1),
    G("refuse-B-base", r(R256, ROWS, 256), 257, 256, 64, ta=1, ones=1, b_off=2),
    G("refuse-C-base-ok", r(ST10, rows=256), 256, 256, 64, c_off=1),
    G("refuse-agent-stride-1", r(R256, rows=128), 128, 256, 64, a_pad=(4, 9)),
    G("refuse-net-stride-2", r(R256, rows=128), 128, 256, 64, nnet=2, b_pad=(6, 8)),
    G("refuse-lda-2", r(R256, rows=128), 128, 256, 64, lda_pad=2),
    G("refuse-K48", r(R256, rows=256), 256, 256, 48),
    G("refuse-K72-TN", r(R256, rows=128), 128, 256, 72, ta=1),
    G("refuse-N384", r(R256, rows=256), 256, 384, 64),
    G("refuse-N320-TT", r(R256, rows=128), 128, 320, 64, ta=1, tb=1),
    # ---- tc_rows: M mod 128 at 3 / 4 / 15 / 16 without and with a full tile before it; ONES moves each by one row
    G("rows-3", (None, ROWS), 3, 256, 64),
    G("rows-4", (None, ROWS), 4, 256, 64),
    G("rows-15", (None, ROWS), 15, 256, 64),
    G("rows-16", r(ST10, rows=16), 16, 256, 64),
    G("rows-131", r(ST10, ROWS, 128), 131, 256, 64),
    G("rows-132", r(ST10, rows=132), 132, 256, 64),
    G("rows-143", r(ST10, rows=143), 143, 256, 64),
    G("rows-144", r(ST10, rows=144), 144, 256, 64),
    G("rows-259", r(R128, ROWS, 256), 259, 128, 64, **FWD),
    G("ones-4", (None, ROWS), 4, 256, 64, ta=1, ones=1),
    G("ones-5", (None, ROWS), 5, 256, 64, ta=1, ones=1),
    G("ones-16", (None, ROWS), 16, 256, 64, ta=1, ones=1),
    G("ones-17", r(ST00, ROWS, 16), 17, 256, 64, ta=1, ones=1),
    G("ones-132", r(R256, ROWS, 128), 132, 256, 64, ta=1, ones=1),
    G("ones-133", r(ST00, ROWS, 132), 133, 256, 64, ta=1, ones=1),
    G("ones-144", r(R256, ROWS, 143), 144, 256, 64, ta=1, ones=1),
    G("ones-145", r(ST00, ROWS, 144), 145, 256, 64, ta=1, ones=1),
    G("r96-small-panel", r(R64, rows=96), 96, 64, 32),
    G("r95-small-panel", (None, SIMT_), 95, 64, 32),
    G("lone-tile-NK-16384", r(R128, rows=20), 20, 128, 128),
    G("lone-tile-NK-16256", (None, ROWS), 20, 128, 127),
    G("N32-refused", (None, COLS), 256, 32, 64),
    G("N33-tc", r(R64, rows=256), 256, 33, 64),
    G("K7-refused", (None, SIMT_), 256, 64, 7),
    G("K8-tc", r(R64, rows=256), 256, 64, 8),
    G("K8-ones-tail", r(R64, ROWS, 128), 129, 64, 8, ta=1, ones=1),
    # ---- skinny rows: every MS bound, both BT variants, the two-pass case, K tails
    G("sk-MS1", (None, ROWS), 1, 300, 70, mode=SIMT),
    G("sk-MS1-BT", (None, ROWS), 1, 300, 70, mode=SIMT, tb=1),
    G("sk-MS4-3", (None, ROWS), 3, 130, 33, mode=SIMT),
    G("sk-MS4-4-BT", (None, ROWS), 4, 130, 33, mode=SIMT, tb=1),
    G("sk-MS8-5", (None, ROWS), 5, 64, 64, mode=SIMT, ta=1),
    G("sk-MS8-8-BT", (None, ROWS), 8, 64, 64, mode=SIMT, ta=1, tb=1),
    G("sk-MS16-9", (None, ROWS), 9, 257, 31, mode=SIMT),
    G("sk-MS16-16-BT", (None, ROWS), 16, 257, 31, mode=SIMT, tb=1),
    G("sk-MS32-17", (None, ROWS), 17, 512, 256, mode=SIMT),
    G("sk-MS32-32-BT", (None, ROWS), 32, 512, 256, mode=SIMT, tb=1),
    G("sk-K1", (None, ROWS), 20, 256, 1, mode=SIMT),
    G("sk-K1-BT", (None, ROWS), 20, 256, 1, mode=SIMT, tb=1),
    G("sk-K1-tc-mode", (None, ROWS), 7, 256, 1),
    G("sk-ones-20", (None, ROWS), 20, 64, 100, mode=SIMT, ta=1, ones=1),
    G("sk-2pass-33", (None, TWO), 33, 64, 100, mode=SIMT),
    G("sk-2pass-36-ones-dW0", (None, TWO), 36, 256, 64, mode=SIMT, ta=1, ones=1),
    G("ones-36-dW0-lone-tile", r(R256, ROWS, 35), 36, 256, 64, ta=1, ones=1),
    G("sk-2pass-48-BT", (None, TWO), 48, 100, 45, mode=SIMT, tb=1),
    G("sk-2pass-64", (None, TWO), 64, 33, 65, mode=SIMT),
    G("sk-2pass-64-tc-K7", (None, TWO), 64, 256, 7),
    G("sk-65-not-2pass", (None, SIMT_), 65, 64, 20, mode=SIMT),
    # ---- role-swapped skinny (N <= 32): heads 1, A, 2A, S+1; ones column; bias by the short index
    G("cols-N1-head", (None, COLS), 256, 1, 256, mode=SIMT),
    G("cols-N1-head-tc", (None, COLS), 256, 1, 256),
    G("cols-N3-A", (None, COLS), 256, 3, 256),
    G("cols-N6-2A", (None, COLS), 100, 6, 64, mode=SIMT),
    G("cols-N8-A", (None, COLS), 33, 8, 64),
    G("cols-N12-S1", (None, COLS), 200, 12, 128, mode=SIMT),
    G("cols-N16-2A", (None, COLS), 45, 16, 40),
    G("cols-N17-A", (None, COLS), 300, 17, 256),
    G("cols-N28-S1", (None, COLS), 64, 28, 64),
    G("cols-N32", (None, COLS), 257, 32, 256, mode=SIMT),
    G("cols-NT-dX-S11", (None, COLS), 256, 11, 256, tb=1),
    G("cols-TN-ones-N1", (None, COLS), 257, 1, 64, ta=1, ones=1),
    G("cols-TN-ones-N3", (None, COLS), 257, 3, 64, ta=1, ones=1, mode=SIMT),
    G("cols-TN-ones-N6", (None, COLS), 65, 6, 32, ta=1, ones=1),
    G("cols-TN-ones-N12", (None, COLS), 129, 12, 256, ta=1, ones=1),
    G("cols-TN-ones-N28", (None, COLS), 513, 28, 20, ta=1, ones=1),
    G("cols-TT-N17", (None, COLS), 40, 17, 35, ta=1, tb=1),
    G("cols-K1", (None, COLS), 100, 4, 1, mode=SIMT),
    G("cols-K33", (None, COLS), 100, 4, 33, mode=SIMT, tb=1),
    # ---- SIMT: all five instantiations and the 64-wide tile edges
    G("simt-NN", (None, SIMT_), 256, 256, 64, mode=SIMT),
    G("simt-NT", (None, SIMT_), 129, 65, 17, mode=SIMT, tb=1),
    G("simt-TN", (None, SIMT_), 65, 64, 16, mode=SIMT, ta=1),
    G("simt-TN-ones", (None, SIMT_), 100, 64, 100, mode=SIMT, ta=1, ones=1),
    G("simt-TT", (None, SIMT_), 128, 127, 15, mode=SIMT, ta=1, tb=1),
    G("simt-edge-65x33", (None, SIMT_), 65, 33, 1, mode=SIMT),
    G("simt-edge-128x128", (None, SIMT_), 128, 128, 128, mode=SIMT),
    G("simt-edge-193x257", (None, SIMT_), 193, 257, 47, mode=SIMT),
    G("simt-tc-mode-K7", (None, SIMT_), 300, 100, 7, ta=1),
    G("simt-tc-mode-ones-K4", (None, SIMT_), 200, 40, 4, ta=1, ones=1),
    # ---- epilogues: bias alone, bias + addend, act and act' from saved outputs, on every engine
    *[G("epi-%s-%s-%s" % (nm, ["relu", "tanh", "elu"][act], ["act", "dact"][epi - 1]), rt, M, N, K, mode=md, act=act,
        epi=epi, addend=True, **x)
      for nm, rt, M, N, K, md, x in (
          ("stream", r(ST10, rows=256), 256, 256, 64, TC, dict(f16=1)),
          ("staged-vec", r(R128, ROWS, 128), 130, 128, 64, TC, dict(tb=1)),
          ("staged-scalar", r(R64, rows=128), 128, 61, 64, TC, dict(ldc_pad=2)),
          ("rows", (None, ROWS), 20, 130, 50, SIMT, {}),
          ("cols", (None, COLS), 100, 7, 50, SIMT, {}),
          ("simt", (None, SIMT_), 100, 70, 30, SIMT, {}))
      for act in (RELU, TANH, ELU) for epi in (EPI_ACT, EPI_MUL_DACT)],
    G("epi-bias-only-stream", r(ST10, rows=256), 256, 256, 64, bias_off=1155),
    G("epi-bias-addend-stream", r(ST10, rows=256), 256, 256, 64, addend=True),
    G("epi-no-bias-staged", r(R256, rows=128), 128, 200, 64, bias=False, addend=True),
    G("epi-bias-1155-cols", (None, COLS), 256, 33 - 1, 35, bias_off=1155),
    G("epi-bias-1155-fwd-l0", r(R64, rows=256), 256, 33, 35, bias_off=1155, **FWD),
    G("epi-bias-1155-simt", (None, SIMT_), 256, 33, 35, mode=SIMT, bias_off=1155),
    G("epi-bias-odd-rows", (None, ROWS), 17, 33, 35, mode=SIMT, bias_off=1155, addend=True),
    G("epi-dact-2pass", (None, TWO), 40, 256, 64, mode=SIMT, epi=EPI_MUL_DACT, act=TANH, addend=True),
    G("epi-dact-tail", r(ST10, ROWS, 128), 131, 256, 64, epi=EPI_MUL_DACT, act=ELU),
    # ---- population strides: 3 agents x 2 nets, padded strides, a zero net stride, leading dims above the minimum
    G("pop-stream", r(ST10, ROWS, 128), 130, 256, 64, agents=3, nnet=2, a_pad=(8, 12), c_pad=(4, 20), **FWD),
    G("pop-stream-TN-ones", r(ST00, ROWS, 128), 130, 256, 64, agents=3, nnet=2, ta=1, ones=1, lda_pad=3),
    G("pop-staged-zero-net", r(R128, rows=150), 150, 100, 41, agents=3, nnet=2, zero_net_a=True, lda_pad=7, **FWD),
    G("pop-stream-zero-net", r(ST10, rows=132), 132, 256, 64, agents=3, nnet=2, zero_net_a=True, lda_pad=4, f16=1),
    G("pop-rows-zero-net", (None, ROWS), 20, 512, 41, mode=SIMT, agents=3, nnet=2, zero_net_a=True, lda_pad=5, **FWD),
    G("pop-2pass", (None, TWO), 36, 256, 64, mode=SIMT, agents=3, nnet=2, ta=1, ones=1, lda_pad=9, c_pad=(3, 5)),
    G("pop-cols", (None, COLS), 150, 3, 64, agents=3, nnet=2, lda_pad=5, ldc_pad=2, a_pad=(1, 3), c_pad=(1, 2)),
    G("pop-cols-ones", (None, COLS), 150, 12, 64, agents=3, nnet=2, ta=1, ones=1, lda_pad=2, b_pad=(5, 7)),
    G("pop-simt", (None, SIMT_), 150, 100, 41, mode=SIMT, agents=3, nnet=2, lda_pad=7, ldb_pad=3, ldc_pad=5,
      a_pad=(1, 2), b_pad=(3, 5), c_pad=(7, 11), epi=EPI_MUL_DACT, act=RELU, addend=True),
    G("pop-simt-tc-mode-K7", (None, SIMT_), 130, 70, 7, nnet=2, epi=EPI_ACT, act=ELU),
    G("pop-staged-ldc", r(R256, rows=256), 256, 200, 64, agents=3, nnet=2, ldc_pad=5, c_pad=(2, 6), tb=1, ldb_pad=3),
    # ---- operand range (INTEGRATION.md 5)
    G("range-f16-stream", r(ST10, rows=256), 256, 256, 64, f16=1, kind="f16mix"),
    G("range-f16-staged", r(R128, rows=144), 144, 100, 72, f16=1, kind="f16mix"),
    G("range-bf16-2^60-stream", r(ST00, ROWS, 256), 257, 256, 64, ta=1, ones=1, scale=(2.0 ** 60, 2.0 ** -60)),
    G("range-bf16-2^-60-stream", r(ST01, rows=128), 128, 256, 64, ta=1, tb=1, scale=(2.0 ** -60, 2.0 ** 60)),
    G("range-bf16-tiny-staged", r(R64, rows=256), 256, 64, 64, tb=1, scale=(2.0 ** -60, 2.0 ** -40)),
    G("range-bf16-huge-staged", r(R256, rows=256), 256, 300, 64, scale=(2.0 ** 40, 2.0 ** 40)),
    G("range-2^60-rows", (None, ROWS), 9, 256, 64, scale=(2.0 ** 60, 2.0 ** -60)),
    G("range-2^-60-cols", (None, COLS), 256, 6, 64, scale=(2.0 ** -60, 2.0 ** -40)),
    G("range-fp32-1e6-simt", (None, SIMT_), 200, 200, 64, mode=SIMT, scale=(1e6, 1e6), addend=True),
    G("range-fp32-1e6-rows", (None, ROWS), 30, 200, 64, mode=SIMT, scale=(1e6, 1e6)),
    G("range-fp32-1e6-cols", (None, COLS), 200, 20, 64, mode=SIMT, scale=(1e6, 1e6)),
]


@pytest.mark.parametrize("case", CASES)
def test_gemm_dispatch(case):
    run_case(dict(case), seed=zlib.crc32(repr(sorted(case.items())).encode()))


@pytest.mark.parametrize("mode", [SIMT, TC])
@pytest.mark.parametrize("M,N,K", [(0, 64, 64), (128, 0, 64), (128, 256, 0), (0, 0, 0), (40, 7, 0)])
def test_gemm_empty_writes_nothing(mode, M, N, K):
    lib = L.load()
    buf = torch.full((4096,), float("nan"), device="cuda")
    src = torch.randn(4096, device="cuda")
    g = L.GemmArgs(gemm_mode=mode, n_agents=2, nnet=1, M=M, N=N, K=K, lda=max(K, 1), ldb=max(N, 1), ldc=max(N, 1),
                   sAa=1024, sBa=1024, sCa=1024, sba=8, A=src.data_ptr(), B=src.data_ptr(), C=buf.data_ptr(),
                   bias=src.data_ptr(), addend=src.data_ptr(), epi=EPI_ACT, act=TANH)
    rep = L.GemmRoute()
    L.check(lib.saceo_test_gemm_ex(C.byref(g), C.byref(rep), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    assert (rep.n_tc, rep.n_skinny, rep.n_simt) == (0, 0, 0)
    assert np.all(buf.cpu().numpy().view(np.uint32) == NAN_BITS)


def test_simt_tail_after_tensor_cores_is_unreachable():
    """gemm()'s SIMT launch with m_off > 0 would finish rows after a tensor-core part, but tc_rows leaves at most 3 rows
    plus the ones row, which always go to the skinny kernel.  Every M of the first four row tiles, with and without the
    ones row, on both tile widths."""
    lib = L.load()
    A, B, Cm = (torch.zeros(600 * 256, device="cuda") for _ in range(3))
    seen = set()
    for N, K in ((33, 8), (256, 64)):
        for ones in (0, 1):
            for M in range(1, 520):
                lda = max(M - 1, 1) if ones else K
                g = L.GemmArgs(gemm_mode=TC, n_agents=1, nnet=1, transA=ones, ones=ones, M=M, N=N, K=K, lda=lda,
                               ldb=N, ldc=N, A=A.data_ptr(), B=B.data_ptr(), C=Cm.data_ptr())
                rep = L.GemmRoute()
                L.check(lib.saceo_test_gemm_ex(C.byref(g), C.byref(rep), torch.cuda.current_stream().cuda_stream))
                if rep.n_tc:
                    assert rep.n_simt == 0 and M - rep.tc_rows <= 3 + ones, (M, N, ones, rep.tc_rows)
                    seen.add(M - rep.tc_rows)
    torch.cuda.synchronize()
    assert seen == {0, 1, 2, 3, 4}


# ---- chain level: depth-3 models through the per-layer GEMM chain at the same thresholds
WIDTHS = {"257-33-7": (257, 33, 7), "32-129-256": (32, 129, 256)}
ACTS3 = ("tanh", "elu", "tanh")
TANH_NETS = dict(actor_acts=("tanh", "tanh"), critic_acts=("tanh", "tanh"), actor_hidden=(64, 64), critic_hidden=(64, 64))


@pytest.mark.parametrize("engine", [SIMT, TC], ids=["fp32", "tc"])
@pytest.mark.parametrize("widths", WIDTHS)
@pytest.mark.parametrize("what", ["fit131", "fit144", "eval"])
def test_depth3_chain_at_dispatch_thresholds(monkeypatch, engine, widths, what):
    """Fit batches of 131 and 144 rows (3 and 16 rows past one 128-row tile) and model_eval on 1, 17 and 45 rows, for
    widths on both sides of the N <= 32 / N % 256 / K % 32 switches: ties the unit cases above to the activation strides
    and the workspace carving of the per-layer chain."""
    monkeypatch.setattr(O, "init_net", init_net_any_depth)
    cfg = NetCfg(S=11, A=3, model_hidden=WIDTHS[widths], model_acts=ACTS3, **TANH_NETS)
    if what.startswith("fit"):
        mb = int(what[3:])
        pop, probs = _setup(cfg, 2, mb, 600, seed=5, fit=dict(model_lr=1e-3, reward_loss_coef=0.7, delta_clip_loss=2.5),
                            gemm_mode=engine)
        w = _run(cfg, pop, probs, mb, steps=2, seed=9)
        assert w["grad"] < GRAD_TOL, w
        pop.close()
        return
    pop, probs = build(cfg, n_agents=2, B=32, E=20, N=200, seed=8, gemm_mode=engine)
    for rows in (1, 17, 45):
        obs = np.stack([p[1]["s"][:rows] for p in probs])
        act = np.stack([p[1]["a"][:rows] for p in probs])
        out = pop.model_eval(torch.from_numpy(obs), torch.from_numpy(act)).cpu().numpy()
        for i, p in enumerate(probs):
            st = to_torch_state(p[0], torch.float64)
            for k in range(2):
                ref = model_sample(cfg, st["m%d" % (k + 1)], torch.from_numpy(obs[i]).double(),
                                   torch.from_numpy(act[i]).double(), st).numpy()
                assert rel(out[i, k] - obs[i], ref - obs[i]) < GRAD_TOL, (rows, i, k)
    pop.close()
