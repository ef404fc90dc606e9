"""The seq2seq decoder's kernels (csrc/decoder.cu) and its hand-written backward through time (decoder.py DecoderStates) against
fp64, at the shapes where they could go wrong, on both sides of the 64-utterance switch: up to SKINNY_MAX_ROWS utterances the
per-symbol projections run on the exact-fp32 slu_skinny_gemm, beyond it on the tcgen05 slu_gemm_tc with pre-split weights.
The dropout masks are compared bit for bit with their definition (oracle/philox_ref.py), the recurrence with the fp64
restatement oracle/torch_ref.decoder_states (pinned to seq2seq.Seq2SeqDecoder by tests/test_decoder_reference_cpu.py).
Every test records the largest error it saw as a junit property (pytest --junitxml)."""
import copy
import importlib
import math

import numpy as np
import pytest
import torch

import seq2seq
from oracle import philox_ref as P
from oracle import torch_ref as R
from util import rel_err

pytestmark = pytest.mark.gpu
FWD_TOL, GRAD_TOL = 1e-4, 2e-3
SENT = -7777.0                       # sentinel in output padding: must survive every call
U32 = 2.0 ** -24                     # fp32 unit roundoff


@pytest.fixture(scope="module")
def pkg():
    p = importlib.import_module("end-to-end-slu_b200")
    p._lib.load()
    return p


def padded(rs, rows, cols, ld, fill=float("nan"), scale=1.0):
    """[rows, ld] fp32 CUDA buffer: random [rows, cols] block, `fill` in the padding columns (NaN: any read of it shows)."""
    buf = torch.full((rows, ld), fill, dtype=torch.float32)
    buf[:, :cols] = torch.from_numpy((scale * rs.standard_normal((rows, cols))).astype(np.float32))
    return buf.cuda()


def call(pkg, name, *args):
    pkg._lib.call(name, *args, pkg._lib.stream())


# ---- slu_skinny_gemm -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M", [1, 63, 64])
@pytest.mark.parametrize("form", ["nt", "nn"])
def test_skinny_gemm_against_fp64(pkg, form, M, record_property):
    """C[m][n] = sum_k A[m*lda + k] W[n*sn + k*sk] (+ bias[n]) in both operand forms of decoder._W: `nt` (x @ W^T, sk = 1: float4
    rows of W) and `nn` (g @ W, sn = 1: the transposed scalar path).  K = 4 / 100 / 128 / 132 / 456 / 868 cover a short chunk, a
    ragged last chunk of the 128-wide K loop and several chunks; N = 868 is the real wcat1.  A has lda > K and W padded rows
    (NaN in the gaps: a read of them would poison the result), C has ldc > N and one row past M, all sentinel-filled.
    Exact fp32: every element must be within the fp32 summation bound gamma_(K+1) * (sum |a w| + |b|) of fp64, and the max error
    over the tensor relative to its largest element within 3e-6 (the bf16x3 tcgen05 GEMM tests allow 2e-5).
    Measured on a B200 at 1000 W: largest relative error 2.1e-6 (M = N = 1, where a single output is the normaliser; the kernel
    is deterministic), largest error / summation bound 0.57."""
    rs = np.random.RandomState(100 * M + (form == "nn"))
    worst_rel = worst_bound = 0.0
    for N in (1, 7, 9, 200, 868):
        for K in (4, 100, 128, 132, 456, 868):
            lda = K + 8
            A = padded(rs, M, K, lda)
            if form == "nt":
                Wb = padded(rs, N, K, K + 4)                     # W [N][K], row pitch K + 4
                sn, sk, Wl = K + 4, 1, Wb[:, :K]
            else:
                Wb = padded(rs, K, N, N + 3)                     # W [K][N] read transposed, row pitch N + 3
                sn, sk, Wl = 1, N + 3, Wb[:, :N].t()
            a64, w64 = A[:, :K].double().cpu(), Wl.double().cpu()
            for with_bias in (False, True):
                bias = torch.from_numpy(rs.standard_normal(N).astype(np.float32)).cuda() if with_bias else None
                ldc = N + 5
                C = torch.full((M + 1, ldc), SENT, device="cuda")
                call(pkg, "slu_skinny_gemm", A.data_ptr(), lda, Wb.data_ptr(), sn, sk, pkg._lib.ptr(bias), C.data_ptr(), ldc, M, N, K)
                Cc = C.cpu()
                ref = a64 @ w64.t()
                mag = a64.abs() @ w64.abs().t()
                if with_bias:
                    ref = ref + bias.double().cpu()
                    mag = mag + bias.double().abs().cpu()
                err = (Cc[:M, :N].double() - ref).abs()
                gamma = (K + 1) * U32 / (1 - (K + 1) * U32)
                assert (err <= gamma * mag).all(), (N, K, with_bias, (err / (gamma * mag)).max().item())
                r = rel_err(Cc[:M, :N], ref)
                assert r < 3e-6, (N, K, with_bias, r)
                assert (Cc[:M, N:] == SENT).all() and (Cc[M:] == SENT).all(), (N, K, with_bias)
                worst_rel = max(worst_rel, r)
                worst_bound = max(worst_bound, (err / (gamma * mag).clamp_min(1e-30)).max().item())
    record_property("max_rel_err", worst_rel)
    record_property("max_err_over_bound", worst_bound)


def test_skinny_gemm_rejects_what_it_cannot_run(pkg):
    """M = 65, K % 4 != 0, an A that is not 16-byte aligned and sk == 1 with sn % 4 != 0 return the library's error (the Python
    binding raises naming the entry point) and write nothing."""
    A = torch.zeros(66, 136, device="cuda")
    W = torch.zeros(200, 136, device="cuda")
    C = torch.full((66, 200), SENT, device="cuda")
    call(pkg, "slu_skinny_gemm", A.data_ptr(), 136, W.data_ptr(), 136, 1, None, C.data_ptr(), 200, 64, 200, 128)
    torch.cuda.synchronize()
    assert (C[:64] == 0).all()
    C.fill_(SENT)
    bad = [(A.data_ptr(), 136, W.data_ptr(), 136, 1, 65, 200, 128),            # M > SK_M
           (A.data_ptr(), 136, W.data_ptr(), 136, 1, 64, 200, 126),            # K % 4 != 0
           (A.data_ptr() + 4, 136, W.data_ptr(), 136, 1, 64, 200, 128),        # A not 16-byte aligned
           (A.data_ptr(), 136, W.data_ptr(), 134, 1, 64, 200, 128)]            # sk == 1 with sn % 4 != 0
    for a, lda, w, sn, sk, M, N, K in bad:
        with pytest.raises(RuntimeError, match="slu_skinny_gemm"):
            call(pkg, "slu_skinny_gemm", a, lda, w, sn, sk, None, C.data_ptr(), 200, M, N, K)
    torch.cuda.synchronize()
    assert (C == SENT).all()


# ---- slu_attn_step_fwd / _bwd --------------------------------------------------------------------------------------------------
def attn_case(pkg, rs, q, keys, values, D=256, saturated=False):
    """Runs both attention kernels the way DecoderStates does (q and dq inside [B][3D+K] rows at column 3D, dkeys / dvalues
    accumulating into random prefills) and returns the errors against fp64 autograd of softmax(keys.q * inv_scale).values,
    relative to each tensor's largest element.  saturated: dq and dkeys are w_t (dctx.values_t - sum_s w_s dctx.values_s)
    times keys / q, which a saturated softmax cancels to ~1e-7 of its terms in any fp32 evaluation; their errors are then
    measured against the size of those terms, inv_scale * max|dctx.values_t| * max|keys| (dq) or max|q| (dkeys)."""
    B, T, K = keys.shape
    V = values.shape[2]
    ld = 3 * D + K
    inv = float(np.float32(1.0 / math.sqrt(K)))                  # the fp32 scale the kernels receive
    g = torch.full((B, ld), float("nan"))
    g[:, 3 * D:] = q
    g = g.cuda()
    kd, vd = keys.cuda(), values.cuda()
    w = torch.full((B * T + 4,), SENT, device="cuda")
    ctx = torch.full((B * V + 4,), SENT, device="cuda")
    call(pkg, "slu_attn_step_fwd", g.data_ptr() + 4 * 3 * D, ld, kd.data_ptr(), vd.data_ptr(), B, T, K, V, inv, w.data_ptr(), ctx.data_ptr())
    q64, k64, v64 = (t.double().requires_grad_(True) for t in (q, keys, values))
    w64 = torch.softmax((k64 @ q64.unsqueeze(2)).squeeze(2) * inv, dim=1)
    c64 = (w64.unsqueeze(1) @ v64).squeeze(1)
    dctx = torch.from_numpy(rs.standard_normal((B, V)).astype(np.float32))
    (c64 * dctx.double()).sum().backward()
    prefill = lambda g: torch.from_numpy(rs.standard_normal(tuple(g.shape)).astype(np.float32)) * (g.abs().max().item() or 1.0)
    pk, pv = prefill(k64.grad), prefill(v64.grad)
    dk, dv = pk.cuda(), pv.cuda()
    dq = torch.full((B, ld), SENT, device="cuda")
    dcd = dctx.cuda()
    call(pkg, "slu_attn_step_bwd", dcd.data_ptr(), w.data_ptr(), g.data_ptr() + 4 * 3 * D, ld, kd.data_ptr(), vd.data_ptr(), B, T, K, V, inv,
         dq.data_ptr() + 4 * 3 * D, ld, dk.data_ptr(), dv.data_ptr())
    torch.cuda.synchronize()
    w, ctx, dq, dk, dv = w.cpu(), ctx.cpu(), dq.cpu(), dk.cpu(), dv.cpu()
    assert (w[B * T:] == SENT).all() and (ctx[B * V:] == SENT).all() and (dq[:, :3 * D] == SENT).all()
    if saturated:
        dsw = (values.double() @ dctx.double().unsqueeze(2)).abs().max().item() * inv
        return {"w": rel_err(w[:B * T].view(B, T), w64), "ctx": rel_err(ctx[:B * V].view(B, V), c64),
                "dq": (dq[:, 3 * D:].double() - q64.grad).abs().max().item() / (dsw * keys.abs().max().item()),
                "dkeys": (dk.double() - pk.double() - k64.grad).abs().max().item() / (dsw * q.abs().max().item()),
                "dvalues": rel_err(dv.double() - pv.double(), v64.grad)}
    return {"w": rel_err(w[:B * T].view(B, T), w64), "ctx": rel_err(ctx[:B * V].view(B, V), c64),
            "dq": rel_err(dq[:, 3 * D:], q64.grad),
            "dkeys": rel_err(dk.double() - pk.double(), k64.grad) if k64.grad.abs().max() > 0 else (dk - pk).abs().max().item(),
            "dvalues": rel_err(dv.double() - pv.double(), v64.grad)}


@pytest.mark.parametrize("B", [1, 130])
@pytest.mark.parametrize("K,V", [(4, 4), (100, 200), (512, 512)])
@pytest.mark.parametrize("T", [1, 7, 25, 94, 255, 256])
def test_attn_step_against_fp64(pkg, T, K, V, B, record_property):
    """One CTA per utterance: T < 8 leaves warps without a frame, 25 / 94 frames are 4 s / 15 s of audio, 256 = ATT_MAXT;
    K = V = 512 is the largest width.  Forward weights and context, backward dq and the accumulated dkeys / dvalues (checked as
    prefill + this step's contribution) within 1e-5 of fp64 relative to each tensor's largest element.
    Measured on a B200 at 1000 W: largest error 7.7e-7 (ctx at T = 255, K = V = 4, B = 130); dq 7.5e-7, w 3.8e-7, dkeys 3.7e-7,
    dvalues 3.4e-7."""
    rs = np.random.RandomState(T * 1000 + K + B)
    q = torch.from_numpy(rs.standard_normal((B, K)).astype(np.float32))
    keys = torch.from_numpy(rs.standard_normal((B, T, K)).astype(np.float32))
    values = torch.from_numpy(rs.standard_normal((B, T, V)).astype(np.float32))
    errs = attn_case(pkg, rs, q, keys, values)
    for k, e in errs.items():
        record_property(k, e)
    assert all(e < 1e-5 for e in errs.values()), errs


@pytest.mark.parametrize("kind", ["scores_1e3", "near_one_hot"])
def test_attn_step_extreme_scores(pkg, kind, record_property):
    """Scores of magnitude ~1e3 (a softmax without the max subtraction overflows expf to inf and returns NaN; keys and q are small
    integers and K = 4, so the scores are exact in fp32 and the reference sees the same ones), and keys in which one frame
    scores 20 above all others, so the softmax puts all but ~1e-7 of the weight on it (dq and dkeys measured
    against the size of the terms the saturated softmax cancels, see attn_case).  Same 1e-5 bound as the regular shapes.
    Measured on a B200 at 1000 W: scores_1e3 1.2e-6 (dq), forward 9.3e-8; near_one_hot 1.2e-7 (dvalues),
    dq / dkeys 2.5e-9 of the cancelled terms."""
    rs = np.random.RandomState(7 if kind == "scores_1e3" else 8)
    B, T = 3, 94
    if kind == "scores_1e3":
        K, V = 4, 200
        q = torch.from_numpy(rs.randint(-5, 6, size=(B, K)).astype(np.float32))
        q[:, 0] = 50.0
        keys = torch.from_numpy(rs.randint(-5, 6, size=(B, T, K)).astype(np.float32))
        keys[:, :, 0] += 40.0                                       # scores = 0.5 * (50 * (35..45) + small) ~ 1e3
    else:
        K, V = 100, 200
        q = torch.from_numpy((3 * rs.standard_normal((B, K))).astype(np.float32))
        keys = torch.from_numpy(rs.standard_normal((B, T, K)).astype(np.float32))
        s = (keys @ q.unsqueeze(2)).squeeze(2) / math.sqrt(K)
        hot = torch.from_numpy(rs.randint(0, T, B))
        for b in range(B):                                          # frame hot[b] scores 20 above the best of the others
            keys[b, hot[b]] += q[b] * float((s[b].max() + 20 - s[b, hot[b]]) * math.sqrt(K) / q[b].square().sum())
    values = torch.from_numpy(rs.standard_normal((B, T, V)).astype(np.float32))
    errs = attn_case(pkg, rs, q, keys, values, saturated=kind == "near_one_hot")
    for k, e in errs.items():
        record_property(k, e)
    assert all(e < 1e-5 for e in errs.values()), errs
    if kind == "near_one_hot":
        inv = 1.0 / math.sqrt(K)
        wmax = torch.softmax((keys.double() @ q.double().unsqueeze(2)).squeeze(2) * inv, 1).max(1)[0]
        assert (wmax > 0.999).all(), wmax


def test_attn_step_rejects_out_of_range_sizes(pkg):
    """T = 257 (> ATT_MAXT), K = 513 and V = 513 (> the 512-float shared-memory rows) return the library's error."""
    for T, K, V in ((257, 4, 4), (4, 513, 4), (4, 4, 513)):
        q = torch.zeros(2, K, device="cuda"); keys = torch.zeros(2, T, K, device="cuda"); values = torch.zeros(2, T, V, device="cuda")
        w = torch.zeros(2, T, device="cuda"); ctx = torch.zeros(2, V, device="cuda"); dq = torch.zeros(2, K, device="cuda")
        with pytest.raises(RuntimeError, match="slu_attn_step_fwd"):
            call(pkg, "slu_attn_step_fwd", q.data_ptr(), K, keys.data_ptr(), values.data_ptr(), 2, T, K, V, 1.0, w.data_ptr(), ctx.data_ptr())
        with pytest.raises(RuntimeError, match="slu_attn_step_bwd"):
            call(pkg, "slu_attn_step_bwd", ctx.data_ptr(), w.data_ptr(), q.data_ptr(), K, keys.data_ptr(), values.data_ptr(), 2, T, K, V, 1.0,
                 dq.data_ptr(), K, keys.data_ptr(), values.data_ptr())


# ---- slu_grucell_fwd / _bwd ----------------------------------------------------------------------------------------------------
def grucell_ref(gi, gh, hp):
    """torch.nn.GRUCell's gate math in fp64 on precomputed gi / gh (biases included) -> h, (r, z, n, gh_n)."""
    D = hp.shape[1]
    r = torch.sigmoid(gi[:, :D] + gh[:, :D])
    z = torch.sigmoid(gi[:, D:2 * D] + gh[:, D:2 * D])
    n = torch.tanh(gi[:, 2 * D:] + r * gh[:, 2 * D:])
    return (1 - z) * n + z * hp, (r, z, n, gh[:, 2 * D:])


@pytest.mark.parametrize("sat", [False, True])
@pytest.mark.parametrize("B,D", [(3, 100), (67, 100), (5, 256), (130, 256)])
def test_grucell_against_fp64(pkg, B, D, sat, record_property):
    """Strided gi_a / gi_b / gh (lda, ldb, ldh > 3D, NaN in the gaps), with and without gi_b, hprev against the broadcast row h0,
    B*D not a multiple of the 256-thread block (except 130 x 256), dropout off / p = 0.5 / p = 0.1 at several steps / a device seed
    word; backward with every combination of NULL db / dc into dgi [B][3D+4] and dgh [B][3D+K] (K = 100: the dq columns of
    DecoderStates' g1 rows, which must stay untouched).  sat: pre-activations up to |x| = 100, where sigmoid / tanh saturate
    and the results must stay finite.  h and the stash r | z | n | gh_n within 1e-5 of fp64, dgi / dgh / dh_direct within 1e-5
    relative to their largest element; `dropped` = h * philox_ref mask bit for bit.
    Measured on a B200 at 1000 W: forward 2.0e-7 / backward 1.8e-7 at most with ordinary inputs, 3.3e-6 / 4.0e-6 with
    saturating ones (B = 130, D = 256)."""
    rs = np.random.RandomState(B * 1000 + D + sat)
    G = 3 * D
    lda, ldb, ldh, ldgi, ldgh = G + 4, G + 8, G + 100, G + 4, G + 100

    def act(rows, cols, ld):
        buf = padded(rs, rows, cols, ld)
        if sat:
            buf[:, :cols] *= torch.from_numpy(10.0 ** rs.uniform(-1, 2, size=(rows, cols)).astype(np.float32)).cuda()
        return buf
    gi_a, gi_b, gh = act(B, G, lda), act(B, G, ldb), act(B, G, ldh)
    hprev = torch.from_numpy(rs.uniform(-1, 1, (B, D)).astype(np.float32)).cuda()
    h0 = torch.from_numpy(rs.uniform(-1, 1, D).astype(np.float32)).cuda()
    word = torch.tensor([0x0F1E2D3C4B5A6978], dtype=torch.int64, device="cuda")
    seed = 0x9E3779B97F4A7C15
    worst_f = worst_b = 0.0
    for use_b in (False, True):
        for use_hprev in (True, False):
            gi64 = gi_a[:, :G].double().cpu() + (gi_b[:, :G].double().cpu() if use_b else 0)
            gh64 = gh[:, :G].double().cpu()
            hp64 = (hprev if use_hprev else h0.expand(B, D)).double().cpu()
            for p, step, dev_word in ((0.0, 0, False), (0.5, 3, False), (0.1, 17, False), (0.5, 5, True)):
                h = torch.full((B, D), SENT, device="cuda"); stash = torch.full((B, 4 * D), SENT, device="cuda")
                dropped = torch.full((B, D), SENT, device="cuda")
                args = (gi_a.data_ptr(), lda, gi_b.data_ptr() if use_b else None, ldb, gh.data_ptr(), ldh,
                        hprev.data_ptr() if use_hprev else None, h0.data_ptr(), B, D, p, seed)
                call(pkg, "slu_grucell_fwd", *args, word.data_ptr() if dev_word else None, step, h.data_ptr(), stash.data_ptr(), dropped.data_ptr())
                mask = torch.from_numpy(P.cell_mask(B, D, p, seed, step, int(word.item()) & (2 ** 64 - 1) if dev_word else None)).cuda()
                assert torch.equal(dropped, h * mask), (use_b, use_hprev, p, step, dev_word)
                if dev_word:                                    # device word w == seed ^ w given on the host
                    d2 = torch.full((B, D), SENT, device="cuda")
                    call(pkg, "slu_grucell_fwd", *args[:-1], seed ^ (int(word.item()) & (2 ** 64 - 1)), None, step, h.data_ptr(), stash.data_ptr(),
                         d2.data_ptr())
                    assert torch.equal(d2, dropped)
                h64, (r, z, n, hn) = grucell_ref(gi64, gh64, hp64)
                hc, sc = h.cpu(), stash.cpu()
                assert torch.isfinite(hc).all() and torch.isfinite(sc).all()
                ef = max((hc.double() - h64).abs().max().item(),
                         max((sc[:, i * D:(i + 1) * D].double() - ref).abs().max().item() for i, ref in enumerate((r, z, n))),
                         rel_err(sc[:, 3 * D:], hn))
                assert ef < 1e-5, (use_b, use_hprev, p, ef)
                worst_f = max(worst_f, ef)
                for use_db in (False, True):
                    for use_dc in (False, True):
                        da, db, dc = (torch.from_numpy(rs.standard_normal((B, D)).astype(np.float32)).cuda() for _ in range(3))
                        dgi = torch.full((B, ldgi), SENT, device="cuda"); dgh = torch.full((B, ldgh), SENT, device="cuda")
                        dhd = torch.full((B, D), SENT, device="cuda")
                        call(pkg, "slu_grucell_bwd", da.data_ptr(), db.data_ptr() if use_db else None, dc.data_ptr() if use_dc else None,
                             stash.data_ptr(), hprev.data_ptr() if use_hprev else None, h0.data_ptr(), B, D, p, seed,
                             word.data_ptr() if dev_word else None, step, dgi.data_ptr(), ldgi, dgh.data_ptr(), ldgh, dhd.data_ptr())
                        dh = (da * mask).double().cpu() + (db.double().cpu() if use_db else 0) + (dc.double().cpu() if use_dc else 0)
                        gi_, gh_, hp_ = (t.clone().requires_grad_(True) for t in (gi64, gh64, hp64))
                        gref = torch.autograd.grad(grucell_ref(gi_, gh_, hp_)[0], (gi_, gh_, hp_), dh)
                        dgi_c, dgh_c, dhd_c = dgi.cpu(), dgh.cpu(), dhd.cpu()
                        assert (dgi_c[:, G:] == SENT).all() and (dgh_c[:, G:] == SENT).all()
                        assert torch.isfinite(dgi_c).all() and torch.isfinite(dgh_c).all() and torch.isfinite(dhd_c).all()
                        eb = max(rel_err(dgi_c[:, :G], gref[0]), rel_err(dgh_c[:, :G], gref[1]), rel_err(dhd_c, gref[2]))
                        assert eb < 1e-5, (use_b, use_hprev, p, step, dev_word, use_db, use_dc, eb)
                        worst_b = max(worst_b, eb)
    record_property("max_fwd_err", worst_f)
    record_property("max_bwd_rel_err", worst_b)


# ---- mask generators -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("p", [0.1, 0.25, 0.5, 0.9])
def test_dropout_mask_generators_are_bit_exact(pkg, p):
    """slu_dropout_mask (n % 4 != 0: a partial last float4 group) and slu_dropout_mask_gru (T % 8 != 0: a partial last group of
    eight 16-bit draws) equal philox_ref's masks bit for bit -- the contract the GRU backward kernels rely on when they
    regenerate the forward's mask from (p, seed)."""
    seed = 0xC0FFEE1234567891
    for n in (7, 1001, 65537):
        buf = torch.full((n + 4,), SENT, device="cuda")
        call(pkg, "slu_dropout_mask", buf.data_ptr(), n, p, seed)
        got = buf.cpu().numpy()
        assert np.array_equal(got[:n], P.dropout_mask(n, p, seed)), n
        assert (got[n:] == SENT).all()
    for B, T in ((3, 13), (2, 1), (5, 94)):
        m = torch.empty(B, T, 256, device="cuda")
        call(pkg, "slu_dropout_mask_gru", m.data_ptr(), B, T, p, seed)
        assert np.array_equal(m.cpu().numpy(), P.gru_mask(B, T, p, seed)), (B, T)


# ---- DecoderStates end to end --------------------------------------------------------------------------------------------------
NAMES = ("keys", "values", "ge_all", "init_state", "wq", "bq", "w_c", "w_hh0", "b_hh0", "w_ih1", "b_ih1", "w_hh1", "b_hh1")


def states_inputs(rs, B, T, U, D, K, V):
    """The 13 inputs of DecoderStates at the magnitudes of the model (PyTorch's default init of the decoder's layers)."""
    u = lambda *s: torch.from_numpy(rs.uniform(-1, 1, s).astype(np.float32) / math.sqrt(D))
    n = lambda *s: torch.from_numpy((0.5 * rs.standard_normal(s)).astype(np.float32))
    return [n(B, T, K), n(B, T, V), n(U, B, 3 * D), n(2, D), u(K, D), u(K), u(3 * D, V), u(3 * D, D), u(3 * D), u(3 * D, D), u(3 * D),
            u(3 * D, D), u(3 * D)]


def check_states(pkg, inputs, gy, p, seed, record_property=None, tag=""):
    """DecoderStates forward + backward on the GPU against autograd of torch_ref.decoder_states in fp64 with philox_ref's masks."""
    U, B, D = gy.shape
    leaves = [t.cuda().requires_grad_(True) for t in inputs]
    out = pkg.decoder.DecoderStates.apply(*leaves, p, seed, None)
    out.backward(gy.cuda())
    ref_leaves = [t.double().requires_grad_(True) for t in inputs]
    masks = None
    if p > 0:
        masks = torch.from_numpy(np.stack([P.cell_mask(B, D, p, seed, u) for u in range(U)])).double()
    ref = R.decoder_states(*ref_leaves, masks)
    ref.backward(gy.double())
    errs = {"states": rel_err(out.detach().cpu(), ref.detach())}
    errs.update({"d" + k: rel_err(a.grad.cpu(), b.grad) for k, a, b in zip(NAMES, leaves, ref_leaves)})
    if record_property is not None:
        for k, e in errs.items():
            record_property(tag + k, e)
    assert errs["states"] < FWD_TOL, errs
    bad = {k: e for k, e in errs.items() if k != "states" and not e < GRAD_TOL}
    assert not bad, (bad, errs)
    return out.detach()


@pytest.mark.parametrize("p", [0.0, 0.5])
@pytest.mark.parametrize("B,T,U,D,K,V", [(1, 1, 1, 256, 100, 200), (3, 25, 7, 256, 100, 200), (64, 25, 40, 256, 100, 200),
                                         (65, 25, 12, 256, 100, 200), (130, 94, 5, 256, 100, 200),
                                         (5, 25, 6, 128, 36, 52), (65, 25, 6, 128, 36, 52)])
def test_decoder_states_against_fp64(pkg, B, T, U, D, K, V, p, record_property):
    """The forward states and the gradients of all 13 inputs under a random upstream gradient on every state, through the
    hand-written backward through time (ping-pong dh buffers, the four slu_wgrad_tc reductions over all (symbol, utterance) rows,
    slu_colsum_acc for the biases and the initial state), against fp64 autograd; p = 0.5 with the philox_ref mask of the seed.
    (64, 25, 40) is the benchmark's shape (config 5), B = 64 the last batch on the skinny kernel, B >= 65 the tcgen05 path.
    Measured on a B200 at 1000 W: states 3.1e-7 / gradients 1.4e-5 at most up to B = 64 (the largest at B = 1, dw_ih1),
    states 3.6e-6 / gradients 9.5e-6 at B >= 65."""
    rs = np.random.RandomState(B * 10000 + T * 100 + U + D)
    inputs = states_inputs(rs, B, T, U, D, K, V)
    gy = torch.from_numpy(rs.standard_normal((U, B, D)).astype(np.float32))
    check_states(pkg, inputs, gy, p, 0x5EED0000 + B, record_property)


@pytest.mark.parametrize("p", [0.0, 0.5])
def test_decoder_states_on_both_sides_of_the_skinny_limit(pkg, p, record_property):
    """The same first 64 utterances run once as a batch of 64 (slu_skinny_gemm) and once inside a batch of 65 (slu_gemm_tc); each
    must match fp64 on its own, and the 64 shared rows agree between the two runs within the forward tolerance.
    Measured on a B200 at 1000 W: B = 64 states 2.4e-7 / gradients 5.2e-6, B = 65 states 2.9e-6 / gradients 7.5e-6."""
    rs = np.random.RandomState(6465)
    D, K, V, T, U = 256, 100, 200, 25, 12
    inputs = states_inputs(rs, 65, T, U, D, K, V)
    gy = torch.from_numpy(rs.standard_normal((U, 65, D)).astype(np.float32))
    first = [t[:64] if i < 2 else (t[:, :64] if i == 2 else t) for i, t in enumerate(inputs)]
    s64 = check_states(pkg, first, gy[:, :64].contiguous(), p, 77, record_property, "b64_")
    s65 = check_states(pkg, inputs, gy, p, 77, record_property, "b65_")
    assert rel_err(s65[:, :64].cpu(), s64.cpu()) < FWD_TOL


# ---- the model surface ---------------------------------------------------------------------------------------------------------
S_LABELS = 23                        # not a multiple of 4: the embedding's operand padding is exercised


def decoders(seed):
    """(fp64 CPU decoder in eval mode, the same weights as an fp32 CUDA decoder)."""
    torch.manual_seed(seed)
    dec64 = seq2seq.Seq2SeqDecoder(S_LABELS, 2, 128, 256, 100, 200).double().eval()
    return dec64, copy.deepcopy(dec64).float().cuda().eval()


class float64_default:
    """Seq2SeqDecoder's CPU path allocates with the default dtype."""

    def __enter__(self):
        self.old = torch.get_default_dtype()
        torch.set_default_dtype(torch.float64)

    def __exit__(self, *a):
        torch.set_default_dtype(self.old)


@pytest.mark.parametrize("B", [64, 65, 130])
def test_teacher_forced_log_likelihood_matches_the_cpu_decoder(pkg, B, record_property):
    """Seq2SeqDecoder.forward on CUDA (decoder.teacher_forced_log_likelihood) against the same module's CPU path in fp64, eval
    mode: per-example log p element by element, and the gradient of log_p.mean() for every decoder parameter and the encoder
    states.  Measured on a B200 at 1000 W: log p 2.6e-7, gradients 1.1e-5 at most (key weight, B = 65), key bias 1.5e-7 of the key
    weight's gradient."""
    dec64, dec = decoders(B)
    rs = np.random.RandomState(B)
    T, U = 25, 9
    enc = torch.from_numpy((0.5 * rs.standard_normal((B, T, 256))).astype(np.float32))
    y = torch.nn.functional.one_hot(torch.from_numpy(rs.randint(0, S_LABELS, (B, U))), S_LABELS).float()
    enc_c = enc.cuda().requires_grad_(True)
    log_p = dec(enc_c, y.cuda())
    log_p.mean().backward()
    enc64 = enc.double().requires_grad_(True)
    with float64_default():
        ref = dec64(enc64, y.double())
        ref.mean().backward()
    errs = {"log_p": rel_err(log_p.detach().cpu(), ref.detach()), "d_encoder_outputs": rel_err(enc_c.grad.cpu(), enc64.grad)}
    for (k, a), b in zip(dec.named_parameters(), dec64.parameters()):
        errs["d" + k] = rel_err(a.grad.cpu(), b.grad)
    # The key bias adds q.b_k to every score of an utterance, which the softmax ignores: its gradient is zero in exact arithmetic
    # and what both sides return is the rounding of a sum of dkeys rows.  Measure it against the key weight's gradient, which
    # sums the same rows times the encoder states.
    kb = dec.attention.key_linear.bias.grad.cpu().double() - dec64.attention.key_linear.bias.grad
    errs["dattention.key_linear.bias"] = kb.abs().max().item() / dec64.attention.key_linear.weight.grad.abs().max().item()
    for k, e in errs.items():
        record_property(k, e)
    assert errs["log_p"] < FWD_TOL, errs
    bad = {k: e for k, e in errs.items() if k != "log_p" and not e < GRAD_TOL}
    assert not bad, (bad, errs)


@pytest.mark.parametrize("B", [1, 64, 65, 200])
def test_beam_step_matches_the_cpu_step(pkg, B, record_property):
    """decoder.beam_step (one beam-search step on the library's kernels) against Seq2SeqDecoder._step in fp64: new state and
    log-probabilities; the first rows feed the all-zero previous symbol of infer's first step.
    Measured on a B200 at 1000 W: state 4.7e-7 / log-probabilities 1.2e-7 at B <= 64, 3.2e-6 / 7.8e-7 at B >= 65."""
    dec64, dec = decoders(1000 + B)
    rs = np.random.RandomState(1000 + B)
    T = 25
    enc = torch.from_numpy((0.5 * rs.standard_normal((B, T, 256))).astype(np.float32))
    y_prev = torch.nn.functional.one_hot(torch.from_numpy(rs.randint(0, S_LABELS, B)), S_LABELS).float()
    y_prev[: max(1, B // 4)] = 0
    state = torch.from_numpy(rs.uniform(-1, 1, (B, 2, 256)).astype(np.float32))
    with torch.no_grad():
        cache = pkg.decoder.StepCache(dec, enc.cuda())
        st, lp = dec._step(enc.cuda(), y_prev.cuda(), state.cuda(), cache)
        with float64_default():
            st64, lp64 = dec64._step(enc.double(), y_prev.double(), state.double())
    e_state, e_logp = rel_err(st.cpu(), st64), rel_err(lp.cpu(), lp64)
    record_property("state", e_state)
    record_property("log_probs", e_logp)
    assert e_state < FWD_TOL and e_logp < FWD_TOL, (e_state, e_logp)


def test_infer_at_batch_65_matches_the_cpu_beam_search(pkg, record_property):
    """Seq2SeqDecoder.infer over 65 utterances (every step on the tcgen05 projections) against the CPU beam search in fp64: the
    beam scores, and the best hypothesis wherever the reference's top two scores are further apart than the tolerance.
    Measured on a B200 at 1000 W: scores 4.6e-7."""
    dec64, dec = decoders(65)
    rs = np.random.RandomState(65)
    enc = torch.from_numpy((0.5 * rs.standard_normal((65, 25, 256))).astype(np.float32))
    Sy = [str(i) for i in range(S_LABELS)]
    scores, beam = dec.infer(enc.cuda(), Sy, B=4, y_lengths=[6])
    with float64_default():
        scores64, beam64 = dec64.infer(enc.double(), Sy, B=4, y_lengths=[6])
    e = rel_err(scores.cpu(), scores64)
    record_property("scores", e)
    assert e < FWD_TOL, e
    tol = FWD_TOL * scores64.abs().max().item()
    sep = (scores64[0] - scores64[1]) > tol
    assert sep.sum().item() > 32
    ids, ids64 = beam.argmax(-1)[0].cpu(), beam64.argmax(-1)[0]
    assert torch.equal(ids[sep], ids64[sep])
