"""CPU tests of the references the decoder kernels are checked against (tests/test_gpu_decoder.py): the numpy Philox4x32-10 and its
dropout masks (oracle/philox_ref.py), and the fp64 restatement of the decoder recurrence (oracle/torch_ref.decoder_states), pinned
to seq2seq.Seq2SeqDecoder's own CPU path, which test_seq2seq_cpu_path_matches_the_reference_golden pins to the reference."""
import numpy as np
import pytest
import torch

import seq2seq
from oracle import philox_ref as P
from oracle import torch_ref as R


# Random123's published known answers for philox4x32_10: (counter words, key words) -> output words
KAT = [((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
       ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
       ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
        (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1))]


@pytest.mark.parametrize("ctr,key,want", KAT)
def test_philox_known_answers(ctr, key, want):
    got = P.philox4x32_10_words([np.array([c]) for c in ctr], *key)[:, 0]
    assert [int(v) for v in got] == list(want)


def test_philox_64_bit_counter_and_key_split():
    """The library's form: counter c0 = low word, c1 = high word, c2 = c3 = 0; key k0 = low word of the seed, k1 = high word."""
    ctr, seed = 0x0123456789ABCDEF, 0xFEDCBA9876543210
    got = P.philox4x32_10(np.array([ctr], dtype=np.uint64), seed)[:, 0]
    want = P.philox4x32_10_words([np.array([ctr & 0xFFFFFFFF]), np.array([ctr >> 32]), np.array([0]), np.array([0])],
                                 seed & 0xFFFFFFFF, seed >> 32)[:, 0]
    assert np.array_equal(got, want)
    assert np.array_equal(P.philox4x32_10(np.array([0], dtype=np.uint64), 0)[:, 0], np.array(KAT[0][2], dtype=np.uint32))


def test_keep_thresholds():
    assert P.keep_threshold(0.0) == 0xFFFFFFFF and P.keep_threshold(0.5) == 1 << 31 and P.keep_threshold(0.75) == 1 << 30
    assert P.keep_threshold(0.1) == int((1.0 - float(np.float32(0.1))) * 2.0 ** 32)
    assert P.keep_threshold16(0.0) == 65536 and P.keep_threshold16(0.5) == 32768 and P.keep_threshold16(0.999999) == 1
    assert P.keep_threshold16(0.1) == int((1.0 - float(np.float32(0.1))) * 65536.0 + 0.5)
    assert P.keep_scale(0.1) == np.float32(1.0 / (1.0 - float(np.float32(0.1))))


def test_mask_definitions_element_by_element():
    """Spot-check each vectorised mask against its definition evaluated for one element at a time."""
    def words(ctr, seed):
        return [int(v) for v in P.philox4x32_10(np.array([ctr], dtype=np.uint64), seed)[:, 0]]
    p, seed = 0.25, 0x1234567890AB
    m = P.dropout_mask(4 * 9 + 3, p, seed)
    for e in (0, 5, 17, 38):
        assert m[e] == (P.keep_scale(p) if words(e // 4, seed)[e % 4] < P.keep_threshold(p) else 0)
    g = P.gru_mask(3, 13, p, seed)
    for b, t, col in ((0, 0, 0), (2, 12, 255), (1, 9, 77), (1, 7, 3)):
        w = words(((b * 256 + col) << 32) | (t >> 3), seed)[(t & 7) >> 1]
        assert g[b, t, col] == (P.keep_scale(p) if ((w >> (16 * (t & 1))) & 0xFFFF) < P.keep_threshold16(p) else 0)
    c = P.cell_mask(5, 100, p, seed, 7, seed_word=0xABCDEF)
    assert np.array_equal(c, P.cell_mask(5, 100, p, seed ^ 0xABCDEF, 7))
    for b, j in ((0, 0), (4, 99), (2, 51)):
        e = b * 100 + j
        assert c[b, j] == (P.keep_scale(p) if words((7 << 40) | (e >> 2), seed ^ 0xABCDEF)[e & 3] < P.keep_threshold(p) else 0)
    assert (P.cell_mask(5, 100, 0.0, seed, 7) == 1).all()
    keep = (P.cell_mask(64, 256, 0.5, seed, 3) > 0).mean()
    assert abs(keep - 0.5) < 4 * 0.5 / 128


@pytest.fixture
def float64_default():
    """Seq2SeqDecoder allocates its start symbol with the default dtype: run it in float64."""
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    yield
    torch.set_default_dtype(old)


class _FixedDropout(torch.nn.Module):
    """Stands in for the Dropout between the decoder cells: multiplies the u-th call's input by masks[u]."""

    def __init__(self, masks):
        super().__init__()
        self.masks, self.u = masks, 0

    def forward(self, x):
        self.u += 1
        return x * self.masks[self.u - 1]


def decoder_inputs(dec, enc, y):
    """The 13 inputs of DecoderStates as teacher_forced_log_likelihood derives them from a Seq2SeqDecoder and one-hot targets."""
    att, c0, c1 = dec.attention, dec.rnn.layers[0], dec.rnn.layers[2]
    D = c0.hidden_size
    B, U, S = y.shape
    sos = torch.zeros(B, 1, S, dtype=y.dtype)
    sos[:, 0, dec.SOS] = 1
    y_prev = torch.cat([sos, y[:, :-1]], 1).transpose(0, 1)
    ge_all = dec.embed(y_prev) @ c0.weight_ih[:, :D].t() + c0.bias_ih
    return (att.key_linear(enc), att.value_linear(enc), ge_all, dec.initial_state, att.query_linear.weight, att.query_linear.bias,
            c0.weight_ih[:, D:], c0.weight_hh, c0.bias_hh, c1.weight_ih, c1.bias_ih, c1.weight_hh, c1.bias_hh)


@pytest.mark.parametrize("B,T,U,p", [(1, 1, 1, 0.0), (3, 7, 5, 0.0), (4, 25, 6, 0.5), (2, 9, 3, 0.1)])
def test_decoder_states_restatement_matches_the_seq2seq_decoder(B, T, U, p, float64_default):
    """decoder_states + the output projection = Seq2SeqDecoder.forward in float64, eval mode (with the inter-cell Dropout
    replaced by the philox_ref masks when p > 0): every state after every symbol, per-example log p, and the gradient of log p
    for every decoder parameter."""
    torch.manual_seed(B * 100 + T)
    S = 23
    dec = seq2seq.Seq2SeqDecoder(S, 2, 128, 256, 100, 200).double().eval()
    enc = torch.randn(B, T, 256, dtype=torch.float64)
    y = torch.nn.functional.one_hot(torch.randint(0, S, (B, U)), S).double()
    masks = None
    if p > 0:
        masks = torch.from_numpy(np.stack([P.cell_mask(B, 256, p, 987654321, u) for u in range(U)])).double()
        dec.rnn.layers[1] = _FixedDropout(masks)
    state = dec.initial_state.unsqueeze(0).expand(B, -1, -1)
    y_prev = torch.zeros(B, S, dtype=torch.float64)
    y_prev[:, dec.SOS] = 1
    want = []
    for u in range(U):
        state, _ = dec._step(enc, y_prev, state)
        want.append(state[:, 1])
        y_prev = y[:, u]
    want = torch.stack(want)
    if p > 0:
        dec.rnn.layers[1].u = 0
    log_p = dec(enc, y)
    states = R.decoder_states(*decoder_inputs(dec, enc, y), masks)
    assert (states - want).abs().max().item() < 1e-12
    mine = (torch.log_softmax(states @ dec.linear.weight.t() + dec.linear.bias, -1) * y.transpose(0, 1)).sum((0, 2))
    assert (mine - log_p).abs().max().item() < 1e-10
    params = [q for q in dec.parameters()]
    g_ref = torch.autograd.grad(log_p.mean(), params)
    g_mine = torch.autograd.grad(mine.mean(), params, allow_unused=True)
    for (name, _), a, b in zip(dec.named_parameters(), g_mine, g_ref):
        assert a is not None, name
        assert (a - b).abs().max().item() <= 1e-10 * (1 + b.abs().max().item()), name
