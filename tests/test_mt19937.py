"""torch's CPU Mersenne Twister without a GPU: the characteristic polynomial re-derived by Berlekamp-Massey, the host jump
against numpy's sequential MT19937 (an independent implementation of the same generator), torch-state packing through
set_rng_state, the device generator through the DEBUG emulator, the C entries' argument checks, and TrainStage.draw with
torch_generator=True against per-sample torch.rand calls."""
import ctypes as C
import shutil

import numpy as np
import pytest
import torch

N_STATE = 624


def _np_gen(seed, skip=0):
    g = np.random.MT19937(0)
    g._legacy_seeding(seed)                  # torch.manual_seed(seed) and numpy's legacy seeding give the same state
    if skip:
        g.random_raw(skip)
    return g


def _torch_view(g, fresh):
    """(words, next, left) of numpy generator g in torch's layout."""
    s = g.state["state"]
    pos = int(s["pos"])
    if fresh:
        return s["key"].astype(np.uint32), 0, 1
    return s["key"].astype(np.uint32), pos, (1 if pos == N_STATE else N_STATE + 1 - pos)


def _np_from(words, next_, left):
    g = np.random.MT19937(0)
    st = g.state
    st["state"]["key"] = np.asarray(words, dtype=np.uint32)
    st["state"]["pos"] = N_STATE if left == 1 else next_
    g.state = st
    return g


def _f32(raw):
    return ((np.asarray(raw, dtype=np.uint64) & 0xFFFFFF).astype(np.float64) * 2.0 ** -24).astype(np.float32)


@pytest.fixture(scope="module")
def L():
    if shutil.which("g++") is None:
        pytest.skip("needs g++ for the emulator build")
    from cuemu import emu
    return emu.lib()


def _advance(L, words, next_, left, n):
    from cuemu import emu
    st = np.ascontiguousarray(words, dtype=np.uint32).copy()
    nx, lf = C.c_int32(next_), C.c_int32(left)
    poly = None
    if n >= 625:
        poly = np.zeros(N_STATE, dtype=np.uint32)
        assert L.mvtb_mt19937_jump_poly(n - 625, emu.ptr(poly)) == 0
    rc = L.mvtb_mt19937_advance(emu.ptr(poly), n, emu.ptr(st), C.byref(nx), C.byref(lf))
    return rc, st, nx.value, lf.value


def test_phi_is_the_minimal_polynomial_of_the_output_bits(L):
    from cuemu import emu
    bits = _np_gen(12345).random_raw(2 * 19937) & 1
    c, b, length, m, window = 1, 1, 0, 1, 0           # Berlekamp-Massey over GF(2), polynomials as Python ints
    for n, s in enumerate(bits):
        window = (window << 1) | int(s)
        if (c & window).bit_count() & 1:
            t = c
            c ^= b << m
            if 2 * length <= n:
                length, b, m = n + 1 - length, t, 1
                continue
        m += 1
    assert length == 19937
    phi = {length - i for i in range(length + 1) if (c >> i) & 1}
    assert len(phi) == 135
    low = np.zeros(N_STATE, dtype=np.uint32)       # t^19937 mod phi = phi - t^19937
    assert L.mvtb_mt19937_jump_poly(19937, emu.ptr(low)) == 0
    got = set(np.nonzero(np.unpackbits(low.view(np.uint8), bitorder="little"))[0].tolist())
    assert got == phi - {19937}


@pytest.mark.parametrize("n", [0, 1, 623, 624, 625, 19937, 10 ** 6 + 3, 10 ** 8])
@pytest.mark.parametrize("skip", [0, 1, 300, 623, 624, 1000])
def test_host_jump_equals_sequential_draws(L, n, skip):
    g = _np_gen(7 + skip, skip)
    words, nx, lf = _torch_view(g, fresh=skip == 0)
    rc, st, nx2, lf2 = _advance(L, words, nx, lf, n)
    assert rc == 0
    if n:
        g.random_raw(n)
    want_words, want_next, want_left = _torch_view(g, fresh=skip == 0 and n == 0)
    assert (nx2, lf2) == (want_next, want_left)
    assert np.array_equal(st, want_words)
    assert np.array_equal(_np_from(st, nx2, lf2).random_raw(700), g.random_raw(700))


def test_torch_state_roundtrip_continues_torch_rand(L, monkeypatch):
    from mvtb import _lib, functional as Fn
    monkeypatch.setattr(_lib, "_lib", L)
    for seed, pre, n in ((3, 0, 10 ** 6 + 3), (4, 17, 625), (5, 624, 5), (6, 1000, 0)):
        torch.manual_seed(seed)
        if pre:
            torch.rand(pre)
        st = torch.get_rng_state()
        words, nx, lf = Fn.mt19937_unpack(st)
        assert torch.equal(Fn.mt19937_pack(words, nx, lf, st), st)
        words, nx, lf = Fn.mt19937_advance(words, nx, lf, n)
        torch.rand(n)
        want = torch.get_rng_state()
        assert torch.equal(Fn.mt19937_pack(words, nx, lf, st), want)
        want_next = torch.rand(1000)
        torch.set_rng_state(Fn.mt19937_pack(words, nx, lf, st))
        assert torch.equal(torch.rand(1000), want_next)


def test_take_leaves_the_generator_where_torch_rand_does(L, monkeypatch):
    from mvtb import _lib, functional as Fn
    monkeypatch.setattr(_lib, "_lib", L)
    torch.manual_seed(21)
    rows = Fn.mt19937_take(1234, 3)
    after = torch.get_rng_state()
    torch.manual_seed(21)
    for s in range(3):
        words, nx, lf = Fn.mt19937_unpack(torch.get_rng_state())
        assert np.array_equal(rows[s, :N_STATE].view(np.uint32), words) and (rows[s, 624], rows[s, 625]) == (nx, lf)
        torch.rand(1234)
    assert torch.equal(torch.get_rng_state(), after)


@pytest.mark.parametrize("n,chunk,n_chunks,segments", [
    (5000, 1253, 2, 3),         # 4 chunks a segment: two rounds, chunks and rounds not multiples of 624
    (7001, 700, 3, 2),          # 11 chunks: four rounds, the last one partial
    (300, 624, 4, 4),           # shorter than one chunk
    (2 * 624, 624, 1, 1),       # one chunk a round
])
def test_emulated_device_generator_equals_sequential_draws(L, n, chunk, n_chunks, segments):
    from cuemu import emu
    table = np.zeros((n_chunks, N_STATE), dtype=np.uint32)
    assert L.mvtb_mt19937_chunk_table(chunk, n_chunks, emu.ptr(table)) == 0
    states = np.zeros((segments, 640), dtype=np.uint32)
    want = []
    for s in range(segments):
        skip = [0, 5, 624, 311][s % 4]
        g = _np_gen(40 + s, skip)
        words, nx, lf = _torch_view(g, fresh=skip == 0)
        states[s, :N_STATE], states[s, 624], states[s, 625] = words, nx, lf
        want.append(_f32(g.random_raw(n)))
    u = np.full((segments, n), -1.0, dtype=np.float32)
    ws = np.zeros(L.mvtb_mt19937_workspace_bytes(segments) // 4, dtype=np.uint32)
    assert L.mvtb_mt19937_uniform_f32(emu.ptr(u), n, segments, emu.ptr(states), emu.ptr(table), chunk, n_chunks,
                                      emu.ptr(ws), None) == 0
    for s in range(segments):
        assert np.array_equal(u[s], want[s]), s


def test_chunk_table_entries_are_powers_of_t(L):
    from cuemu import emu
    table = np.zeros((3, N_STATE), dtype=np.uint32)
    assert L.mvtb_mt19937_chunk_table(30000, 3, emu.ptr(table)) == 0
    for c in range(3):
        p = np.zeros(N_STATE, dtype=np.uint32)
        assert L.mvtb_mt19937_jump_poly(30000 * c, emu.ptr(p)) == 0
        assert np.array_equal(table[c], p)


def test_argument_checks(L):
    from cuemu import emu
    from mvtb import _lib
    words = _np_gen(1).state["state"]["key"].astype(np.uint32)
    for nx, lf in ((0, 2), (625, 1), (3, 5), (0, 625), (-1, 1)):
        assert _advance(L, words, nx, lf, 10)[0] == _lib.MVTB_EINVAL
    nx, lf = C.c_int32(0), C.c_int32(1)
    assert L.mvtb_mt19937_advance(None, 625, emu.ptr(words.copy()), C.byref(nx), C.byref(lf)) == _lib.MVTB_EINVAL
    assert L.mvtb_mt19937_advance(None, 624, None, C.byref(nx), C.byref(lf)) == _lib.MVTB_EINVAL
    assert L.mvtb_mt19937_jump_poly(5, None) == _lib.MVTB_EINVAL
    t = np.zeros((2, N_STATE), dtype=np.uint32)
    assert L.mvtb_mt19937_chunk_table(623, 2, emu.ptr(t)) == _lib.MVTB_EINVAL
    assert L.mvtb_mt19937_chunk_table(1000, 0, emu.ptr(t)) == _lib.MVTB_EINVAL
    assert L.mvtb_mt19937_chunk_table(1000, 2, None) == _lib.MVTB_EINVAL
    u = np.zeros(10, dtype=np.float32)
    st = np.zeros((1, 640), dtype=np.uint32)
    ws = np.zeros(L.mvtb_mt19937_workspace_bytes(1) // 4, dtype=np.uint32)
    args = dict(u=emu.ptr(u), n=10, S=1, st=emu.ptr(st), t=emu.ptr(t), chunk=1000, nch=2, ws=emu.ptr(ws))

    def call(**kw):
        a = {**args, **kw}
        return L.mvtb_mt19937_uniform_f32(a["u"], a["n"], a["S"], a["st"], a["t"], a["chunk"], a["nch"], a["ws"], None)
    assert call(S=-1) == _lib.MVTB_EINVAL and call(S=65536) == _lib.MVTB_EINVAL
    assert call(chunk=623) == _lib.MVTB_EINVAL and call(nch=0) == _lib.MVTB_EINVAL
    for k in ("u", "st", "t", "ws"):
        assert call(**{k: None}) == _lib.MVTB_EINVAL
    assert call(n=0, u=None) == 0 and call(S=0, u=None) == 0
    assert L.mvtb_mt19937_workspace_bytes(0) == 0


def test_train_stage_draw_advances_the_generator_as_per_sample_calls(L, monkeypatch):
    import filters_and_operators as F
    from mvtb import _lib, spatial as S
    from mvtb.train_stage import TrainStage
    from test_train_stage import _fake_cache
    monkeypatch.setattr(_lib, "_lib", L)
    shapes = [(20, 18, 9), (16, 14, 8), (12, 10, 6)]

    def tail(seed):
        t = [S.RandSpatialCropd(["image", "label"], roi_size=[12, 10, 6], random_size=False), F.SelectChanneld("image", 1),
             F.SaltAndPepper(0.05, "image", prob=1.0, rng="torch")]
        t[0].set_random_state(seed=seed)
        t[2].set_random_state(seed=seed + 1)
        return t
    cache = _fake_cache(shapes)
    with pytest.raises(NotImplementedError, match="torch_generator=True"):
        TrainStage(cache, tail(0))
    stage = TrainStage(cache, tail(0), torch_generator=True)
    torch.manual_seed(5)
    torch.rand(77)
    rec = stage.draw([2, 0, 1, 1])
    after = torch.get_rng_state()
    torch.manual_seed(5)
    torch.rand(77)
    # the first sample records the stream's start, the others continue it
    assert np.array_equal(rec["sp_state"][0][:N_STATE].view(np.uint32), F_words(torch.get_rng_state()))
    assert rec["sp_state"][1:] == [None] * 3
    for j in range(4):
        torch.rand(1 * 12 * 10 * 6)                    # what the per-sample SaltAndPepper draws: one channel of the crop
    assert torch.equal(torch.get_rng_state(), after)
    assert stage.sp.offset == 0
    recs = [stage[i] for i in (1, 2)]                  # one record per sample, as forked workers make them
    assert all(r["sp_state"][0] is not None for r in recs)


def F_words(st):
    from mvtb import functional as Fn
    return Fn.mt19937_unpack(st)[0]
