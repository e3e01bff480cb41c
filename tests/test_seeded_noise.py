"""Seeded prior noise (ev_prior_noise, MatchaTTS.synthesise(seed=...), synthesise_corpus / synthesise_file(seed=...)): an
utterance's noise is a function of (seed, feature, frame) only, drawn on the GPU by Philox4x32-10 and Box-Muller in float64.

CPU: the oracle's known answers (Philox, splitmix64), its Box-Muller bounds, the parsing of seeds and the corpus driver's
refusals.  GPU: the kernel against the oracle, its invariances, synthesise(seed=) against synthesise(z=) with the same noise,
the oracle's mel, corpus invariance under rank splits / lanes / graphs / RNG history, statistics, launches and refusals."""
import ctypes as C

import numpy as np
import pytest
import torch

import emojivoice_b200 as ev
from emojivoice_b200 import _lib, batch, synthetic
from emojivoice_b200.config import HIFIGAN_V1, VCTK
from emojivoice_b200.matcha import per_item_seed
from oracle import matcha_oracle as mo
from oracle import prior_noise as pn
from tests.conftest import rel_l2

gpu = pytest.mark.gpu
TOL = {"fp32": 1e-4, "bf16": 1e-2}
U64 = 1 << 64
SEEDS = [0, 1, 1 << 32, 1 << 63, U64 - 1, -1]


# ------------------------------------------------------------------------------------------------ CPU
def test_oracle_philox_known_answers():
    m = 0xFFFFFFFF
    kat = [((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
           ((m,) * 4, (m, m), (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
           ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0), (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1))]
    for ctr, key, want in kat:
        assert tuple(int(w) for w in pn.philox4x32_10(*ctr, *key)) == want
    # vectorised: the same answers inside an array
    got = pn.philox4x32_10(np.array([0, m]), np.array([0, m]), np.array([0, m]), np.array([0, m]), np.array([0, m]), np.array([0, m]))
    assert [int(w[1]) for w in got] == list(kat[1][2]) and [int(w[0]) for w in got] == list(kat[0][2])


def test_splitmix64_known_answers():
    want = {0: [0xE220A8397B1DCDAF, 0x6E789E6AA1B965F4, 0x06C45D188009454F],
            1234567: [0x599ED017FB08FC85, 0x2C73F08458540FA5, 0x883EBCE5A3F27C77]}
    for s, w in want.items():
        assert pn.splitmix64(s, 3) == w
        assert batch.splitmix64(s, 3) == w                 # the corpus driver's own copy
    assert batch.splitmix64(-1, 5) == pn.splitmix64(U64 - 1, 5)


def test_box_muller_is_finite_and_bounded():
    edge = np.array([0, 1, 0x7FFFFFFF, 0x80000000, 0xFFFFFFFE, 0xFFFFFFFF], dtype=np.uint64)
    a, b = np.meshgrid(edge, edge)
    z0, z1 = pn.box_muller(a, b)
    bound = np.sqrt(-2.0 * np.log(2.0 ** -33))
    assert bound < 6.77
    for z in (z0, z1):
        assert np.all(np.isfinite(z)) and np.all(np.abs(z) <= bound)
    z = pn.prior_noise([0, 5, U64 - 1], 80, 999)
    assert z.dtype == np.float32 and np.all(np.isfinite(z)) and float(np.abs(z).max()) <= 6.77
    # a frame's value does not depend on T or on the other seeds
    assert np.array_equal(pn.prior_noise([5], 80, 333)[0], z[1, :, :333])


def test_per_item_seed_parsing():
    assert per_item_seed(None, 3) is None
    assert per_item_seed(7, 3).tolist() == [7, 7, 7]
    assert per_item_seed(np.int64(7), 2).tolist() == [7, 7]
    assert per_item_seed(-1, 1).tolist() == [-1]                    # mod 2^64: 2^64 - 1 in two's complement
    assert per_item_seed(U64 - 1, 1).tolist() == [-1]
    assert per_item_seed(1 << 63, 1).tolist() == [-(1 << 63)]
    assert per_item_seed(-(1 << 63), 1).tolist() == [-(1 << 63)]
    assert per_item_seed([1, U64 - 1, 3], 3).tolist() == [1, -1, 3]
    assert per_item_seed(np.array([4, 5]), 2).tolist() == [4, 5]
    assert per_item_seed(torch.tensor([1, 2], dtype=torch.int32), 2).tolist() == [1, 2]
    t = torch.tensor([9, -5, 3], dtype=torch.int64)
    got = per_item_seed(t, 3)
    assert got.dtype == torch.int64 and got.data_ptr() == t.data_ptr()            # taken as it is, not read back
    assert per_item_seed(torch.tensor(11), 2).tolist() == [11, 11]
    for bad in (True, 1.0, 1.5, "3", U64, -(1 << 63) - 1, [1, True], [1, 2.0], [1, None], torch.tensor([1.0, 2.0]),
                torch.tensor([True, False]), [1, 2], [1, 2, 3, 4], torch.tensor([1, 2], dtype=torch.int64)):
        with pytest.raises(ValueError):
            per_item_seed(bad, 3)


def test_corpus_seeds_and_refusals():
    d = dict(length_scale=1.0, temperature=0.667, n_timesteps=10, denoiser_strength=None)
    utts = [([1, 2], 3), ([4], 5, {"seed": 99}), ([6], 7, {"temperature": 0.5})]
    s, own = batch.utterance_settings(utts, d)
    assert own and s[1]["seed"] == 99
    s2, own2 = batch.utterance_settings(utts[:2], d)
    assert not own2                                                  # a seed is not a synthesis setting: the plan keeps its shape
    derived = pn.splitmix64(1234567, 3)
    assert batch.utterance_seeds(s, 1234567) == [derived[0], 99, derived[2]]
    assert batch.utterance_seeds(s[:1] + s[2:], None) is None
    every = [dict(x, seed=i - 1) for i, x in enumerate(s)]
    assert batch.utterance_seeds(every, None) == [U64 - 1, 0, 1]
    with pytest.raises(ValueError, match="others do not"):
        batch.utterance_seeds(s, None)                                # one utterance seeded, the others not
    with pytest.raises(ValueError, match="z_fn"):
        batch.utterance_seeds(s, 5, z_fn=lambda *a: None)
    for bad in (True, 2.5, U64):
        with pytest.raises(ValueError):
            batch.utterance_seeds(s, bad)
        with pytest.raises(ValueError):
            batch.utterance_seeds([dict(d, seed=bad)], None)
    # refused before any work is done (no model is touched)
    with pytest.raises(ValueError, match="others do not"):
        batch.synthesise_corpus(None, None, utts)
    with pytest.raises(ValueError, match="z_fn"):
        batch.synthesise_corpus(None, None, utts[:1], seed=3, z_fn=lambda *a: None)


def test_plan_does_not_depend_on_seeds(monkeypatch):
    from emojivoice_b200 import sharding

    seen = []

    def shard(*a, **kw):
        seen.append((a, kw))
        raise RuntimeError("stop")

    monkeypatch.setattr(sharding, "shard", shard)
    plain = [([1] * (3 + i % 7), i % 4) for i in range(20)]
    for utts, kw in ((plain, {}), (plain, {"seed": 5}), ([u + ({"seed": i},) for i, u in enumerate(plain)], {})):
        with pytest.raises(RuntimeError, match="stop"):
            batch.synthesise_corpus(None, None, utts, batch_size=4, **kw)
    assert seen[0] == seen[1] == seen[2]


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def ctx():
    return _lib.Context()


@pytest.fixture(scope="module")
def matcha(matcha_sd):
    m = ev.MatchaTTS(**VCTK.constructor_kwargs())
    m.load_state_dict(matcha_sd)
    return m


@pytest.fixture(scope="module")
def gen_den():
    g = ev.Generator(HIFIGAN_V1)
    g.load_state_dict(synthetic.hifigan_state_dict(HIFIGAN_V1, seed=4321, gain=1.0))
    g.remove_weight_norm()
    return g, ev.Denoiser(g)


def _noise(ctx, seeds, F, T, offset=0):
    """ev_prior_noise into a NaN-filled buffer with guard words on both sides (offset shifts z off 16-byte alignment)."""
    s = per_item_seed(seeds, len(seeds)).cuda()
    B, n = len(seeds), len(seeds) * F * T
    buf = torch.full((n + offset + 64,), float("nan"), device="cuda")
    z = buf[offset: offset + n]
    ctx.check(_lib.lib().ev_prior_noise(ctx.handle, _lib.ptr(s), B, F, T, _lib.ptr(z), _lib.stream_ptr()), "ev_prior_noise")
    torch.cuda.synchronize()
    assert torch.isnan(buf[:offset]).all() and torch.isnan(buf[offset + n:]).all()          # nothing written outside z
    return z.reshape(B, F, T).clone()


def _within_oracle(got, ref32):
    got = got.cpu().numpy()
    tol = np.maximum(np.spacing(np.abs(ref32)), np.float32(2.0 ** -40))
    err = np.abs(got.astype(np.float64) - ref32.astype(np.float64))
    return bool(np.all(err <= tol)), float(err.max())


@gpu
@pytest.mark.parametrize("T", [1, 4, 5, 668, 1001, 20000])
def test_kernel_matches_oracle(ctx, T):
    for seeds in (SEEDS[:3], SEEDS[3:5], SEEDS[5:]):                  # B = 3, 2, 1
        got = _noise(ctx, seeds, 80, T)
        assert torch.isfinite(got).all()
        ok, err = _within_oracle(got, pn.prior_noise(seeds, 80, T))
        assert ok, (seeds, T, err)


@gpu
@pytest.mark.parametrize("T", [5, 668, 1001])
def test_unaligned_output_takes_the_scalar_stores(ctx, T):
    """z one float past a 16-byte boundary: every group is stored by scalars, with the same bits."""
    assert torch.equal(_noise(ctx, [3, 4], 80, T, offset=1), _noise(ctx, [3, 4], 80, T))


@gpu
def test_rows_do_not_depend_on_batch_position_size_or_length(ctx):
    seeds = [11, U64 - 7, 1 << 40, 11]
    full = _noise(ctx, seeds, 80, 1001)
    assert torch.equal(full[0], full[3])                             # equal seeds, equal rows
    for b, s in enumerate(seeds):
        assert torch.equal(_noise(ctx, [s], 80, 1001)[0], full[b])  # B = 1
        assert torch.equal(_noise(ctx, [5, s], 80, 333)[1], full[b, :, :333])   # another row, B, T
        assert torch.equal(_noise(ctx, [s, 6, 7], 80, 1002)[0, :, :1001], full[b])
    rev = _noise(ctx, seeds[::-1], 80, 1001)
    assert torch.equal(rev, full.flip(0))


@gpu
def test_statistics(ctx):
    """About 4 M draws over fixed seeds: moments, KS against N(0, 1), lag-1 correlation along t and f, and between seeds s, s+1."""
    from scipy import stats

    seeds = list(range(100, 108))
    z = _noise(ctx, seeds, 80, 6556).double().cpu().numpy()        # 8 x 80 x 6556 = 4.2 M
    x = z.reshape(-1)
    n = x.size
    assert abs(x.mean()) < 5 / np.sqrt(n)
    assert abs(x.var() - 1.0) < 5 * np.sqrt(2.0 / n)
    assert stats.kstest(x, "norm").pvalue > 1e-3
    assert abs(stats.kurtosis(x)) < 0.02 and abs(stats.skew(x)) < 0.01

    def corr(a, b):
        return float(np.corrcoef(a.reshape(-1), b.reshape(-1))[0, 1])

    bound = 5 / np.sqrt(n / 2)
    assert abs(corr(z[:, :, 1:], z[:, :, :-1])) < bound             # along t (within and across groups of four)
    assert abs(corr(z[:, :, 1::4], z[:, :, 0::4])) < 2 * bound       # the two values of one Box-Muller pair
    assert abs(corr(z[:, 1:, :], z[:, :-1, :])) < bound             # along f
    assert abs(corr(z[1:], z[:-1])) < bound                          # seeds s and s + 1


@gpu
def test_kernel_refusals(ctx):
    L = _lib.lib()
    s = torch.zeros(2, dtype=torch.int64, device="cuda")
    z = torch.empty(2 * 80 * 8, device="cuda")
    before = ctx.launch_count()
    for args in ((None, 2, 80, 8, z), (s, 2, 80, 8, None), (s, 0, 80, 8, z), (s, 2, 0, 8, z), (s, 2, 80, 0, z), (s, -1, 80, 8, z)):
        assert L.ev_prior_noise(ctx.handle, _lib.ptr(args[0]), *args[1:4], _lib.ptr(args[4]), _lib.stream_ptr()) == -1
    assert L.ev_prior_noise(None, _lib.ptr(s), 2, 80, 8, _lib.ptr(z), _lib.stream_ptr()) == -1
    assert ctx.launch_count() == before
    assert L.ev_prior_noise(ctx.handle, _lib.ptr(s), 2, 80, 8, _lib.ptr(z), _lib.stream_ptr()) == 0
    assert ctx.launch_count() == before + 1                          # one launch per call


def _batch(seed=41, B=4):
    return synthetic.phoneme_batch(B, 8, 40, seed=seed)


@gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
@pytest.mark.parametrize("per_item", [False, True])
def test_seed_equals_the_same_z_passed_in(matcha, ctx, prec, per_item):
    x, xl, spk = _batch()
    settings = (dict(n_timesteps=[2, 3, 1, 2], temperature=[0.667, 0.5, 1.0, 0.3], length_scale=[1.0, 0.9, 1.1, 0.8]) if per_item
                else dict(n_timesteps=2, temperature=0.667, length_scale=1.0))
    seeds = [5, U64 - 2, 1 << 33, 5]
    out = matcha.synthesise(x, xl, spks=spk, dtype=prec, seed=seeds, **settings)
    z = _noise(ctx, seeds, 80, out["t_pad"])
    assert torch.equal(out["z"], z)
    ref = matcha.synthesise(x, xl, spks=spk, dtype=prec, z=z, **settings)
    for k in ("mel", "decoder_outputs", "z", "mel_lengths", "attn"):
        assert torch.equal(out[k], ref[k]), k
    # a number is every utterance with that seed; an int64 device tensor is the same seeds
    one = matcha.synthesise(x, xl, spks=spk, dtype=prec, seed=-1, **settings)
    ref1 = matcha.synthesise(x, xl, spks=spk, dtype=prec, seed=[U64 - 1] * 4, **settings)
    dev = matcha.synthesise(x, xl, spks=spk, dtype=prec, seed=per_item_seed(seeds, 4).cuda(), **settings)
    for k in ("mel", "decoder_outputs", "z"):
        assert torch.equal(one[k], ref1[k]), k
        assert torch.equal(dev[k], out[k]), k


@gpu
def test_graph_replay_reads_new_seeds(matcha_sd):
    graphed = ev.MatchaTTS(**VCTK.constructor_kwargs(), cuda_graphs=True)
    graphed.load_state_dict(matcha_sd)
    eager = ev.MatchaTTS(**VCTK.constructor_kwargs(), cuda_graphs=False)
    eager.load_state_dict(matcha_sd)
    x, xl, spk = _batch(seed=43)
    for prec in ("fp32", "bf16"):
        for _ in range(3):                                             # captured on the second call, replayed on the third
            graphed.synthesise(x, xl, 2, 0.667, spk, seed=[1, 2, 3, 4], dtype=prec)
        before = graphed._replayed_launches
        new = [10, U64 - 1, 1 << 63, 7]
        got = graphed.synthesise(x, xl, 2, 0.667, spk, seed=new, dtype=prec)
        assert graphed._replayed_launches > before
        ref = eager.synthesise(x, xl, 2, 0.667, spk, seed=new, dtype=prec)
        for k in ("z", "decoder_outputs", "mel"):
            assert torch.equal(got[k], ref[k]), (prec, k)


def _near_tie_free_batch(matcha_sd, B, seed):
    for s in range(seed, seed + 50):
        x, xl, spk = synthetic.phoneme_batch(B, 8, 30, seed=s)
        r = mo.synthesise(matcha_sd, VCTK, x, xl, 1, 0.667, spk, 1.0, z=None)
        w = torch.exp(r["logw"]) * r["x_mask"]
        if not bool((((w - torch.round(w)).abs() < 1e-4) & (r["x_mask"] > 0)).any()):
            return x, xl, spk
    raise AssertionError("no near-tie-free batch")


@gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_seeded_mel_matches_oracle(matcha, matcha_sd, prec):
    """The oracle with the generated z injected: durations bit-exact, mel within the tolerance of test_gpu_parity.py."""
    x, xl, spk = _near_tie_free_batch(matcha_sd, 3, 51)
    out = matcha.synthesise(x, xl, 2, 0.667, spk, 1.0, dtype=prec, seed=[123, 456, 789])
    ref = mo.synthesise(matcha_sd, VCTK, x, xl, 2, 0.667, spk, 1.0, z=out["z"].cpu())
    assert torch.equal(out["w_ceil"].cpu(), ref["w_ceil"])
    assert rel_l2(out["mel"].cpu(), ref["mel"]) < TOL[prec]
    assert rel_l2(out["decoder_outputs_full"].cpu(), ref["decoder_outputs_full"]) < TOL[prec]


@gpu
def test_launches_and_refusals(matcha):
    x, xl, spk = _batch(seed=47)
    matcha.cuda_graphs = False
    try:
        counts = {}
        for n in (2, 3):
            for seed in (None, 9):
                matcha.launch_count(reset=True)
                matcha.synthesise(x, xl, n, 0.667, spk, dtype="bf16", seed=seed)
                counts[n, seed] = matcha.launch_count(reset=True)
    finally:
        matcha.cuda_graphs = True
    assert counts[2, 9] == counts[2, None] + 1 and counts[3, 9] == counts[3, None] + 1, counts
    assert counts[3, 9] - counts[2, 9] == 24, counts                 # 24 launches per Euler step
    z = torch.zeros(4, 80, 8)
    for kw in (dict(seed=1, z=z), dict(seed=[1, 2]), dict(seed=[1, 2, 3, 4, 5]), dict(seed=True), dict(seed=1.0), dict(seed=U64),
               dict(seed=[1, 2, 3, "4"]), dict(seed=torch.ones(4))):
        with pytest.raises(ValueError):
            matcha.synthesise(x, xl, 2, 0.667, spk, **kw)


def _corpus_utts(n, seed):
    x, xl, spks = synthetic.phoneme_batch(n, 5, 40, seed=seed)
    dn = [None, "default", 0.001]                                    # not denoised, the call's strength, its own strength
    out = []
    for i in range(n):
        s = dn[i % 3]
        out.append((x[i, : int(xl[i])].tolist(), int(spks[i])) + (() if s == "default" else ({"denoiser_strength": s},)))
    return out


@gpu
def test_corpus_waveforms_do_not_depend_on_the_split(matcha, gen_den):
    gen, den = gen_den
    utts = _corpus_utts(24, 61)
    S = 1234567
    kw = dict(batch_size=4, n_timesteps=2, denoiser=den, denoiser_strength=0.0005, seed=S)
    ref, _ = ev.synthesise_corpus(matcha, gen, utts, **kw)
    assert sorted(ref) == list(range(24))

    def same(got, items=None):
        for i in (sorted(got) if items is None else items):
            assert torch.equal(got[i]["waveform"], ref[i]["waveform"]), i

    for ws in (2, 3):                                                # the union of every rank's share, one after another
        union = {}
        for r in range(ws):
            part, _ = ev.synthesise_corpus(matcha, gen, utts, rank=r, world_size=ws, **kw)
            assert not set(part) & set(union)
            union.update(part)
        assert sorted(union) == list(range(24))
        same(union)
    same(ev.synthesise_corpus(matcha, gen, utts, in_flight=3, **kw)[0], range(24))
    for _ in range(2):                                               # second run: the repeated shapes are graph replays
        same(ev.synthesise_corpus(matcha, gen, utts, cuda_graphs=True, **kw)[0], range(24))
    torch.randn(1000, device="cuda")                                 # unrelated draws move the RNG state
    torch.randn(3, 7)
    part, _ = ev.synthesise_corpus(matcha, gen, utts, rank=1, world_size=3, **kw)
    assert part
    same(part)
    # a "seed" setting overrides the derived value; the derived value itself changes nothing
    derived = pn.splitmix64(S, 24)
    own = [u[:2] + (dict(u[2] if len(u) > 2 else {}, seed=derived[i]),) for i, u in enumerate(utts)]
    same(ev.synthesise_corpus(matcha, gen, own, **dict(kw, seed=None))[0], range(24))
    over = list(utts)
    over[5] = utts[5][:2] + (dict(utts[5][2] if len(utts[5]) > 2 else {}, seed=42),)
    got, _ = ev.synthesise_corpus(matcha, gen, over, **kw)
    assert not torch.equal(got[5]["waveform"], ref[5]["waveform"])
    same(got, [i for i in range(24) if i != 5])                     # the other utterances keep their noise and their mel
    # another corpus seed gives other audio
    other, _ = ev.synthesise_corpus(matcha, gen, utts, **dict(kw, seed=S + 1))
    assert all(not torch.equal(other[i]["waveform"], ref[i]["waveform"]) for i in range(24))


@gpu
def test_synthesise_file_same_files_for_any_world_size(matcha, gen_den, tmp_path):
    gen, _ = gen_den
    g2p = {"one": "wˈʌn", "two words here": "tˈuː wˈɜːdz hˈɪɹ", "three": "θɹˈiː", "a longer line of text": "ɐ lˈɔŋɡɚ lˈaɪn ʌv tˈɛkst",
           "five": "fˈaɪv"}
    script = tmp_path / "script.txt"
    script.write_text("\n".join(f"{t}|{10 + i}" for i, t in enumerate(g2p)) + "\n", encoding="utf-8")
    kw = dict(phonemizer=lambda t: g2p[" ".join(t.split())], n_timesteps=2, batch_size=2, seed=77)
    one, _ = ev.synthesise_file(matcha, gen, script, tmp_path / "ws1", **kw)
    two = []
    for r in range(2):
        two += ev.synthesise_file(matcha, gen, script, tmp_path / "ws2", rank=r, world_size=2, **kw)[0]
    assert sorted(w[0] for w in two) == [w[0] for w in one] == list(range(5))
    names = {w[0]: w[1] for w in two}
    for i, path, _ in one:
        with open(path, "rb") as a, open(names[i], "rb") as b:
            assert a.read() == b.read(), i
