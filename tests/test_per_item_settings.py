"""Padded batches whose utterances each have their own speaking rate (length_scale), temperature and step count.

CPU: the per-item Euler tables, the argument checks of MatchaTTS.synthesise, the micro-batch cost.  GPU: per-item calls against
the scalar calls they are defined by (bit for bit), against the oracle run per utterance at the batch's padded length, graph
replays, the corpus driver and the kernels a mixed batch runs."""
import ctypes as C

import numpy as np
import pytest
import torch

import emojivoice_b200 as ev
from emojivoice_b200 import _lib, sharding, synthetic
from emojivoice_b200.config import HIFIGAN_V1, VCTK
from emojivoice_b200.matcha import per_item_setting
from oracle import matcha_oracle as mo
from tests.conftest import rel_l2

gpu = pytest.mark.gpu
TOL = {"fp32": 1e-4, "bf16": 1e-2}


# ------------------------------------------------------------------------------------------------ CPU
def _schedule(n):
    t, dt = (C.c_float * n)(), (C.c_float * n)()
    assert _lib.lib().ev_test_euler_schedule(n, t, dt) == 0
    return list(t), list(dt)


@pytest.mark.parametrize("ns", [[1, 2, 4, 10], [10, 1], [3, 3, 3], [50, 7, 1, 2, 49]])
def test_per_item_tables_are_the_scalar_schedules_with_held_rows(ns):
    B, n_max = len(ns), max(ns)
    t, dt = (C.c_float * (B * n_max))(), (C.c_float * (B * n_max))()
    assert _lib.lib().ev_test_euler_tables((C.c_int32 * B)(*ns), B, t, dt) == 0
    t = np.array(t, dtype=np.float32).reshape(n_max, B)
    dt = np.array(dt, dtype=np.float32).reshape(n_max, B)
    for b, n in enumerate(ns):
        ts, dts = _schedule(n)
        assert np.array_equal(t[:n, b], np.array(ts, dtype=np.float32))      # bit for bit
        assert np.array_equal(dt[:n, b], np.array(dts, dtype=np.float32))
        assert np.all(t[n:, b] == np.float32(ts[-1])) and np.all(dt[n:, b] == 0.0)   # held rows


def test_per_item_tables_reject_bad_counts():
    t, dt = (C.c_float * 8)(), (C.c_float * 8)()
    assert _lib.lib().ev_test_euler_tables((C.c_int32 * 2)(2, 0), 2, t, dt) == -1
    assert _lib.lib().ev_test_euler_tables(None, 2, t, dt) == -1


def test_per_item_setting_arguments():
    assert per_item_setting(10, 3, "n_timesteps") == 10
    assert per_item_setting(torch.tensor(0.5), 3, "temperature") == 0.5
    assert per_item_setting([4, 4, 4], 3, "n_timesteps") == 4                       # equal values are the scalar call
    assert per_item_setting(torch.tensor([0.8, 1.0]), 2, "length_scale") == (pytest.approx(0.8), 1.0)
    assert per_item_setting(np.array([2, 10]), 2, "n_timesteps") == (2, 10)
    with pytest.raises(ValueError, match="expected a number or 3 values"):
        per_item_setting([1, 2], 3, "n_timesteps")
    with pytest.raises(ValueError, match="integers >= 1"):
        per_item_setting([2, 0], 2, "n_timesteps")
    with pytest.raises(ValueError, match="integers >= 1"):
        per_item_setting([2, 2.5], 2, "n_timesteps")
    with pytest.raises(ValueError, match="positive"):
        per_item_setting([0.8, 0.0], 2, "length_scale")
    with pytest.raises(ValueError, match="positive"):
        per_item_setting([0.8, -1.0], 2, "length_scale")
    for bad in (float("nan"), float("inf")):
        with pytest.raises(ValueError, match="finite"):
            per_item_setting([0.8, bad], 2, "length_scale")
        with pytest.raises(ValueError, match="finite"):
            per_item_setting([0.5, bad], 2, "temperature")


def test_sharding_cost_uses_each_utterances_steps():
    lens = [10, 30, 20, 40, 25]
    steps = [4, 10, 1, 10, 2]
    mbs = sharding.microbatches(lens, 2, n_timesteps=steps)
    uniform = sharding.microbatches(lens, 2, n_timesteps=10)
    assert [m.items for m in mbs] == [m.items for m in uniform]                     # the plan does not change
    for m in mbs:
        frames = int(round(m.tx_max * 2.9))
        assert m.cost == sum(sharding.estimate_flops(m.tx_max, frames, steps[i]) for i in m.items)
    assert mbs[0].cost < uniform[0].cost
    with pytest.raises(ValueError):
        sharding.microbatches(lens, 2, n_timesteps=[1, 2])
    st = sharding.ShardStats()
    st.add([30, 60], [10, 20], [2, 4], 0.0)
    assert st.flops == sharding.estimate_flops(10, 30, 2) + sharding.estimate_flops(20, 60, 4)


def test_corpus_settings_take_the_keyword_defaults():
    from emojivoice_b200.batch import utterance_settings

    d = dict(length_scale=1.0, temperature=0.667, n_timesteps=10)
    s, own = utterance_settings([([1, 2], 3), ([4], 5)], d)
    assert not own and s == [d, d]
    s, own = utterance_settings([([1, 2], 3), ([4], 5, {"n_timesteps": 4, "length_scale": 0.8})], d)
    assert own and s[0] == d and s[1] == dict(length_scale=0.8, temperature=0.667, n_timesteps=4)
    with pytest.raises(ValueError, match="unknown"):
        utterance_settings([([1], 3, {"speed": 2})], d)


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def matcha(matcha_sd):
    m = ev.MatchaTTS(**VCTK.constructor_kwargs())
    m.load_state_dict(matcha_sd)
    return m


@pytest.fixture(scope="module")
def gen():
    g = ev.Generator(HIFIGAN_V1)
    g.load_state_dict(synthetic.hifigan_state_dict(HIFIGAN_V1, seed=7))
    g.remove_weight_norm()
    return g


def _decode(model, mu, yl, z, spk, n, temp, prec, items=False):
    """ev_decode (n, temp scalars) or ev_decode_items (n, temp sequences) on a fixed T_pad -> (decoder_out, mel)."""
    ctx, L = model._ctx, _lib.lib()
    B, Fm, T = mu.shape
    dec, mel = torch.empty_like(mu), torch.empty_like(mu)
    if items:
        nb = L.ev_decode_items_workspace_bytes(ctx.handle, B, T, max(n))
        ws = ctx.workspace(nb)
        temps = torch.tensor(temp, dtype=torch.float32, device=mu.device)
        ctx.check(L.ev_decode_items(ctx.handle, _lib.ptr(mu), _lib.ptr(yl), _lib.ptr(z), _lib.ptr(spk), B, T, (C.c_int32 * B)(*n),
                                    _lib.ptr(temps), _lib.PREC[prec], _lib.ptr(dec), _lib.ptr(mel), _lib.ptr(ws), ws.numel(),
                                    _lib.stream_ptr()), "ev_decode_items")
    else:
        ws = ctx.workspace(L.ev_decode_workspace_bytes(ctx.handle, B, T, n))
        ctx.check(L.ev_decode(ctx.handle, _lib.ptr(mu), _lib.ptr(yl), _lib.ptr(z), _lib.ptr(spk), B, T, n, temp, _lib.PREC[prec],
                              _lib.ptr(dec), _lib.ptr(mel), _lib.ptr(ws), ws.numel(), _lib.stream_ptr()), "ev_decode")
    torch.cuda.synchronize()
    return dec, mel


def _decoder_inputs(B, T, lens, seed):
    g = torch.Generator().manual_seed(seed)
    yl = torch.tensor(lens, dtype=torch.int64)
    mask = (torch.arange(T)[None, :] < yl[:, None]).float()[:, None, :]
    mu = (torch.randn(B, 80, T, generator=g) * mask).cuda()
    z = torch.randn(B, 80, T, generator=g).cuda()
    spk = torch.randn(B, VCTK.spk_emb_dim, generator=g).cuda()
    return mu, yl.cuda(), z, spk


@gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
@pytest.mark.parametrize("lanes", [1, 2])
def test_decoder_items_equal_scalar_calls_per_item(matcha, matcha_sd, prec, lanes, monkeypatch):
    """ev_decode_items with n in {1, 2, 4, 10} and three temperatures: item b is bit-identical to item b of ev_decode called with
    (n_b, temperature_b) for the whole batch at the same T_pad.  Ragged (one item at T_pad, one far shorter); lanes = 2 runs the
    decoder's multi-lane path (B >= 8), where the per-item arrays are offset by each lane's first item."""
    model = matcha
    if lanes > 1:
        monkeypatch.setenv("EV_DEC_LANES", str(lanes))
        model = ev.MatchaTTS(**VCTK.constructor_kwargs())
        model.load_state_dict(matcha_sd)
    T = 200
    lens = [200, 23, 150, 91, 200, 64, 177, 120, 37]
    B = len(lens)
    ns = [1, 2, 4, 10, 2, 10, 4, 1, 2]
    temps = [0.5, 0.667, 1.0, 0.667, 1.0, 0.5, 0.667, 1.0, 0.5]
    mu, yl, z, spk = _decoder_inputs(B, T, lens, seed=3)
    dec, mel = _decode(model, mu, yl, z, spk, ns, temps, prec, items=True)
    for pair in sorted(set(zip(ns, temps))):
        ref_dec, ref_mel = _decode(model, mu, yl, z, spk, pair[0], pair[1], prec)
        for b in range(B):
            if (ns[b], temps[b]) == pair:
                assert torch.equal(dec[b], ref_dec[b]), (b, pair)
                assert torch.equal(mel[b], ref_mel[b]), (b, pair)
    # equal per-item arrays are the scalar call
    ref_dec, ref_mel = _decode(model, mu, yl, z, spk, 4, 0.667, prec)
    dec, mel = _decode(model, mu, yl, z, spk, [4] * B, [0.667] * B, prec, items=True)
    assert torch.equal(dec, ref_dec) and torch.equal(mel, ref_mel)


@gpu
def test_decoder_items_hold_by_select(matcha):
    """A held item's state is not touched after its last step: -0.0 stays -0.0 where x + 0*v would give +0.0."""
    T, lens = 64, [64, 64]
    mu, yl, z, spk = _decoder_inputs(2, T, lens, seed=5)
    z[:, :, :8] = -0.0
    dec1, _ = _decode(matcha, mu, yl, z, spk, 1, 0.0, "fp32")                       # temperature 0: x0 = -0.0 * 0 = -0.0
    dec, _ = _decode(matcha, mu, yl, z, spk, [1, 3], [0.0, 0.0], "fp32", items=True)
    assert torch.equal(dec[0], dec1[0])
    assert torch.equal(torch.signbit(dec[0]), torch.signbit(dec1[0]))


@gpu
def test_decoder_items_reject_bad_arguments(matcha):
    ctx, L = matcha._ctx, _lib.lib()
    mu, yl, z, spk = _decoder_inputs(2, 16, [16, 8], seed=1)
    temps = torch.ones(2, device="cuda")
    ws = ctx.workspace(L.ev_decode_items_workspace_bytes(ctx.handle, 2, 16, 2))
    args = lambda n, t: (ctx.handle, _lib.ptr(mu), _lib.ptr(yl), _lib.ptr(z), _lib.ptr(spk), 2, 16, n, t, 0, _lib.ptr(mu.clone()),
                         None, _lib.ptr(ws), ws.numel(), _lib.stream_ptr())
    assert L.ev_decode_items(*args((C.c_int32 * 2)(2, 0), _lib.ptr(temps))) == -1
    assert L.ev_decode_items(*args(None, _lib.ptr(temps))) == -1
    assert L.ev_decode_items(*args((C.c_int32 * 2)(2, 1), None)) == -1
    assert L.ev_encode_items(ctx.handle, None, None, None, 2, 4, None, None, None, None, None, None, None, None, 0, None) == -1


def _near_tie_free_batch(matcha_sd, B, lo, hi, seed, ls):
    for s in range(seed, seed + 50):
        x, xl, spk = synthetic.phoneme_batch(B, lo, hi, seed=s)
        ok = True
        for v in sorted(set(ls)):
            r = mo.synthesise(matcha_sd, VCTK, x, xl, 1, 0.667, spk, v, z=None)
            w = torch.exp(r["logw"]) * r["x_mask"]
            ok &= not bool((((w - torch.round(w)).abs() < 1e-4) & (r["x_mask"] > 0)).any())
        if ok:
            return x, xl, spk
    raise AssertionError("no near-tie-free batch")


@gpu
def test_length_stage_items_equal_scalar_calls(matcha):
    """Mixed length scales (0.8 and 1.2 included, where the float32 sum order matters, SURVEY H2b): item b's w_ceil and
    y_lengths equal those of the scalar call with length_scale[b], bit for bit."""
    x, xl, spk = synthetic.phoneme_batch(8, 20, 70, seed=31)
    ls = [0.8, 1.2, 0.9, 1.0, 1.1, 0.8, 1.2, 0.95]
    out = matcha.synthesise(x, xl, 1, 0.667, spk, ls, dtype="fp32")
    for v in sorted(set(ls)):
        ref = matcha.synthesise(x, xl, 1, 0.667, spk, v, dtype="fp32")
        for b in range(8):
            if ls[b] == v:
                assert torch.equal(out["w_ceil"][b], ref["w_ceil"][b]), (b, v)
                assert int(out["mel_lengths"][b]) == int(ref["mel_lengths"][b]), (b, v)
                n = int(ref["mel_lengths"][b])
                assert torch.equal(out["attn"][b, :, :, :n], ref["attn"][b, :, :, :n])
                assert float(out["attn"][b, :, :, n:].abs().sum()) == 0.0


@torch.inference_mode()
def _oracle_at_t_pad(sd, x, x_lengths, n_timesteps, temperature, spks, length_scale, z, t_pad):
    """oracle/matcha_oracle.py's synthesise (matcha_tts.py:116-143) from its own pieces, at a given padded length t_pad >= the
    batch's longest utterance: one utterance computed alone at the padded length of the batch it belongs to."""
    spk_emb = torch.nn.functional.embedding(spks.long(), sd["spk_emb.weight"]) if VCTK.n_spks > 1 else None
    mu_x, logw, x_mask = mo.text_encoder(sd, VCTK, x, x_lengths, spk_emb)
    w_ceil = torch.ceil(torch.exp(logw) * x_mask) * length_scale
    y_lengths = torch.clamp_min(torch.sum(w_ceil, [1, 2]), 1).long()
    assert t_pad % 4 == 0 and t_pad >= int(y_lengths.max()), (t_pad, int(y_lengths.max()))
    y_mask = mo.sequence_mask(y_lengths, t_pad).unsqueeze(1).to(x_mask.dtype)
    attn = mo.generate_path(w_ceil.squeeze(1), (x_mask.unsqueeze(-1) * y_mask.unsqueeze(2)).squeeze(1)).unsqueeze(1)
    mu_y = torch.matmul(attn.squeeze(1).transpose(1, 2), mu_x.transpose(1, 2)).transpose(1, 2)
    dec = mo.solve_euler(sd, VCTK, z * temperature, torch.linspace(0, 1, n_timesteps + 1), mu_y, y_mask, spk_emb, return_all=True)[-1]
    n = int(y_lengths.max())
    return {"w_ceil": w_ceil, "mel_lengths": y_lengths, "attn_full": attn, "decoder_outputs_full": dec,
            "mel": dec[:, :, :n] * sd["mel_std"] + sd["mel_mean"]}


def test_oracle_at_t_pad_is_the_oracle_at_its_own_padded_length(matcha_sd):
    """The padded-length oracle run above is oracle/matcha_oracle.py's synthesise when t_pad is the batch's own padded length."""
    x, xl, spk = synthetic.phoneme_batch(2, 5, 12, seed=17)
    ref = mo.synthesise(matcha_sd, VCTK, x, xl, 1, 0.667, spk, 0.9)
    z = synthetic.prior_noise(2, 80, ref["t_pad"], seed=18)
    ref = mo.synthesise(matcha_sd, VCTK, x, xl, 2, 0.667, spk, 0.9, z=z)
    got = _oracle_at_t_pad(matcha_sd, x, xl, 2, 0.667, spk, 0.9, z, ref["t_pad"])
    for k in ("w_ceil", "mel_lengths", "attn_full", "decoder_outputs_full", "mel"):
        assert torch.equal(got[k], ref[k]), k


@gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_synthesise_items_match_oracle_per_item(matcha, matcha_sd, prec):
    """Mixed settings through synthesise against the oracle run per utterance at the batch's T_pad: durations and alignment
    bit-exact, mel (padded frames included) within the tolerance of test_gpu_parity.py."""
    ls, temps, ns = [0.8, 1.2, 1.0, 0.9], [0.5, 0.667, 1.0, 0.667], [1, 4, 2, 10]
    x, xl, spk = _near_tie_free_batch(matcha_sd, 4, 8, 30, 61, ls)
    probe = matcha.synthesise(x, xl, 1, 0.667, spk, ls, dtype="fp32")
    T_pad = probe["t_pad"]
    z = synthetic.prior_noise(4, 80, T_pad, seed=62)
    out = matcha.synthesise(x, xl, ns, temps, spk, ls, z=z, dtype=prec)
    assert out["t_pad"] == T_pad
    for b in range(4):
        ref = _oracle_at_t_pad(matcha_sd, x[b:b + 1], xl[b:b + 1], ns[b], temps[b], spk[b:b + 1], ls[b], z[b:b + 1], T_pad)
        assert torch.equal(out["w_ceil"][b].cpu(), ref["w_ceil"][0])
        assert int(out["mel_lengths"][b]) == int(ref["mel_lengths"][0])
        assert torch.equal(out["attn"][b].cpu(), ref["attn_full"][0][:, : out["attn"].shape[2]])
        assert rel_l2(out["decoder_outputs_full"][b].cpu(), ref["decoder_outputs_full"][0]) < TOL[prec], b
        n = int(ref["mel_lengths"][0])
        assert rel_l2(out["mel"][b, :, :n].cpu(), ref["mel"][0]) < TOL[prec], b


@gpu
def test_graph_replay_reads_new_per_item_values(matcha_sd):
    """A replay of the captured encoder / decoder graphs with new per-item temperatures and length scales gives the eager result."""
    graphed = ev.MatchaTTS(**VCTK.constructor_kwargs(), cuda_graphs=True)
    graphed.load_state_dict(matcha_sd)
    eager = ev.MatchaTTS(**VCTK.constructor_kwargs(), cuda_graphs=False)
    eager.load_state_dict(matcha_sd)
    x, xl, spk = synthetic.phoneme_batch(4, 10, 40, seed=71)
    ns = [2, 4, 1, 3]
    a = dict(temperature=[0.5, 0.667, 1.0, 0.667], length_scale=[1.0, 0.8, 0.9, 1.1])
    probe = eager.synthesise(x, xl, 1, 0.667, spk, a["length_scale"])
    t_pad, longest = probe["t_pad"], int(probe["mel_lengths"].argmax())
    # new values; the longest utterance keeps its length scale and the others only get shorter: same T_pad, same graph keys
    b = dict(temperature=[1.0, 0.3, 0.667, 0.9], length_scale=[v if i == longest else v * 0.9 for i, v in enumerate(a["length_scale"])])
    assert eager.synthesise(x, xl, 1, 0.667, spk, b["length_scale"])["t_pad"] == t_pad
    z = synthetic.prior_noise(4, 80, t_pad, seed=72)
    for prec in ("fp32", "bf16"):
        for _ in range(3):                                             # captured on the second call, replayed on the third
            graphed.synthesise(x, xl, ns, spks=spk, z=z, dtype=prec, **a)
        before = graphed._replayed_launches
        got = graphed.synthesise(x, xl, ns, spks=spk, z=z, dtype=prec, **b)
        assert graphed._replayed_launches > before
        ref = eager.synthesise(x, xl, ns, spks=spk, z=z, dtype=prec, **b)
        for k in ("w_ceil", "mel_lengths", "attn", "decoder_outputs", "mel"):
            assert torch.equal(got[k], ref[k]), (prec, k)


@gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_equal_per_item_values_are_the_scalar_call(matcha, prec):
    """Per-item sequences whose values are all equal give the scalar call's results bit for bit (eager and graph replay) and
    launch the same kernels."""
    x, xl, spk = synthetic.phoneme_batch(4, 10, 40, seed=81)
    t_pad = matcha.synthesise(x, xl, 1, 0.667, spk, 0.9)["t_pad"]
    z = synthetic.prior_noise(4, 80, t_pad, seed=82)
    runs, launches = [], []
    for args in ((3, 0.667, 0.9), ([3] * 4, [0.667] * 4, torch.full((4,), 0.9))):
        matcha.cuda_graphs = False
        try:
            matcha.launch_count(reset=True)
            runs.append(matcha.synthesise(x, xl, args[0], args[1], spk, args[2], z=z, dtype=prec))
            launches.append(matcha.launch_count(reset=True))           # eager
        finally:
            matcha.cuda_graphs = True
        for _ in range(3):                                                # first sight, capture, replay
            matcha.launch_count(reset=True)
            runs.append(matcha.synthesise(x, xl, args[0], args[1], spk, args[2], z=z, dtype=prec))
        launches.append(matcha.launch_count(reset=True))                  # replay
    for o in runs[1:]:
        for k in ("mel", "mel_lengths", "attn", "w_ceil", "decoder_outputs"):
            assert torch.equal(o[k], runs[0][k]), k
    assert launches[0] == launches[2] and launches[1] == launches[3], launches


@gpu
def test_mixed_steps_run_the_fused_kernels(matcha):
    """bf16, mixed n: the decoder still runs resnet_tc, ff_tc, attention_tc and final_block_tc -- 24 launches per Euler step --
    with no GroupNorm fallback."""
    T, lens = 200, [200, 120, 64, 180]
    mu, yl, z, spk = _decoder_inputs(4, T, lens, seed=9)
    ctx = matcha._ctx
    ctx.launch_count(reset=True)
    _decode(matcha, mu, yl, z, spk, [2, 4, 1, 4], [0.667] * 4, "bf16", items=True)
    l4 = ctx.launch_count(reset=True)
    _decode(matcha, mu, yl, z, spk, [2, 3, 1, 3], [0.667] * 4, "bf16", items=True)
    l3 = ctx.launch_count(reset=True)
    assert l4 - l3 == 24
    ctx.profile_begin()
    _decode(matcha, mu, yl, z, spk, [2, 4, 1, 4], [0.667] * 4, "bf16", items=True)
    stats = {s["name"]: s["launches"] for s in ctx.profile_end()}
    for k, per_step in (("resnet_tc", 6), ("ff_tc", 6), ("attention_tc", 6), ("final_block_tc", 1)):
        assert stats.get(k) == 4 * per_step, (k, stats)
    assert not any(k.startswith("gn_stats") or k.startswith("gn_apply") for k in stats), stats


def _corpus(n_utts, seed):
    x, xl, spks = synthetic.phoneme_batch(n_utts, 8, 40, seed=seed)
    return [(x[i, : int(xl[i])].tolist(), int(spks[i])) for i in range(n_utts)]


@gpu
def test_corpus_per_utterance_settings(matcha, gen):
    """synthesise_corpus with per-utterance settings equals, per utterance, synthesise + the ragged vocoder of its micro-batch
    with the same per-item values; in_flight=2 equals in_flight=1; settings equal to the keywords change nothing."""
    base = _corpus(7, 91)
    opts = [{"length_scale": 0.8, "n_timesteps": 4}, {"temperature": 0.5}, {}, {"n_timesteps": 1, "temperature": 1.0},
            {"length_scale": 1.2}, {"n_timesteps": 3, "length_scale": 0.9, "temperature": 0.3}, {"n_timesteps": 2}]
    utts = [u + (o,) for u, o in zip(base, opts)]
    kw = dict(batch_size=3, n_timesteps=2, temperature=0.667, length_scale=1.0)
    zs, direct = {}, {}

    def z_fn(mb, model, x_, xl_, spks_):
        s = [dict(kw_defaults, **opts[i]) for i in mb.items]
        probe = model.synthesise(x_, xl_, 1, 0.667, spks_, [v["length_scale"] for v in s])
        z = zs.setdefault(tuple(mb.items), synthetic.prior_noise(len(mb.items), 80, probe["t_pad"], seed=len(zs) + 5))
        out = model.synthesise(x_, xl_, [v["n_timesteps"] for v in s], [v["temperature"] for v in s], spks_,
                               [v["length_scale"] for v in s], z=z)
        wav = gen(out["mel"], lengths=out["mel_lengths"]).clamp(-1, 1)
        for j, i in enumerate(mb.items):
            direct[i] = wav[j, 0, : int(out["mel_lengths"][j]) * 256].cpu()
        return z

    kw_defaults = dict(length_scale=1.0, temperature=0.667, n_timesteps=2)
    r1, s1 = ev.synthesise_corpus(matcha, gen, utts, z_fn=z_fn, **kw)
    assert sorted(r1) == list(range(7)) and s1.utterances == 7
    for i in r1:
        assert torch.equal(r1[i]["waveform"], direct[i]), i
    r2, _ = ev.synthesise_corpus(matcha, gen, utts, z_fn=z_fn, in_flight=2, **kw)
    for i in r1:
        assert torch.equal(r1[i]["waveform"], r2[i]["waveform"]), i
    # no settings vs settings equal to the keywords (the per-utterance path collapses to the scalar call)
    plain, _ = ev.synthesise_corpus(matcha, gen, base, z_fn=lambda mb, m, x_, xl_, s_: zs.setdefault(("p",) + tuple(mb.items),
                                    synthetic.prior_noise(len(mb.items), 80, m.synthesise(x_, xl_, 1, 0.667, s_, 1.0)["t_pad"], seed=9)), **kw)
    same = [u + (dict(kw_defaults),) for u in base]
    same_r, _ = ev.synthesise_corpus(matcha, gen, same, z_fn=lambda mb, m, x_, xl_, s_: zs[("p",) + tuple(mb.items)], **kw)
    for i in plain:
        assert torch.equal(plain[i]["waveform"], same_r[i]["waveform"]), i
