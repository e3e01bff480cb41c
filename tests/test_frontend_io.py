"""Host-side rows f2/f3 of SURVEY.md 8f: symbol table / id mapping, script formats, PCM_24 WAV + NPY writers."""
import json
import os
import sys
import wave

import numpy as np
import pytest
import torch

import emojivoice_b200 as ev
from emojivoice_b200 import audio_io, text_frontend as tf
from oracle import reference_shim as shim


def test_symbol_table_shape_and_mapping_rules():
    assert len(tf.SYMBOLS) == 198 and tf.SYMBOLS[0] == "_" and tf.SPACE_ID == 16          # symbols.py:14-17
    assert len(set(tf.SYMBOLS)) == 198 - 4 and len(tf.DUPLICATES) >= 1                   # SURVEY H7: 4 duplicate entries
    for s in tf.DUPLICATES:                                                              # dict comprehension: last index wins
        assert tf.SYMBOL_TO_ID[s] == max(i for i, t in enumerate(tf.SYMBOLS) if t == s)
    ids = tf.cleaned_text_to_sequence("həlˈoʊ wˈɜːld!")
    assert tf.sequence_to_text(ids) == "həlˈoʊ wˈɜːld!" and all(0 < i < 198 for i in ids)
    with pytest.raises(KeyError):
        tf.cleaned_text_to_sequence("日本")


def test_symbol_table_equals_the_reference_file():
    """Against the reference's table as committed (tests/golden/symbols.json) and, where the reference tree is present, against
    its own symbols.py imported where it lies (EV_WRITE_GOLDEN=1 then rewrites the fixture from it)."""
    golden = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "symbols.json")
    if shim.available():
        sys.path.insert(0, os.path.join(shim.REFERENCE_ROOT, "Matcha-TTS", "matcha", "text"))
        try:
            import symbols as ref_symbols
        finally:
            sys.path.pop(0)
        if os.environ.get("EV_WRITE_GOLDEN"):
            with open(golden, "w", encoding="utf-8") as f:
                json.dump({"symbols": ref_symbols.symbols, "space_id": ref_symbols.SPACE_ID}, f, ensure_ascii=False, indent=0)
                f.write("\n")
        assert tf.SYMBOLS == ref_symbols.symbols and tf.SPACE_ID == ref_symbols.SPACE_ID
    with open(golden, encoding="utf-8") as f:
        ref = json.load(f)
    assert tf.SYMBOLS == ref["symbols"] and tf.SPACE_ID == ref["space_id"]
    assert tf.SYMBOL_TO_ID == {s: i for i, s in enumerate(ref["symbols"])}


def test_process_text_intersperses_blanks_like_the_cli():
    out = tf.process_text("Hi there", phonemizer=lambda t: "haɪ ðɛɹ")
    ids = tf.cleaned_text_to_sequence("haɪ ðɛɹ")
    assert out["x"].shape == (1, 2 * len(ids) + 1) and int(out["x_lengths"]) == 2 * len(ids) + 1
    assert out["x"][0, 1::2].tolist() == ids and set(out["x"][0, 0::2].tolist()) == {0}            # utils.py:131-135


def test_script_formats():
    assert audio_io.parse_script(["Hello there|107", "", " a|b|c |12 "]) == [("Hello there", 107), ("a|b|c", 12)]
    with pytest.raises(ValueError):
        audio_io.parse_script(["no speaker here"])
    story = ["Once upon a time, there lived a brave Pixel Prince \U0001F60E.", "The dragon appeared (\U0001F621)!", "Plain line."]
    got = audio_io.parse_emoji_script(story, ev.EMOJI_MAPPING_FEMALE, default=12)
    assert [s for _, s in got] == [79, 58, 12]
    assert "\U0001F60E" not in got[0][0] and "(" not in got[1][0] and got[2][0] == "Plain line."


def test_pcm24_wav_and_npy_writers(tmp_path):
    g = torch.Generator().manual_seed(0)
    wav = (torch.rand(22050, generator=g) * 2.4 - 1.2)                    # includes samples beyond [-1, 1] -> clipped
    wav[:4] = torch.tensor([0.0, 1.0, -1.0, 0.5])
    mel = torch.randn(80, 87, generator=g)
    path = audio_io.save_to_folder("utterance_000_speaker_107", {"mel": mel, "waveform": wav}, tmp_path / "out")
    with wave.open(path, "rb") as w:                                     # an independent reader agrees on the container
        assert (w.getnchannels(), w.getsampwidth(), w.getframerate(), w.getnframes()) == (1, 3, 22050, 22050)
    back, sr = audio_io.read_wav_pcm24(path)
    assert sr == 22050 and back.shape == (22050,)
    pcm = audio_io.float_to_pcm24(wav)
    assert pcm[:4].tolist() == [0, 8388607, -8388607, 4194304] and pcm.max() == 8388607 and pcm.min() == -8388608
    assert np.abs(back - np.clip(wav.numpy(), -1.0000001, 1.0)).max() <= 0.5 / 8388607 + 1e-7 + 1.2e-7   # half an LSB
    assert np.array_equal(np.load(str(tmp_path / "out" / "utterance_000_speaker_107.npy")), mel.numpy())
