"""GPU parity tests (run on the B200 box with -m gpu).  Kernel-level tests compare each CUDA kernel, called through the
C ABI, with a plain torch fp32 reference of the same op; path-level tests compare with the oracle / golden fixtures."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import gpu_diag as D  # noqa: E402  (tests/ is on sys.path via conftest)
from conftest import NOTE_CASES, note_variants, report, unpack_notes  # noqa: E402


@pytest.fixture(scope="module")
def extractor():
    ex, sd = D.make_extractor(max_windows=4)
    return ex, sd


def test_gemm_epilogues_vs_torch():
    assert D.diag_gemm()


def test_chain_vs_torch():
    assert D.diag_chain()


def test_embed_tensor_core_vs_torch():
    assert D.diag_embed()


def test_attention_shapes_vs_torch():
    assert D.diag_attn()


def test_fused_qkv_attention_vs_torch():
    assert D.diag_attn_qkv()


def test_fused_qkv_attention_pair_vs_cta1_kernel():
    """CTA-pair kernel == the independent cta_group::1 kernel, incl. first-layer-sized activations (one-hot softmax rows)."""
    assert D.diag_attn_qkv_cross()


def test_cta_pair_mma_primitives():
    assert D.diag_pairmma()


def test_decoder_launch_sequences_are_deterministic():
    """Back-to-back decoder kernel sequences reproduce their first pass bit for bit (tests/race_stress_diag.py: the race
    hunt that found the skipped parity wait in chain3's MMA warp; it fired in 1 - 4 % of the passes before the fix)."""
    import race_stress_diag
    assert race_stress_diag.main(150) == 0


def test_model_forward_is_deterministic(extractor, golden):
    ex, _ = extractor
    x = torch.from_numpy(golden("model_window")["input_spec"]).cuda()
    ref = [t.clone() for t in ex.model(x)]
    for _ in range(40):
        o = ex.model(x)
        assert all(torch.equal(a, b) for a, b in zip(o, ref))


@pytest.mark.parametrize("rates", [(44100, 16000), (48000, 16000), (22050, 16000), (8000, 16000), (16000, 16000)])
def test_ingest_vs_torchaudio(extractor, rates):
    """CUDA ingest (channel mean + sinc resampling, extractor.py:181-184) against torchaudio and the oracle: fp32, <= 1e-5."""
    import torchaudio

    from oracle import resample as oresample
    ex, sd = extractor
    orig, new = rates
    rng = np.random.default_rng(orig + 1)
    for channels, n in ((2, orig // 2 + 123), (1, 3 * orig + 5), (2, 7)):
        x = rng.uniform(-0.5, 0.5, (channels, n)).astype(np.float32)
        got = ex.engine.ingest(x, orig, new).cpu().numpy()
        ref = torchaudio.transforms.Resample(orig, new)(torch.mean(torch.from_numpy(x), dim=0)).numpy()
        assert got.shape == ref.shape, (channels, n)
        assert np.abs(got - ref).max() <= 1e-5
        assert np.abs(got - oresample.resample(x, orig, new)).max() <= 1e-5


def test_wav2feature_resamples_on_device(extractor, monkeypatch):
    """_wav2feature on a 44.1 kHz stereo file = reference ingest (torchaudio mean + Resample) + reference log-mel (oracle)."""
    import torchaudio

    from etude_b200 import synth
    from oracle import logmel as ologmel
    ex, sd = extractor
    rng = np.random.default_rng(5)
    mono = synth.tones(44100 * 2, 77).astype(np.float32)
    stereo = np.stack([mono + rng.normal(0, 1e-3, mono.shape).astype(np.float32), mono * 0.8])
    monkeypatch.setattr(torchaudio, "load", lambda p: (torch.from_numpy(stereo), 44100))
    feat = ex._wav2feature("x.wav").numpy()
    ref_wave = torchaudio.transforms.Resample(44100, 16000)(torch.mean(torch.from_numpy(stereo), dim=0)).numpy()
    ref = ologmel.logmel(ref_wave)
    assert feat.shape == ref.shape
    assert np.abs(feat - ref).max() <= 2e-3


def test_logmel_vs_golden(extractor):
    assert D.diag_logmel()


def test_logmel_edge_cases_and_errors(extractor):
    ex, _ = extractor
    from etude_b200 import _lib
    with pytest.raises(_lib.EtudeError):
        ex.wave_to_feature(np.zeros(1024, np.float32))      # reflect padding needs > n_fft/2 samples (torch errors too)
    f = ex.wave_to_feature(np.zeros(1025, np.float32))
    assert f.shape == (5, 256) and torch.all(f == float(np.log(np.float32(1e-8))))


def test_logmel_padding_rows_and_batch(extractor):
    ex, _ = extractor
    from etude_b200 import synth
    from oracle import logmel as ologmel
    waves = [synth.noise(256 * 700 + 3, 5), synth.tones(256 * 100, 6), synth.noise(256 * 512, 7)]
    n = [len(w) for w in waves]
    off = np.concatenate([[0], np.cumsum(n)])
    wave_dev = torch.from_numpy(np.concatenate(waves)).cuda()
    feat, row_off = ex.engine.logmel(wave_dev, off[:-1], n)
    feat = feat.cpu().numpy()
    for s, w in enumerate(waves):
        blk = feat[row_off[s] : row_off[s + 1]]
        t = 1 + len(w) // 256
        assert blk.shape[0] == (t + 511) // 512 * 512 + 64
        assert np.all(blk[:32] == -18.0) and np.all(blk[32 + t :] == -18.0)
        assert np.abs(blk[32 : 32 + t] - ologmel.logmel(w)).max() <= 1e-3


def test_notes_c_entry_equals_begin_fetch(extractor):
    """etude_notes (records in library-owned pinned memory: what a C caller binds) returns the same records as the
    begin/fetch pair the Python mirror uses (records straight into a caller-owned pinned array)."""
    import ctypes, torch
    from etude_b200 import _lib, engine
    ex, _ = extractor
    eng = ex.engine
    rng = np.random.default_rng(11)
    rows = [700, 1, 1536]
    off = np.concatenate([[0], np.cumsum(rows)])
    t = int(off[-1])
    rolls = [torch.from_numpy(rng.random((t, 88)).astype(np.float32)).to(ex.device) for _ in range(3)]
    vel = torch.from_numpy(rng.integers(0, 128, (t, 88)).astype(np.int8)).to(ex.device)
    a = eng.notes(rolls[0], rolls[1], rolls[2], vel, off[:-1].tolist(), rows, 0.5, 1.0, 0.5)
    out = ctypes.POINTER(_lib.Note)()
    counts = (ctypes.c_int64 * len(rows))()
    _lib.check(eng.lib.etude_notes(eng._h, engine._ptr(rolls[0]), engine._ptr(rolls[1]), engine._ptr(rolls[2]), engine._ptr(vel),
                                   _lib.i64_array(off[:-1].tolist()), _lib.i64_array(rows), len(rows), 21, 256 / 16000, 0.5, 1.0, 0.5,
                                   0, 0, ctypes.byref(out), counts, eng._stream()), "etude_notes")
    b = engine._take_notes(out, int(sum(counts)))
    assert list(counts) == [len(x) for x in a] and sum(counts) > 0
    assert np.array_equal(np.concatenate(a), b)
    assert all(x.flags.owndata is False and x.base is not None for x in a)   # views of the pinned result, no staging copy


@pytest.mark.parametrize("case", NOTE_CASES)
def test_notes_bit_exact_vs_golden(extractor, golden, case):
    ex, _ = extractor
    z = golden("notes")
    t_on, t_off, t_mpe = z[case + "__thr"]
    for mo, mv, ref in note_variants(z, case):
        got = ex._mpe2note(z[case + "__onset"], z[case + "__offset"], z[case + "__mpe"], z[case + "__velocity"],
                           thred_onset=t_on, thred_offset=t_off, thred_mpe=t_mpe, mode_velocity=mv, mode_offset=mo)
        assert got == ref, (case, mo, mv)


def test_notes_random_rolls_vs_oracle(extractor):
    """Property test at larger T: device notes == C oracle on seeded random rolls (plateaus, saturation, ragged T)."""
    ex, _ = extractor
    from oracle import notes as onotes
    rng = np.random.default_rng(5)
    for t in (1, 2, 3, 511, 4096):
        q = rng.integers(2, 40)
        on = (np.round(rng.random((t, 88)) * q) / q).astype(np.float32)
        off = np.minimum(1.0, rng.random((t, 88)) * 1.3).astype(np.float32)
        mpe = rng.random((t, 88)).astype(np.float32)
        vel = rng.integers(0, 128, (t, 88)).astype(np.int8)
        got = ex._mpe2note(on, off, mpe, vel, 0.5, 1.0, 0.5)
        assert got == onotes.mpe2note(on, off, mpe, vel, 0.5, 1.0, 0.5), t


def test_model_9tuple_vs_golden(extractor, golden):
    """Model_SPEC2MIDI.forward parity on the reference-generated window: sigmoid rolls max-abs <= 2e-2 (bf16 MMA
    operands, fp32 residual/LN/softmax), velocity argmax agreement >= 98 %."""
    ex, _ = extractor
    z = golden("model_window")
    o = ex.model(torch.from_numpy(z["input_spec"]).cuda())
    assert [tuple(t.shape) for t in o] == [(1, 512, 88)] * 3 + [(1, 512, 88, 128), (1, 512, 4, 88, 256)] + [(1, 512, 88)] * 3 + [(1, 512, 88, 128)]
    errs = {k: float(np.abs(o[i].cpu().numpy() - z[k]).max())
            for i, k in [(0, "onset_f"), (1, "offset_f"), (2, "mpe_f"), (5, "onset_t"), (6, "offset_t"), (7, "mpe_t")]}
    fr = z["frames"]
    e_att = float(np.abs(o[4][0, fr].cpu().numpy() - z["attention_sample"]).max())
    e_vf = float(np.abs(o[3][0, fr].cpu().numpy() - z["velocity_f_sample"]).max())
    e_vt = float(np.abs(o[8][0, fr].cpu().numpy() - z["velocity_t_sample"]).max())
    a_vf = float((o[3].argmax(3).cpu().numpy() == z["velocity_f_argmax"]).mean())
    a_vt = float((o[8].argmax(3).cpu().numpy() == z["velocity_t_argmax"]).mean())
    # how often a threshold decision of extract() (0.5 on onset / mpe) flips against the reference
    flips = {k: float(((o[i].cpu().numpy() >= 0.5) != (z[k] >= 0.5)).mean()) for i, k in [(5, "onset_t"), (7, "mpe_t")]}
    report("model_9tuple_vs_reference", **{"maxabs_" + k: v for k, v in errs.items()}, attention_maxabs=e_att,
           vel_logits_f_maxabs=e_vf, vel_logits_t_maxabs=e_vt, vel_logit_scale=float(np.abs(z["velocity_t_sample"]).max()),
           vel_argmax_f_agree=a_vf, vel_argmax_t_agree=a_vt, onset_t_flip_rate=flips["onset_t"], mpe_t_flip_rate=flips["mpe_t"])
    for k, v in errs.items():
        assert v <= 2e-2, (k, v)
    assert e_att <= 5e-3
    assert e_vf <= 0.15 and e_vt <= 0.15   # fp32 logits of |ref| <= ~2.6 (margin on record in profiles/r2_parity_margins.txt)
    assert a_vf >= 0.98 and a_vt >= 0.98


def test_encode_decode_split(extractor, golden):
    """_Spec2MIDI.encode / .decode (extractor.py:58-75): decode(encode(x)) is bit-identical to forward(x); the encoder output
    matches the reference's (sampled frames of the golden window)."""
    ex, _ = extractor
    z = golden("model_window")
    x = torch.from_numpy(z["input_spec"]).cuda()
    h = ex.model.encode(x)
    assert tuple(h.shape) == (1, 512, 256, 256) and h.dtype == torch.float32
    ref = z["enc_sample"]
    d = np.abs(h[0, z["frames"]].cpu().numpy() - ref).ravel()
    mean, p999, mx = float(d.mean()), float(np.sort(d)[int(0.999 * d.size)]), float(d.max())
    report("encoder_output_vs_reference", mean_abs=mean, p99_9=p999, maxabs=mx, scale=float(np.abs(ref).max()))
    # bf16 MMA operands by specification: the x16-scaled token embedding reaches |x| ~ 320, so the first layer's softmax is
    # near one-hot and a few tokens flip between almost-tied keys.  A CPU emulation of exactly these roundings (bf16 embedding
    # output, bf16 weights, bf16 layer outputs; fp32 everything else) gives mean 3.4e-3, p99.9 6.8e-2, max 0.35 on these frames;
    # the rolls downstream agree with the reference to 7e-3 (test_model_9tuple_vs_golden).
    assert mean <= 0.01 and p999 <= 0.15 and mx <= 1.0
    a, b = ex.model.decode(h), ex.model(x)
    for i in range(9):
        assert torch.equal(a[i], b[i]), i


def test_transcript_frequency_axis_only_mode(extractor, golden):
    """_transcript(mode != "combination") returns the four frequency-axis arrays only (extractor.py:236, 250-253)."""
    ex, _ = extractor
    z = golden("transcript")
    outs = ex._transcript(z["feature"], mode="single")
    full = ex._transcript(z["feature"])
    assert len(outs) == 4
    for a, b in zip(outs, full[:4]):
        assert a.dtype == b.dtype and np.array_equal(a, b)


def test_model_batch_independence(extractor, golden):
    """Per-window results must not depend on batch composition (SURVEY 8(e)): B=3 rows equal B=1 runs bit for bit."""
    ex, _ = extractor
    z = golden("model_window")
    x = torch.from_numpy(z["input_spec"]).cuda()
    xs = torch.cat([x, x.flip(2), x * 0.5 - 3.0], 0)
    ob = ex.model(xs)
    for b in range(3):
        o1 = ex.model(xs[b : b + 1])
        for i in (0, 1, 2, 5, 6, 7):
            assert torch.equal(ob[i][b], o1[i][0]), (b, i)


def test_transcript_vs_golden(extractor, golden):
    ex, _ = extractor
    z = golden("transcript")
    outs = ex._transcript(z["feature"])
    names = ["onset_A", "offset_A", "mpe_A", "velocity_A", "onset_B", "offset_B", "mpe_B", "velocity_B"]
    vals = {}
    for n, a in zip(names, outs):
        assert a.shape == z[n].shape == (1024, 88) and a.dtype == z[n].dtype, n
        vals[n] = float((a == z[n]).mean()) if a.dtype == np.int8 else float(np.abs(a - z[n]).max())
    report("transcript_vs_reference (maxabs of the rolls, agreement of the int8 velocities)", **vals)
    for n, a in zip(names, outs):
        if a.dtype == np.int8:
            assert vals[n] >= 0.98, n
        else:
            assert vals[n] <= 2e-2, n


def test_extract_json_and_extract_many(extractor, golden, tmp_path, monkeypatch):
    """extract() writes the reference's JSON format; extract_many == extract per song; note F1 vs oracle reported."""
    import json

    import torchaudio

    from etude_b200 import synth
    ex, sd = extractor
    waves = [synth.tones(256 * 600 + 19, 21), synth.noise(256 * 300, 22)]
    many = ex.extract_many(waves)
    for i, w in enumerate(waves):
        monkeypatch.setattr(torchaudio, "load", lambda p, w=w: (torch.from_numpy(w)[None], 16000))
        out = tmp_path / f"extract{i}.json"
        ex.extract("x.wav", str(out))
        notes = json.loads(out.read_text())
        assert all(list(n.keys()) == ["onset", "offset", "pitch", "velocity"] for n in notes)
        want = [{"onset": n["onset"], "offset": n["offset"], "pitch": n["pitch"], "velocity": n["velocity"]}
                for n in many[i] if not (n["offset"] - n["onset"] < 0.08)]
        assert notes == want
    # golden clip: our rolls -> our notes vs the reference's notes (not bit-exact by design: rolls differ by ~1e-2)
    z = golden("transcript")
    ref = unpack_notes(z, "notes")
    key = lambda n: (n["pitch"], round(n["onset"] / 0.016))
    a, b = {key(n) for n in many[0]}, {key(n) for n in ref}
    f1 = 2 * len(a & b) / (len(a) + len(b))
    report("transcript_clip_notes_vs_reference", notes_ours=len(many[0]), notes_reference=len(ref), onset_f1=f1)
    assert f1 >= 0.90


def test_config1_clip30_extract_vs_reference(extractor, golden, tmp_path, monkeypatch):
    """BASELINE config 1 / the hand-off of config 5: `extract()` on the 30 s noise clip against the reference's own
    `extract()` (tests/golden/clip30.npz, generated by oracle/gen_golden.py): rolls within 2e-2, velocity argmax agreement,
    extract.json schema / ordering, and note agreement with the reference's extract.json."""
    import json

    import torchaudio

    from etude_b200 import synth
    ex, sd = extractor
    z = golden("clip30")
    wave = synth.noise(480000, 1234)
    monkeypatch.setattr(torchaudio, "load", lambda p: (torch.from_numpy(wave)[None], 16000))
    feat = ex._wav2feature("x.wav")
    assert feat.shape[0] == int(z["n_frames"][0]) == 1876
    outs = ex._transcript(feat)
    assert all(o.shape == (2048, 88) for o in outs)
    errs = {}
    for name, got in zip(("onset_B", "offset_B", "mpe_B"), outs[4:7]):
        err = np.abs(got - z[name].astype(np.float32)).max()
        errs["maxabs_" + name] = float(err)
        assert err <= 2e-2 + 1e-3, (name, err)          # + fp16 storage of the fixture
    agree = (outs[7] == z["velocity_B"]).mean()
    assert agree >= 0.98, agree
    out = tmp_path / "extract.json"
    ex.extract("x.wav", str(out))
    notes = json.loads(out.read_text())
    assert all(list(n.keys()) == ["onset", "offset", "pitch", "velocity"] for n in notes)
    assert all(n["offset"] - n["onset"] >= 0.08 for n in notes)
    assert [n["onset"] for n in notes] == sorted(n["onset"] for n in notes)
    ref = unpack_notes(z, "json")
    key = lambda n: (n["pitch"], round(n["onset"] / 0.016))
    a, b = {key(n) for n in notes}, {key(n) for n in ref}
    f1 = 2 * len(a & b) / max(1, len(a) + len(b))
    report("config1_clip30_extract_vs_reference", **errs, velocity_agree=float(agree), notes_ours=len(notes), notes_reference=len(ref), onset_f1=f1)
    assert f1 >= 0.8


def test_full_size_song_properties():
    """BASELINE config 3 size (one 4-minute song = 30 windows, window batch 32): size-independent properties.
    (a) the device note stage is bit-exact against the oracle's C restatement when both read the SAME device rolls
        (365 k notes at random-init density); (b) the whole path is deterministic run to run; (c) rolls do not depend on
        how the windows are batched (batch 32 vs batch 7)."""
    from etude_b200 import synth
    from oracle import notes as onotes
    ex32, sd = D.make_extractor(max_windows=32)
    wave = synth.noise(16000 * 240, 1234)
    notes, rolls, row_off, rows = ex32.extract_many([wave], return_rolls=True)
    assert rows == [15360] and len(notes) == 1
    host = [r.cpu().numpy() for r in rolls]
    ref = onotes.mpe2note(host[0], host[1], host[2], host[3], thred_onset=0.5, thred_offset=1.0, thred_mpe=0.5)
    assert len(ref) > 100000
    assert notes[0] == ref                                   # (a) bit-exact, float repr included
    again, rolls2, _, _ = ex32.extract_many([wave], return_rolls=True)
    assert all(torch.equal(a, b) for a, b in zip(rolls, rolls2)) and again[0] == notes[0]      # (b)
    ex7, _ = D.make_extractor(max_windows=7)
    _, rolls7, _, _ = ex7.extract_many([wave], return_rolls=True)
    assert all(torch.equal(a, b) for a, b in zip(rolls, rolls7))                                # (c)


def test_extract_many_grouping_independence(extractor):
    """The three-stream group pipeline of extract_many returns the same records whatever the group / notes-batch sizes."""
    from etude_b200 import synth
    ex, sd = extractor
    waves = [synth.tones(256 * 700 + 3, 31), synth.noise(256 * 300, 32), synth.noise(256 * 1100 + 77, 33), synth.tones(256 * 20, 34),
             synth.noise(256 * 513, 35)]
    one = ex.extract_many(waves, as_dicts=False, group_songs=None)
    for g, nb in ((1, 1), (2, 2), (4, 12), (2, 3), (1, 2)):
        got = ex.extract_many(waves, as_dicts=False, group_songs=g, notes_batch=nb)
        assert len(got) == len(one)
        for a, b in zip(got, one):
            assert a.tobytes() == b.tobytes(), f"group_songs={g} notes_batch={nb}"


def test_smoke_entry():
    import __graft_entry__ as g
    g.smoke()


def test_rolls_with_outlier_weights_vs_oracle(tmp_path):
    """The parity goldens use default-initialised weights.  A trained checkpoint has outlier LayerNorm gains, larger FFN
    weights and more confident heads, which stress the bf16 activation stream between the kernels (ADVICE round 1).  This
    perturbs the seeded weights that way (no checkpoint can be downloaded here) and holds one window of the device path
    against the fp32 oracle on the same weights; the margins go on record like every other parity number."""
    from etude_b200 import AMTAPC_Extractor, ExtractorConfig, synth
    from oracle import logmel as ologmel, model as omodel
    sd = {k: v.clone() for k, v in omodel.init_state_dict(0).items()}
    g = torch.Generator().manual_seed(99)
    for k, v in sd.items():
        if k.endswith("layer_norm.weight"):
            idx = torch.randperm(256, generator=g)[:6]
            v[idx] = torch.tensor([6.0, 5.0, 4.0, 0.05, 3.0, 8.0])
        elif k.endswith("layer_norm.bias"):
            v += 0.5 * torch.randn(256, generator=g)
        elif "positionwise_feedforward" in k and k.endswith("weight"):
            v *= 1.6
        elif ("fc_onset" in k or "fc_offset" in k or "fc_mpe" in k or "fc_velocity" in k) and k.endswith("weight"):
            v *= 2.0
    path = tmp_path / "outlier_sd.pth"
    torch.save(sd, path)
    ex = AMTAPC_Extractor(ExtractorConfig(), path, device="cuda:0", max_windows=2)
    wave = synth.tones(256 * 500 + 7, 5)                     # one window
    feat_ref = ologmel.logmel(wave)
    ref = omodel.transcript(sd, feat_ref, batch=1)           # 8 arrays
    got = ex._transcript(ex.wave_to_feature(wave).cpu().numpy())
    names = ["onset_A", "offset_A", "mpe_A", "velocity_A", "onset_B", "offset_B", "mpe_B", "velocity_B"]
    vals = {n: (float((a == r).mean()) if a.dtype == np.int8 else float(np.abs(a - r).max())) for n, a, r in zip(names, got, ref)}
    spread = {n: float(np.abs(r - 0.5).max()) for n, r in zip(names, ref) if r.dtype != np.int8}
    report("rolls_with_outlier_weights_vs_oracle (maxabs / int8 agreement)", **vals, ref_spread_onset_B=spread["onset_B"])
    for n in names:
        if n.startswith("velocity"):
            # argmax over 128 logits that random heads leave almost flat: measured 0.934 (A) / 1.0 (B) on this input
            assert vals[n] >= 0.90, (n, vals[n])
        else:
            assert vals[n] <= 2e-2, (n, vals[n])     # the same contract as the default-initialised goldens (measured <= 8.2e-3)
