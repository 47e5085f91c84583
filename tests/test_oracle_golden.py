"""CPU: the oracle restatement (oracle/ref_megatts2.py) against the fixtures produced by the
REAL reference (tests/golden/*.npz, written by oracle/make_golden.py in the build container).
This is what pins the oracle; the GPU parity tests then compare the CUDA path to the oracle
and to the same fixtures."""
import json

import numpy as np
import os

import pytest
import torch

from oracle import ref_megatts2 as R
from oracle import weights

from conftest import GOLDEN



def test_state_dict_keys_match_reference():
    with open(os.path.join(GOLDEN, "state_dict_keys.json")) as f:
        ref = json.load(f)
    for name, spec in (("G", weights.g_spec()), ("plm", weights.plm_spec()), ("adm", weights.adm_spec())):
        assert list(spec.keys()) == list(ref[name].keys()), name
        assert {k: list(v) for k, v in spec.items()} == ref[name], name
    assert len(ref["G"]) == 840


def test_mel_frontend(golden):
    g = golden("mel_frontend")
    out = R.mel_spectrogram(g["wav"])
    assert out.shape == g["mel"].shape == (3, 80, 16)
    assert (out - g["mel"]).abs().max() < 2e-5
    # the silent clip sits on the clamp floor log(1e-5)
    assert torch.allclose(out[2], torch.full_like(out[2], -11.512925), atol=1e-4)


def test_filterbank_vs_torchaudio():
    ta = pytest.importorskip("torchaudio")
    fb = ta.functional.melscale_fbanks(513, 0.0, 8000.0, 80, 16000, norm="slaney", mel_scale="slaney")
    mine = R.slaney_fbanks()
    assert (mine - fb).abs().max() < 2e-7
    assert int((mine != 0).sum()) == 1001


def test_vqpe_c1_bit_exact(golden, weights_cpu):
    g = golden("vqpe")
    sd = R.SD(weights_cpu("g"), "vqpe.")
    zq, commit, vql, codes, ze = R.vqpe_forward(sd, g["mel1"], weights.G_CFG)
    assert torch.equal(codes, g["codes1"]) and codes.shape == (1, 1, 16)
    assert (zq - g["zq1"]).abs().max() <= 1e-5
    assert (ze - g["ze1"]).abs().max() <= 1e-4
    assert abs(float(vql) - float(g["vq_loss1"])) < 1e-4
    zq2, _, _, codes2, _ = R.vqpe_forward(sd, g["mel2"], weights.G_CFG)
    assert torch.equal(codes2, g["codes2"]) and zq2.shape == (2, 61, 256)


def test_vq_search(golden, weights_cpu):
    g = golden("vq_search")
    embed = weights_cpu("g")["vqpe.vq.vq.layers.0._codebook.embed"]
    assert torch.equal(R.vq_quantize(g["x"], embed), g["idx"])


def test_encoders(golden, weights_cpu):
    g = golden("encoder")
    y = R.encoder(R.SD(weights_cpu("g"), "mrte.phone_encoder."), g["x_phone"], 8, 2, True)
    assert (y - g["y_phone"]).abs().max() < 2e-4
    psd = R.SD(weights_cpu("plm"), "plm.")
    lens = torch.tensor([7, 7], dtype=torch.int32)
    assert (R.encoder(psd, g["x_plm"], 12, 16, False, lens=lens, causal=True) - g["y_plm_causal"]).abs().max() < 5e-4
    assert (R.encoder(psd, g["x_plm"], 12, 16, False) - g["y_plm_nomask"]).abs().max() < 5e-4


def test_mrte(golden, weights_cpu):
    g = golden("mrte")
    tc, ctx, _ = R.mrte_tc_latent(R.SD(weights_cpu("g"), "mrte."), g["phone"], g["mel"], weights.G_CFG)
    assert (tc - g["tc_latent"]).abs().max() < 2e-4
    assert (ctx - g["mel_context"]).abs().max() < 2e-4
    assert float(tc.min()) >= 0.0


def test_length_regulator_reference_case(golden):
    g = golden("length_regulator")
    y = R.length_regulate(g["x"], g["d"])
    assert y.shape == (2, 11, 128)          # the reference's own assertion (modules/mrte.py:187-194)
    assert torch.equal(y, g["y"])


def test_adm(golden, weights_cpu):
    g = golden("adm")
    dur, raw = R.adm_infer(R.SD(weights_cpu("adm")), g["tc_latent"], weights.ADM_CFG, return_raw=True)
    assert torch.equal(dur, g["dur"])
    assert (raw - g["raw"]).abs().max() < 2e-3
    fwd, _ = R.adm_forward(R.SD(weights_cpu("adm")), g["tc_latent"], g["dtok"],
                           torch.tensor([10, 10], dtype=torch.int32), weights.ADM_CFG)
    assert (fwd - g["fwd"]).abs().max() < 2e-3


def test_plm(golden, weights_cpu):
    g = golden("plm")
    ids, lg = R.plm_infer(R.SD(weights_cpu("plm")), g["tc8"], weights.PLM_CFG, return_logits=True)
    assert torch.equal(ids, g["ids"])
    assert (lg - g["logits"]).abs().max() < 2e-3
    assert ids.unique().numel() >= 8        # the fixture is not degenerate


def test_causal_decode_next_row(golden, weights_cpu):
    """SURVEY.md 8f-1: the opt-in causal decode's checker vs the fixture produced by looping the REAL reference's
    teacher-forced forward (causal=True).  It is a different function from infer() - the ids differ."""
    g = golden("causal_decode")
    ids, lg = R.plm_infer_causal(R.SD(weights_cpu("plm")), g["tc8"], weights.PLM_CFG, return_logits=True)
    assert torch.equal(ids, g["plm_ids"])
    assert (lg - g["plm_logits"]).abs().max() < 2e-3
    assert not torch.equal(ids, golden("plm")["ids"])
    dur, raw = R.adm_infer_causal(R.SD(weights_cpu("adm")), g["tc_latent"], weights.ADM_CFG, return_raw=True)
    assert torch.equal(dur, g["adm_dur"])
    assert (raw - g["adm_raw"]).abs().max() < 2e-3


def test_e2e_body(golden, weights_cpu):
    g = golden("e2e")
    o = R.synthesize(weights_cpu("g"), weights_cpu("plm"), weights_cpu("adm"), weights_cpu("hifigan"), g["phone"],
                     g["mel_prompt"], (weights.G_CFG, weights.PLM_CFG, weights.ADM_CFG, weights.HIFIGAN_CFG),
                     forced_durations=g["dt_used"])
    assert torch.equal(o["dt"], g["dt"]) and torch.equal(o["p_codes"], g["p_codes"])
    assert (o["mel"] - g["mel"]).abs().mean() < 1e-4
    assert (o["wav"] - g["wav_oracle"]).abs().max() < 1e-5


def test_hifigan_shape_and_regression(golden, weights_cpu):
    g = golden("hifigan")
    wav = R.hifigan_generator(weights_cpu("hifigan"), g["mel"], weights.HIFIGAN_CFG)
    assert wav.shape == (2, 1, 256 * (12 + 10))
    assert (wav - g["wav"]).abs().max() < 1e-5
    n = sum(v.numel() for v in weights_cpu("hifigan").values())
    assert n == 13_926_017                 # HiFi-GAN V1 generator size (SURVEY.md §8c)


def test_reference_loads_oracle_weights_strict(weights_cpu):
    """The real reference accepts the oracle's state dicts with strict=True: the same keys, each with the shape of the
    reference's own tensor.  The reference's layout is the one oracle/make_golden.py recorded from its modules."""
    with open(os.path.join(GOLDEN, "state_dict_keys.json")) as f:
        ref = json.load(f)
    for name, sd in (("G", weights_cpu("g")), ("plm", weights_cpu("plm")), ("adm", weights_cpu("adm"))):
        assert sorted(sd) == sorted(ref[name]), name
        assert {k: list(v.shape) for k, v in sd.items()} == ref[name], name
        assert all(v.dtype == torch.float32 for v in sd.values()), name


def test_c_oracle_vq_matches_reference_fixture(golden, weights_cpu):
    """the plain-C VQ restatement (oracle/vq_argmin.c) against the reference's indices"""
    import ctypes
    import subprocess
    from conftest import ROOT
    so = os.path.join(ROOT, "oracle", "_build", "libvq_oracle.so")
    if not os.path.exists(so):
        os.makedirs(os.path.dirname(so), exist_ok=True)
        subprocess.check_call(["gcc", "-O2", "-shared", "-fPIC", "-o", so, os.path.join(ROOT, "oracle", "vq_argmin.c")])
    lib = ctypes.CDLL(so)
    g = golden("vq_search")
    x = g["x"].contiguous()
    embed = weights_cpu("g")["vqpe.vq.vq.layers.0._codebook.embed"].contiguous()
    idx = torch.empty(x.shape[0], dtype=torch.int64)
    lib.vq_argmin_oracle(ctypes.c_void_p(x.data_ptr()), ctypes.c_void_p(embed.data_ptr()), ctypes.c_int64(x.shape[0]),
                         ctypes.c_int(256), ctypes.c_int(1024), ctypes.c_void_p(idx.data_ptr()))
    mism = idx != g["idx"]
    assert bool((g["gap64"][mism] < 2e-4).all())      # only genuine fp32 near-ties may differ
    assert torch.equal(idx[:512], g["idx"][:512])


def test_audio_front_end_restatement_vs_torchaudio():
    """8f-3: the oracle's polyphase resampler == torchaudio.functional.resample (the published definition it restates),
    and the product's host-built fp32 filter table is bit-identical to torchaudio's own."""
    import math
    import torchaudio
    from torchaudio.functional.functional import _get_sinc_resample_kernel
    from megatts2_b200 import audio
    from oracle import ref_audio
    g = torch.Generator().manual_seed(11)
    for o, n in ((44100, 16000), (48000, 16000), (22050, 16000), (24000, 16000), (8000, 16000)):
        x = torch.rand(7000, generator=g) * 2 - 1
        ref = torchaudio.functional.resample(x[None], o, n, resampling_method="sinc_interp_kaiser", **ref_audio.KAISER_BEST)[0]
        got = ref_audio.resample(x.numpy(), o, n)
        assert got.shape == tuple(ref.shape)
        assert np.abs(got - ref.numpy()).max() < 5e-5
        k, w = _get_sinc_resample_kernel(o, n, math.gcd(o, n), resampling_method="sinc_interp_kaiser", **audio.KAISER_BEST)
        up, down, width, h = audio.resample_table(o, n, **audio.KAISER_BEST)
        assert width == w and np.array_equal(h, k[:, 0].numpy())
    y = ref_audio.peak_normalize(np.array([0.25, -0.5, 0.125], dtype=np.float32))
    assert np.array_equal(y, np.array([0.5, -1.0, 0.25], dtype=np.float32))
    assert np.array_equal(ref_audio.peak_normalize(np.zeros(4, dtype=np.float32)), np.zeros(4, dtype=np.float32))


def test_wav_framing_round_trip(tmp_path):
    """The host half of the wav writer / reader: RIFF framing of float32 and int16 payloads, readable by the stdlib."""
    import wave
    from megatts2_b200 import audio
    x = (np.random.RandomState(0).rand(1234).astype(np.float32) * 2 - 1)
    pf = tmp_path / "f.wav"
    pf.write_bytes(audio.wav_bytes(x, 16000, "PCM_F"))
    y, sr = audio.read_wav(str(pf))
    assert sr == 16000 and np.array_equal(x, y)
    q = np.clip(np.rint(x * 32768.0), -32768, 32767).astype(np.int16)
    pi = tmp_path / "i.wav"
    pi.write_bytes(audio.wav_bytes(q, 22050, "PCM_S"))
    with wave.open(str(pi)) as w:
        assert (w.getnchannels(), w.getsampwidth(), w.getframerate(), w.getnframes()) == (1, 2, 22050, 1234)
        assert w.readframes(1234) == q.tobytes()
    y2, sr2 = audio.read_wav(str(pi))
    assert sr2 == 22050 and np.array_equal(y2, q.astype(np.float32) / 32768.0)


def test_vq_train_restatement_replays_reference_fixture():
    """oracle/ref_vq_train.py reproduces the REAL reference's train-mode VectorQuantization (three steps: k-means init,
    dead-code expiry, EMA update, straight-through + commitment loss, backward) from the recorded draws."""
    import numpy as np
    from oracle import ref_vq_train as RV
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "vq_train.npz"))
    K, D, B, N, iters, steps = (int(v) for v in g["meta"])
    cb = RV.Codebook(D, K, kmeans_iters=iters, decay=float(g["decay"]), threshold_ema_dead_code=2)
    for s in range(steps):
        x = torch.from_numpy(g[f"s{s}_x"]).requires_grad_(True)
        kw = {"expire_pick": torch.from_numpy(g[f"s{s}_expire_pick"])}
        if s == 0:
            kw["init_indices"] = torch.from_numpy(g["s0_init_indices"])
        q, ind, loss, used = RV.vq_forward_train(cb, x, float(g["commitment_weight"]), **kw)
        ((q * torch.from_numpy(g[f"s{s}_wq"])).sum() + 3.0 * loss.sum()).backward()
        assert used == bool(g[f"s{s}_expired"])
        assert torch.equal(ind, torch.from_numpy(g[f"s{s}_ind"]))
        for name, got in (("q", q), ("loss", loss), ("gx", x.grad), ("embed", cb.embed), ("embed_avg", cb.embed_avg),
                          ("cluster_size", cb.cluster_size)):
            assert (got.detach() - torch.from_numpy(g[f"s{s}_{name}"])).abs().max().item() <= 1e-6, (s, name)
