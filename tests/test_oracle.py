"""The C oracle (oracle/melgan_oracle.c) against the reference's own outputs (tests/golden)."""
import numpy as np
import pytest

import cases
from conftest import rel_errors
from melgan_multi_b200 import synth
from oracle import cport

TOL = 2e-5  # fp32 reference (oneDNN summation order) vs double-accumulating oracle


@pytest.fixture(scope="module")
def gen_folded():
    return cport.fold_generator(synth.generator_state(1234))


@pytest.fixture(scope="module")
def msd_folded():
    return cport.fold_discriminators(synth.discriminator_state(4321))


def test_primitive_ops_match_reference(golden):
    for key, kind, prm, x, w, b in cases.op_inputs():
        if kind == "conv":
            y = cport.conv1d(x, w, b, *prm)
        elif kind == "convT":
            y = cport.conv_transpose1d(x, w, b, *prm)
        else:
            y = cport.avgpool1d(x, *prm)
        ref = golden[key]
        assert y.shape == ref.shape, key
        m, l2 = rel_errors(y, ref)
        assert m < 1e-5 and l2 < 1e-5, (key, m, l2)


def test_weight_norm_fold_matches_reference_hook(golden):
    st = synth.generator_state(1234)
    for key, name in (("fold_conv_pre_every8th", "conv_pre"), ("fold_ups3", "ups.3"),
                      ("fold_res2_c1_1", "resblocks.2.convs1.1")):
        for w in (cport.fold_weight_norm(st[name + ".weight_g"], st[name + ".weight_v"]),
                  synth.fold_weight_norm(st[name + ".weight_g"], st[name + ".weight_v"])):
            if name == "conv_pre":  # the fixture keeps every 8th output channel and the norms of all of them
                norms = np.sqrt((w.astype(np.float64) ** 2).reshape(len(w), -1).sum(axis=1))
                np.testing.assert_allclose(norms, golden["fold_conv_pre_norms"], rtol=2e-6)
                w = w[::8]
            np.testing.assert_allclose(w, golden[key], rtol=2e-6, atol=1e-8)


@pytest.mark.parametrize("case", cases.GEN_CASES)
def test_generator_matches_reference(golden, gen_folded, case):
    B, T, seed, realistic = case
    ws, bs = gen_folded
    y = cport.generator_forward(ws, bs, synth.mel_input(B, T, seed, realistic))
    ref = golden[cases.gen_key(*case)]
    assert y.shape == ref.shape == (B, 1, 256 * T)
    m, l2 = rel_errors(y, ref)
    assert m < TOL and l2 < TOL, (case, m, l2)


def test_generator_stage_taps_match_reference(golden, gen_folded):
    ws, bs = gen_folded
    y, stages = cport.generator_forward(ws, bs, synth.mel_input(1, 3, 5), want_stages=True)
    for i, s in enumerate(stages):
        m, l2 = rel_errors(s, golden["gen_taps_T3_s5_%d" % i])
        assert m < TOL and l2 < TOL, (i, m, l2)
    assert rel_errors(y, golden["gen_taps_T3_s5_audio"])[0] < TOL


def test_generator_long_utterance_matches_reference(golden, gen_folded):
    ws, bs = gen_folded
    y = cport.generator_forward(ws, bs, synth.mel_input(1, 1000, 0)).reshape(-1)
    scale = np.abs(golden["gen_T1000_mid"]).max()
    assert np.abs(y[:4096] - golden["gen_T1000_head"]).max() < TOL * scale
    assert np.abs(y[128000 - 2048:128000 + 2048] - golden["gen_T1000_mid"]).max() < TOL * scale
    assert np.abs(y[-4096:] - golden["gen_T1000_tail"]).max() < TOL * scale
    bs_ = y.astype(np.float64).reshape(250, 1024).sum(axis=1)
    assert np.abs(bs_ - golden["gen_T1000_blocksum"]).max() < 1024 * TOL * scale


@pytest.mark.parametrize("case", cases.MSD_CASES)
def test_msd_matches_reference(golden, msd_folded, case):
    B, L, seed = case
    y = synth.audio_input(B, L, seed)
    y_hat = synth.audio_input(B, L, seed + 7)
    rs, gs, frs, fgs = cport.msd_forward(msd_folded, y, y_hat)
    tag = "msd_B%d_L%d_s%d" % (B, L, seed)
    for i in range(3):
        for nm, lg, fm in (("r", rs, frs), ("g", gs, fgs)):
            ref = golden["%s_logit_%s%d" % (tag, nm, i)]
            assert lg[i].shape == ref.shape
            m, l2 = rel_errors(lg[i], ref)
            assert m < 5e-5 and l2 < 5e-5, (i, nm, m, l2)
            for j in range(7):
                a = fm[i][j]
                assert tuple(golden["%s_fmap_%s%d_%d_shape" % (tag, nm, i, j)]) == a.shape
                head = golden["%s_fmap_%s%d_%d_head" % (tag, nm, i, j)]
                m, _ = rel_errors(a[:, :4, :48], head)
                assert m < 5e-5, (i, j, nm, m)
                s = golden["%s_fmap_%s%d_%d_sum" % (tag, nm, i, j)]
                assert abs(np.abs(a.astype(np.float64)).sum() - s[1]) < 1e-5 * s[1]


def test_torch_cpu_port_matches_reference(golden):
    """oracle/torch_port.py (bench.py's CPU baseline) against the reference's outputs."""
    import torch
    from oracle import torch_port
    ws, bs = torch_port.fold_state(synth.generator_state(1234))
    for case in (cases.GEN_CASES[1], cases.GEN_CASES[4]):
        y = torch_port.generator_forward(ws, bs, torch.from_numpy(synth.mel_input(*case))).numpy()
        m, l2 = rel_errors(y, golden[cases.gen_key(*case)])
        assert m < TOL and l2 < TOL, (case, m, l2)


def test_torch_cpu_port_matches_reference_at_config2():
    """The timed CPU arm of bench.py (oracle/torch_port.generator_forward_reference: per-forward weight-norm + the conv
    graph) at BASELINE config 2 full size against the unmodified reference's output (tests/golden/config2_outputs.npz)."""
    import os
    import torch
    from oracle import torch_port
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "config2_outputs.npz"))
    params = torch_port.reference_state(synth.generator_state(1234))
    for realistic in (False, True):
        y = torch_port.generator_forward_reference(params, torch.from_numpy(synth.mel_input(64, 32, 0, realistic))).numpy()
        key = "gen_B64_T32_s0_r%d" % int(realistic)
        ys, bsum = cases.config2_digest(y, g["sample_index"])
        m, l2 = rel_errors(ys, g[key + "_sample"])
        assert m < TOL and l2 < TOL, (realistic, m, l2)
        scale = float(g[key + "_absmax"])
        assert np.abs(bsum - g[key + "_blocksum"]).max() < cases.CONFIG2_BLOCK * TOL * scale, realistic


def test_mel_oracle_stft_matches_scipy_and_filterbank_properties():
    """oracle/mel_oracle.py restates librosa (absent here; parity of this row is unpinned by any reference fixture): its STFT
    magnitudes against scipy.signal.stft (an independent implementation), its filter bank against closed-form properties
    of Slaney-normalised triangles on the Slaney mel scale."""
    import scipy.signal
    from oracle import mel_oracle as mo
    rs = np.random.RandomState(5)
    y = (rs.uniform(-1, 1, 8192) * 0.7).astype(np.float32)
    yp = np.pad(y, (384, 384))
    S = mo.stft_magnitude(yp, 1024, 256, 1024)
    win = scipy.signal.get_window("hann", 1024, fftbins=True)
    _, _, Z = scipy.signal.stft(yp, window=win, nperseg=1024, noverlap=768, boundary=None, padded=False, scaling="spectrum")
    assert S.shape == (513, 32) and np.abs(S - np.abs(Z) * win.sum()).max() <= 1e-6 * S.max()
    w = mo.mel_filterbank(22050, 1024, 80, 55, 9000, norm=1).astype(np.float64)
    assert w.shape == (80, 513) and (w >= 0).all() and ((w > 0).sum(axis=0) <= 2).all()
    freqs = np.linspace(0, 11025, 513)
    edges = mo.mel_to_hz(np.linspace(mo.hz_to_mel(55), mo.hz_to_mel(9000), 82))
    assert abs(mo.hz_to_mel(1000.0) - 15.0) < 1e-12 and abs(mo.mel_to_hz(mo.hz_to_mel(4321.0)) - 4321.0) < 1e-9
    for m in (0, 17, 40, 79):
        nz = np.nonzero(w[m])[0]
        assert edges[m] < freqs[nz[0]] and freqs[nz[-1]] < edges[m + 2]           # support = (f_m, f_m+2)
        assert abs(freqs[w[m].argmax()] - edges[m + 1]) <= 11025 / 512              # peak at the centre frequency
        assert w[m].max() <= 2.0 / (edges[m + 2] - edges[m]) + 1e-12                # Slaney: triangle of unit AREA in Hz
    wide = [m for m in range(80) if edges[m + 2] - edges[m] > 150]
    area = (w[wide].sum(axis=1) * (11025 / 512))
    assert np.abs(area - 1).max() < 0.05
    un = mo.mel_filterbank(22050, 1024, 80, 55, 9000, norm=None)
    inner = (freqs > edges[1]) & (freqs < edges[80])
    assert np.abs(un[:, inner].sum(axis=0) - 1).max() < 1e-5                         # un-normalised triangles partition unity
    out = mo.mel_spectrogram(y)
    assert out.shape == (80, 32) and np.isfinite(out).all()
    assert np.allclose(mo.mel_spectrogram(np.zeros(4096, np.float32)), np.log(1e-5))  # silence sits on the clip floor
