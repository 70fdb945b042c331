"""GPU parity: the sm_100a generator (tcgen05 split-bf16 tensor-core kernels, through the C ABI) against the C oracle and
the reference's golden outputs.  Tolerance (BASELINE.json north_star): 1e-3 relative fp32; asserted much tighter: 1e-4
(3-pass split-bf16, measured ~1e-5).  (The fp32 SIMT second implementation is cross-checked in
tests/test_simt_crosscheck_gpu.py from its own test-only library.)"""
import os

import numpy as np
import pytest
import torch

import cases
from conftest import rel_errors
from melgan_multi_b200 import engine, synth
from oracle import cport

pytestmark = pytest.mark.gpu
TOL = 1e-4


@pytest.fixture(scope="module")
def state():
    return synth.generator_state(1234)


@pytest.fixture(scope="module")
def host_engine(state):
    e = engine.GeneratorHost(2, 33)
    e.load_state(state)
    yield e
    e.close()


@pytest.fixture(scope="module")
def gen_module(state):
    from melgan_multi_b200 import models
    g = models.Generator()
    g.load_state_dict({k: torch.from_numpy(v) for k, v in state.items()})
    return g.cuda().eval()


@pytest.fixture(scope="module")
def folded(state):
    return cport.fold_generator(state)


def test_device_is_supported():
    engine.check(engine.lib().mg_device_check())


@pytest.mark.parametrize("case", cases.GEN_CASES)
def test_host_engine_matches_golden(golden, host_engine, case):
    B, T, seed, realistic = case
    y = host_engine.forward(synth.mel_input(B, T, seed, realistic))
    ref = golden[cases.gen_key(*case)]
    assert y.shape == ref.shape
    m, l2 = rel_errors(y, ref)
    assert m < TOL and l2 < TOL, (case, m, l2)


def test_module_forward_matches_golden_and_stage_taps(golden, gen_module):
    x = torch.from_numpy(synth.mel_input(1, 3, 5)).cuda()
    with torch.no_grad():
        y = gen_module(x)
    torch.cuda.synchronize()
    m, l2 = rel_errors(y.cpu().numpy(), golden["gen_taps_T3_s5_audio"])
    assert m < TOL and l2 < TOL, (m, l2)
    with pytest.raises(engine.EngineError):  # the default chain never writes the ResBlock outputs to memory
        gen_module._dev.stage_output(1, 1, 3)
    # the per-stage taps exist in the unfused chain (one kernel per ConvT / ResBlock)
    engine.check(engine.lib().mg_gen_set_pipeline(0))
    try:
        with torch.no_grad():
            y0 = gen_module(x)
        torch.cuda.synchronize()
        m, l2 = rel_errors(y0.cpu().numpy(), golden["gen_taps_T3_s5_audio"])
        assert m < TOL and l2 < TOL, (m, l2)
        for which in range(4):
            tap = gen_module._dev.stage_output(which, 1, 3).cpu().numpy()
            m, l2 = rel_errors(tap, golden["gen_taps_T3_s5_%d" % which])
            assert m < TOL and l2 < TOL, (which, m, l2)
    finally:
        engine.check(engine.lib().mg_gen_set_pipeline(-1))


@pytest.mark.parametrize("B,T", [(1, 1), (1, 2), (3, 5), (1, 13), (2, 40), (1, 97)])
def test_matches_oracle_on_ragged_shapes(host_engine, folded, B, T):
    """Tile-boundary / tiny-sequence edge cases vs the C oracle on the same seeded inputs."""
    ws, bs = folded
    x = synth.mel_input(B, T, 100 + T)
    ref = cport.generator_forward(ws, bs, x)
    y = host_engine.forward(x)
    m, l2 = rel_errors(y, ref)
    assert m < TOL and l2 < TOL, (B, T, m, l2)


def test_long_utterance_matches_golden(golden, host_engine):
    y = host_engine.forward(synth.mel_input(1, 1000, 0)).reshape(-1)
    scale = np.abs(golden["gen_T1000_mid"]).max()
    assert np.abs(y[:4096] - golden["gen_T1000_head"]).max() < TOL * scale
    assert np.abs(y[128000 - 2048:128000 + 2048] - golden["gen_T1000_mid"]).max() < TOL * scale
    assert np.abs(y[-4096:] - golden["gen_T1000_tail"]).max() < TOL * scale
    bsum = y.astype(np.float64).reshape(250, 1024).sum(axis=1)
    assert np.abs(bsum - golden["gen_T1000_blocksum"]).max() < 1024 * TOL * scale


@pytest.fixture(scope="module")
def config2_golden():
    return np.load(os.path.join(os.path.dirname(__file__), "golden", "config2_outputs.npz"))


@pytest.mark.parametrize("realistic", [False, True])
def test_config2_full_size_matches_reference(host_engine, gen_module, config2_golden, realistic):
    """BASELINE config 2 at FULL size (B=64, 80x32 mel -> 64x8192 samples), every one of the 64 items against the
    unmodified reference's CPU-fp32 output (tests/golden/config2_outputs.npz, written by make_golden.py --config2: a
    seeded sample of every item and block sums over every sample), for N(0,1) and log-mel-like inputs, through both
    entry points (host buffers, torch module)."""
    x = synth.mel_input(64, 32, 0, realistic)
    key = "gen_B64_T32_s0_r%d" % int(realistic)
    ref, ref_bsum = config2_golden[key + "_sample"], config2_golden[key + "_blocksum"]
    y = host_engine.forward(x)
    assert y.shape == (64, 1, 8192)
    ys, bsum = cases.config2_digest(y, config2_golden["sample_index"])
    scale = float(config2_golden[key + "_absmax"])
    per_item = np.abs(ys.astype(np.float64) - ref).max(axis=1) / scale
    assert per_item.max() <= TOL, (int(per_item.argmax()), float(per_item.max()))
    m, l2 = rel_errors(ys, ref)
    assert m <= TOL and l2 <= TOL, (m, l2)
    assert np.abs(bsum - ref_bsum).max() <= cases.CONFIG2_BLOCK * TOL * scale
    with torch.no_grad():
        yd = gen_module(torch.from_numpy(x).cuda()).cpu().numpy()
    assert np.array_equal(yd, y)
    print("config 2 (realistic=%s): max-rel %.2e, l2-rel %.2e" % (realistic, m, l2))


def test_full_size_properties_config2(host_engine, gen_module):
    """Size-independent properties at BASELINE config 2 (B=64, T=32): batch items are independent (item i of the batch ==
    the same mel run alone), the device-pointer and host-buffer entry points agree bit for bit, and a long mel equals
    its chunks computed with an 8-frame halo (receptive field 7 frames, SURVEY section 5)."""
    x = synth.mel_input(64, 32, 0)
    y = host_engine.forward(x)
    assert np.isfinite(y).all() and np.abs(y).max() <= 1.0
    for i in (0, 17, 63):
        yi = host_engine.forward(x[i:i + 1])
        assert np.array_equal(yi[0], y[i])
    with torch.no_grad():
        yd = gen_module(torch.from_numpy(x).cuda()).cpu().numpy()
    assert np.array_equal(yd, y)
    # chunked == whole
    xl = synth.mel_input(1, 200, 9)
    whole = host_engine.forward(xl)[0, 0]
    lo, hi, halo = 64, 136, 8
    part = host_engine.forward(xl[:, :, lo - halo:hi + halo])[0, 0]
    np.testing.assert_allclose(part[halo * 256:(halo + hi - lo) * 256], whole[lo * 256:hi * 256], rtol=0, atol=1e-6)


def test_stalled_pipeline_status_is_not_silent(gen_module):
    """ADVICE r1: the kernels' bounded waits raise a device status word and carry on; Generator.forward must surface it.
    The status word of a forward is copied to the host asynchronously and checked at the next forward / poll."""
    x = torch.from_numpy(synth.mel_input(1, 4, 3)).cuda()
    with torch.no_grad():
        gen_module(x)
        torch.cuda.synchronize()
        engine.poll_status()  # healthy: nothing raised
        dev = gen_module._dev
        dev._watch.pin[0] = 3   # what a timed-out MMA issuer would have left behind
        dev._watch.pending = True
        engine._StatusWatch._live.add(dev._watch)
        with pytest.raises(engine.EngineError, match="timed out"):
            gen_module(x)
        gen_module(x)  # the error is reported once; the module keeps working
        torch.cuda.synchronize()
        engine.poll_status(wait=True)


def test_repack_follows_parameter_updates(gen_module):
    x = torch.from_numpy(synth.mel_input(1, 4, 3)).cuda()
    with torch.no_grad():
        y0 = gen_module(x).clone()
        gen_module.conv_post.bias.add_(0.25)
        y1 = gen_module(x).clone()
        gen_module.conv_post.bias.sub_(0.25)
        y2 = gen_module(x)
    assert not torch.equal(y0, y1)
    assert torch.allclose(y0, y2, atol=1e-6)


def test_backward_reaches_every_parameter(gen_module):
    """Gradients arrive on weight_g / weight_v / bias leaves through autograd (distributed.py:131-135
    hooks rely on it).  Forward is the native path; backward is the stock-op recomputation."""
    gen_module.zero_grad()
    x = torch.from_numpy(synth.mel_input(1, 4, 3)).cuda()
    y = gen_module(x)
    assert y.requires_grad
    y.square().mean().backward()
    for n, p in gen_module.named_parameters():
        assert p.grad is not None and torch.isfinite(p.grad).all(), n
    gen_module.zero_grad()


def test_deterministic_stream_ordered_and_layout_robust(gen_module):
    """Bitwise run-to-run determinism (no atomics on the data path), correct ordering on a non-default stream, and
    non-contiguous inputs (the shim makes them contiguous like the reference's Conv1d would accept them)."""
    x = torch.from_numpy(synth.mel_input(3, 9, 21)).cuda()
    with torch.no_grad():
        y0 = gen_module(x).clone()
        y1 = gen_module(x).clone()
        assert torch.equal(y0, y1)
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            y2 = gen_module(x * 1.0)  # producer and consumer both on the side stream
        torch.cuda.current_stream().wait_stream(s)
        assert torch.equal(y0, y2)
        xt = x.transpose(1, 2).contiguous().transpose(1, 2)  # same values, non-contiguous strides
        assert not xt.is_contiguous()
        assert torch.equal(gen_module(xt), y0)


def test_streaming_long_utterance_equals_whole(host_engine):
    """BASELINE config 5 (80 x 1000 mel, 11.6 s): chunked streaming with an 8-frame halo == the whole utterance."""
    mel = synth.mel_input(1, 1000, 0)
    whole = host_engine.forward(mel)
    chunks = list(host_engine.stream(mel, chunk_frames=96))
    assert len(chunks) == 11 and sum(c.shape[2] for c in chunks) == 256000
    np.testing.assert_allclose(np.concatenate(chunks, axis=2), whole, rtol=0, atol=1e-6)


def test_time_sharded_utterance_equals_whole(gen_module):
    """SURVEY 8e row 2: one utterance cut along time for N ranks (each reads its frames +- 8): the concatenation of the
    ranks' slices equals the whole-utterance forward.  The ranks are emulated on one GPU (no collective on this path)."""
    from melgan_multi_b200 import distributed as mgd
    mel = torch.from_numpy(synth.mel_input(1, 203, 9)).cuda()
    with torch.no_grad():
        whole = gen_module(mel)
        for world in (2, 3, 8):
            parts = [mgd.generate_sharded(gen_module, mel, rank=r, world_size=world, gather=False) for r in range(world)]
            got = torch.cat(parts, dim=2)
            assert got.shape == whole.shape
            assert (got - whole).abs().max().item() <= 1e-6


def test_batch_slices_are_bit_identical_to_single_chain(gen_module):
    """launch_generator_tc cuts large batches into concurrent slices (forked streams); the arithmetic per item is the
    same, so a sliced forward equals the per-item forwards bit for bit."""
    assert engine.lib().mg_gen_forward_slices(64, 32) == 4 and engine.lib().mg_gen_forward_slices(1, 1000) == 1
    x = torch.from_numpy(synth.mel_input(40, 32, 3)).cuda()  # 1280 frames -> 2 slices
    assert engine.lib().mg_gen_forward_slices(40, 32) == 2
    with torch.no_grad():
        y = gen_module(x)
        for i in (0, 19, 20, 39):
            assert torch.equal(y[i:i + 1], gen_module(x[i:i + 1]))


@pytest.mark.parametrize("B,T", [(2, 8), (40, 32)])
def test_forward_is_cuda_graph_capturable(gen_module, B, T):
    """The whole forward (including the forked batch-slice streams, which join the capture through their events) records
    into a CUDA graph and replays on new inputs: no host synchronisation or allocation on the library's side."""
    x = torch.from_numpy(synth.mel_input(B, T, 31)).cuda()
    static_x = x.clone()
    with torch.no_grad():
        ref = gen_module(x).clone()  # warm-up: packs the weights, sizes the workspace, configures the kernels
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            gen_module(static_x)
        torch.cuda.current_stream().wait_stream(s)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            static_y = gen_module(static_x)
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(static_y, ref)
        x2 = torch.from_numpy(synth.mel_input(B, T, 32)).cuda()
        static_x.copy_(x2)
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(static_y, gen_module(x2))


def test_large_odd_batch_slices(gen_module):
    """B = 301 x T = 7 (2107 frames -> 4 uneven slices of 76 / 75 items): items at the slice borders equal their
    single-item forwards bit for bit."""
    B, T = 301, 7
    assert engine.lib().mg_gen_forward_slices(B, T) == 4
    x = torch.from_numpy(synth.mel_input(B, T, 77)).cuda()
    with torch.no_grad():
        y = gen_module(x)
        gen_module._dev.check_status(B, T)
        for i in (0, 75, 76, 150, 151, 225, 226, 300):
            assert torch.equal(y[i:i + 1], gen_module(x[i:i + 1])), i
