"""Ragged generator batches on the B200 (mg_gen_forward_varlen through models.Generator(x, lengths) and the host engine):
every item's audio is bit-identical to the forward of that item alone, the audio past its end is exactly zero, and
nothing depends on the mel padding or on stale workspace contents."""
import numpy as np
import pytest
import torch

from conftest import rel_errors
from melgan_multi_b200 import engine, synth
from oracle import cport

pytestmark = pytest.mark.gpu

MIXED_T = 97
MIXED_LENGTHS = [1, 2, 3, 7, 16, 17, 31, 32, 33, 64, 96, 97]  # stage-0 pair threshold (16 / 17 frames) and tile edges


@pytest.fixture(scope="module")
def state():
    return synth.generator_state(1234)


@pytest.fixture(scope="module")
def gen_module(state):
    from melgan_multi_b200 import models
    g = models.Generator()
    g.load_state_dict({k: torch.from_numpy(v) for k, v in state.items()})
    return g.cuda().eval()


def _single(gen, x, b, n):
    return gen(x[b:b + 1, :, :n].contiguous())


def _check_items(gen, x, y, lengths, items):
    for b in items:
        n = int(lengths[b])
        assert torch.equal(y[b:b + 1, :, :256 * n], _single(gen, x, b, n)), (b, n)
        assert bool((y[b, :, 256 * n:] == 0).all()), (b, n)  # (== 0 also holds for -0.0; the kernel writes +0.0)


@pytest.fixture(scope="module")
def mixed(gen_module):
    x = torch.from_numpy(synth.mel_input(len(MIXED_LENGTHS), MIXED_T, 41)).cuda()
    with torch.no_grad():
        y = gen_module(x, lengths=MIXED_LENGTHS)
        gen_module._dev.check_status(len(MIXED_LENGTHS), MIXED_T)
    return x, y


def test_mixed_lengths_equal_single_item_forwards(gen_module, mixed):
    x, y = mixed
    assert y.shape == (len(MIXED_LENGTHS), 1, 256 * MIXED_T)
    with torch.no_grad():
        _check_items(gen_module, x, y, MIXED_LENGTHS, range(len(MIXED_LENGTHS)))
        # an integer CUDA tensor of lengths gives the same call
        y2 = gen_module(x, lengths=torch.tensor(MIXED_LENGTHS, dtype=torch.int32, device="cuda"))
    assert torch.equal(y2, y)


def test_padding_values_and_stale_workspace_change_nothing(gen_module, mixed):
    x, y = mixed
    B = len(MIXED_LENGTHS)
    with torch.no_grad():
        for fill in (float("nan"), 1e30):
            xp = x.clone()
            for b, n in enumerate(MIXED_LENGTHS):
                xp[b, :, n:] = fill
            gen_module._dev.workspace(B, MIXED_T).fill_(float("nan"))
            yp = gen_module(xp, lengths=MIXED_LENGTHS)
            gen_module._dev.check_status(B, MIXED_T)
            assert torch.equal(yp, y), fill


def test_full_lengths_equal_uniform_config2(gen_module):
    B, T = 64, 32
    assert engine.lib().mg_gen_forward_slices(B, T) == 4
    x = torch.from_numpy(synth.mel_input(B, T, 0)).cuda()
    with torch.no_grad():
        assert torch.equal(gen_module(x, lengths=[T] * B), gen_module(x))


def test_many_items_and_slice_borders(gen_module):
    rs = np.random.RandomState(5)
    lengths = rs.randint(1, 14, size=301)
    T = int(lengths.max())
    x = torch.from_numpy(synth.mel_input(301, T, 78)).cuda()
    with torch.no_grad():
        y = gen_module(x, lengths=lengths.tolist())
        gen_module._dev.check_status(301, T)
        _check_items(gen_module, x, y, lengths, range(301))  # every item, so every slice border is covered
        # more items than one launch's table holds: a slice runs as several launches
        lengths = rs.randint(1, 5, size=1500)
        x = torch.from_numpy(synth.mel_input(1500, 4, 79)).cuda()
        y = gen_module(x, lengths=torch.from_numpy(lengths))
        gen_module._dev.check_status(1500, 4)
        _check_items(gen_module, x, y, lengths, range(1500))


def test_ragged_items_match_the_oracle(gen_module, state):
    lengths, T = [3, 11, 6], 11
    mel = synth.mel_input(3, T, 12)
    with torch.no_grad():
        y = gen_module(torch.from_numpy(mel).cuda(), lengths=lengths).cpu().numpy()
    ws, bs = cport.fold_generator(state)
    for b, n in enumerate(lengths):
        ref = cport.generator_forward(ws, bs, mel[b:b + 1, :, :n])
        m, l2 = rel_errors(y[b:b + 1, :, :256 * n], ref)
        assert m < 1e-4 and l2 < 1e-4, (b, m, l2)
        assert not y[b, :, 256 * n:].any()


def test_host_engine_pinned_and_pageable_equal_device_path(gen_module, state, mixed):
    x, y = mixed
    B = len(MIXED_LENGTHS)
    e = engine.GeneratorHost(B, MIXED_T)
    try:
        e.load_state(state)
        mel = x.cpu().numpy()
        out = e.forward(mel, lengths=MIXED_LENGTHS)  # pageable in and out
        assert np.array_equal(out, y.cpu().numpy())
        pin_in = torch.empty(mel.shape, dtype=torch.float32).pin_memory()
        pin_out = torch.full((B, 1, 256 * MIXED_T), float("nan")).pin_memory()
        pin_in.numpy()[...] = mel
        e.forward(pin_in.numpy(), out=pin_out.numpy(), lengths=tuple(MIXED_LENGTHS))
        assert torch.equal(pin_out, y.cpu())
    finally:
        e.close()


def test_varlen_forward_is_cuda_graph_capturable(gen_module):
    lengths, T = [5, 32, 1, 19, 27, 8], 32
    x = torch.from_numpy(synth.mel_input(len(lengths), T, 51)).cuda()
    static_x = x.clone()
    with torch.no_grad():
        ref = gen_module(x, lengths=lengths).clone()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            gen_module(static_x, lengths=lengths)
        torch.cuda.current_stream().wait_stream(s)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            static_y = gen_module(static_x, lengths=lengths)
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(static_y, ref)
        x2 = torch.from_numpy(synth.mel_input(len(lengths), T, 52)).cuda()
        static_x.copy_(x2)
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(static_y, gen_module(x2, lengths=lengths))


def test_long_utterances(gen_module):
    lengths = np.random.RandomState(16).randint(100, 1001, size=16)
    T = int(lengths.max())
    x = torch.from_numpy(synth.mel_input(16, T, 61)).cuda()
    with torch.no_grad():
        y = gen_module(x, lengths=lengths.tolist())
        gen_module._dev.check_status(16, T)
        _check_items(gen_module, x, y, lengths, (0, int(np.argmin(lengths)), 15))


def test_ragged_forward_refuses_autograd(gen_module):
    x = torch.from_numpy(synth.mel_input(2, 8, 3)).cuda()
    with torch.enable_grad():
        with pytest.raises(engine.EngineError):
            gen_module(x, lengths=[8, 5])  # the parameters require grad
        with torch.no_grad():
            gen_module(x, lengths=[8, 5])  # fine without autograd
