"""Generate the golden fixtures in tests/golden/ by running the UNMODIFIED reference.

It imports models.py from a checkout of the reference, named by MG_REFERENCE_DIR:

    MG_REFERENCE_DIR=<reference checkout> python tests/golden/make_golden.py

Weights come from melgan_multi_b200.synth (seeded numpy MT19937), loaded into the reference
modules through load_state_dict, so the fixtures hold inputs' seeds and the reference's
OUTPUTS only.  Everything is computed by the reference's own forward() on CPU in fp32.
"""
import os
import sys
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
REFERENCE = os.environ.get("MG_REFERENCE_DIR", "")
if not os.path.isfile(os.path.join(REFERENCE, "models.py")):
    raise SystemExit("set MG_REFERENCE_DIR to the reference checkout (the directory holding its models.py)")
sys.path.insert(0, REFERENCE)
warnings.filterwarnings("ignore")

import models as ref_models  # noqa: E402  (the reference)
from melgan_multi_b200 import synth  # noqa: E402
sys.path.insert(0, HERE)
import cases  # noqa: E402


def load_state(module, state):
    module.load_state_dict({k: torch.from_numpy(v) for k, v in state.items()}, strict=True)
    return module.eval()


def generator_stage_outputs(gen, x):
    """Re-run Generator.forward step by step with the reference's own submodules to tap the
    per-stage activations (same calls as models.py:61-71)."""
    import torch.nn.functional as F
    taps = []
    h = gen.conv_pre(x); taps.append(h)
    for i in range(4):
        h = F.leaky_relu(h)
        h = gen.ups[i](h)
        h = gen.resblocks[i](h)
        taps.append(h)
    h = F.leaky_relu(h)
    h = gen.conv_post(h); taps.append(h)
    return [t.detach().numpy() for t in taps], torch.tanh(h).detach().numpy()


TRAIN_CASE = dict(B=2, T=4, mel_seed=21, audio_seed=22)  # one train.py:108-129 step on a 1024-sample segment


def grad_digest(named_params):
    d = {}
    for n, p in named_params:
        g = p.grad.detach().double().reshape(-1)
        d[n + "/l2"] = np.array(float(g.norm()))
        d[n + "/sum"] = np.array(float(g.sum()))
        d[n + "/head"] = g[:16].numpy().copy()
    return d


TRAIN_CASE_B16 = dict(B=16, T=32, mel_seed=0, audio_seed=0)  # BASELINE config 3: batch 16, 8192-sample segments


def config2_golden():
    """BASELINE config 2 at full size (B=64, 80x32 mel -> 64x8192 samples) through the unmodified reference on CPU, for
    N(0,1) and log-mel-like inputs: every item of the bench workload is pinned, not just item 0.  Of each output the
    fixture keeps cases.config2_digest (a seeded sample of every item, block sums over every sample) and max |y|."""
    gen = load_state(ref_models.Generator(), synth.generator_state(1234))
    index = cases.config2_sample_index()
    out = {"sample_index": index}
    with torch.no_grad():
        for realistic in (False, True):
            x = synth.mel_input(64, 32, 0, realistic)
            y = gen(torch.from_numpy(x)).numpy()
            key = "gen_B64_T32_s0_r%d" % int(realistic)
            out[key + "_sample"], out[key + "_blocksum"] = cases.config2_digest(y, index)
            out[key + "_absmax"] = np.abs(y).max()
    path = os.path.join(HERE, "config2_outputs.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, "%.2f MB" % (os.path.getsize(path) / 1e6), len(out), "arrays")


def train_step_golden(c=None, fname="train_step_grads.npz"):
    """Losses and parameter-gradient digests of ONE reference training step (train.py:108-129, without the optimizer
    updates): generator step through the discriminators, then the discriminator step on the detached audio."""
    c = c or TRAIN_CASE
    gen = load_state(ref_models.Generator(), synth.generator_state(1234)).train()
    msd = load_state(ref_models.MultiScaleDiscriminator(), synth.discriminator_state(4321)).train()
    x = torch.from_numpy(synth.mel_input(c["B"], c["T"], c["mel_seed"]))
    y = torch.from_numpy(synth.audio_input(c["B"], 256 * c["T"], c["audio_seed"]))
    out = {}
    y_ghat = gen(x)
    dr, dg, fr, fg = msd(y, y_ghat)
    loss_gen = ref_models.generator_loss(dg) + ref_models.feature_loss(fr, fg)
    loss_gen.backward()
    out["loss_gen"] = np.array(loss_gen.item())
    for k, v in grad_digest(gen.named_parameters()).items():
        out["gstep/G/" + k] = v
    for k, v in grad_digest(msd.named_parameters()).items():
        out["gstep/D/" + k] = v
    msd.zero_grad()
    dr, dg, _, _ = msd(y, y_ghat.detach())
    loss_disc, _, _ = ref_models.discriminator_loss(dr, dg)
    loss_disc.backward()
    out["loss_disc"] = np.array(loss_disc.item())
    for k, v in grad_digest(msd.named_parameters()).items():
        out["dstep/D/" + k] = v
    out["y_ghat_head"] = y_ghat.detach().numpy()[:2, 0, :256].copy()
    path = os.path.join(HERE, fname)
    np.savez_compressed(path, **out)
    print("wrote", path, "%.2f MB" % (os.path.getsize(path) / 1e6), len(out), "arrays")


def main():
    if "--train-step" in sys.argv:  # only the training-step fixture (leaves reference_outputs.npz untouched)
        torch.set_num_threads(os.cpu_count())
        return train_step_golden()
    if "--train-step-b16" in sys.argv:  # BASELINE config 3 shape (B=16 x 8192 samples)
        torch.set_num_threads(os.cpu_count())
        return train_step_golden(TRAIN_CASE_B16, "train_step_grads_b16.npz")
    if "--config2" in sys.argv:
        torch.set_num_threads(os.cpu_count())
        return config2_golden()
    torch.manual_seed(0)
    torch.set_num_threads(os.cpu_count())
    out = {}

    # ---------------- generator ----------------
    gstate = synth.generator_state(1234)
    gen = load_state(ref_models.Generator(), gstate)
    with torch.no_grad():
        for (B, T, seed, realistic) in cases.GEN_CASES:
            x = synth.mel_input(B, T, seed, realistic)
            y = gen(torch.from_numpy(x)).numpy()
            out[cases.gen_key(B, T, seed, realistic)] = y
        # per-stage taps on a tiny case
        x = synth.mel_input(1, 3, 5)
        taps, y = generator_stage_outputs(gen, torch.from_numpy(x))
        y_direct = gen(torch.from_numpy(x)).numpy()
        assert np.array_equal(y, y_direct)
        for i, t in enumerate(taps):
            out["gen_taps_T3_s5_%d" % i] = t
        out["gen_taps_T3_s5_audio"] = y
        # long utterance (config 5): keep three windows and block sums
        x = synth.mel_input(1, 1000, 0)
        y = gen(torch.from_numpy(x)).numpy().reshape(-1)
        out["gen_T1000_head"] = y[:4096].copy()
        out["gen_T1000_mid"] = y[128000 - 2048:128000 + 2048].copy()
        out["gen_T1000_tail"] = y[-4096:].copy()
        out["gen_T1000_blocksum"] = y.astype(np.float64).reshape(250, 1024).sum(axis=1)
        # weight-norm fold as the reference modules apply it (pre-forward hook output)
        # conv_pre's fold is 1.1 MB: keep every 8th output channel, and the L2 norm of every channel
        fold = gen.conv_pre.weight.detach().numpy()
        out["fold_conv_pre_every8th"] = fold[::8].copy()
        out["fold_conv_pre_norms"] = np.sqrt((fold.astype(np.float64) ** 2).reshape(len(fold), -1).sum(axis=1))
        out["fold_ups3"] = gen.ups[3].weight.detach().numpy()
        out["fold_res2_c1_1"] = gen.resblocks[2].convs1[1].weight.detach().numpy()

    # ---------------- discriminator ----------------
    dstate = synth.discriminator_state(4321)
    msd = load_state(ref_models.MultiScaleDiscriminator(), dstate)
    with torch.no_grad():
        for (B, L, seed) in cases.MSD_CASES:
            y = synth.audio_input(B, L, seed)
            y_hat = synth.audio_input(B, L, seed + 7)
            rs, gs, frs, fgs = msd(torch.from_numpy(y), torch.from_numpy(y_hat))
            tag = "msd_B%d_L%d_s%d" % (B, L, seed)
            for i in range(3):
                out["%s_logit_r%d" % (tag, i)] = rs[i].numpy()
                out["%s_logit_g%d" % (tag, i)] = gs[i].numpy()
                for j in range(7):
                    for nm, fm in (("r", frs[i][j]), ("g", fgs[i][j])):
                        a = fm.numpy()
                        out["%s_fmap_%s%d_%d_shape" % (tag, nm, i, j)] = np.array(a.shape)
                        out["%s_fmap_%s%d_%d_sum" % (tag, nm, i, j)] = np.array(
                            [a.astype(np.float64).sum(), np.abs(a.astype(np.float64)).sum()])
                        out["%s_fmap_%s%d_%d_head" % (tag, nm, i, j)] = a[:, :4, :48].copy()
            out[tag + "_feature_loss"] = np.array(ref_models.feature_loss(frs, fgs).item())
            out[tag + "_generator_loss"] = np.array(ref_models.generator_loss(gs).item())
            dl, rl, gl = ref_models.discriminator_loss(rs, gs)
            out[tag + "_discriminator_loss"] = np.array([dl.item()] + rl + gl)

    # ---------------- primitive ops (edge cases) ----------------
    import torch.nn.functional as F
    for key, kind, prm, x, w, b in cases.op_inputs():
        tx = torch.from_numpy(x)
        if kind == "conv":
            y = F.conv1d(tx, torch.from_numpy(w), torch.from_numpy(b), *prm)
        elif kind == "convT":
            y = F.conv_transpose1d(tx, torch.from_numpy(w), torch.from_numpy(b), *prm)
        else:
            y = torch.nn.AvgPool1d(prm[0], prm[1], padding=prm[2])(tx)
        out[key] = y.numpy()

    # ---------------- module ABI: state_dict keys / shapes / parameter order ----------------
    import json
    abi = {}
    for nm, mod in (("Generator", ref_models.Generator()), ("MultiScaleDiscriminator", ref_models.MultiScaleDiscriminator())):
        abi[nm] = {"state_dict": [[k, list(v.shape)] for k, v in mod.state_dict().items()],
                   "parameters": [n for n, _ in mod.named_parameters()]}
    with open(os.path.join(HERE, "module_abi.json"), "w") as f:
        json.dump(abi, f, indent=0)

    path = os.path.join(HERE, "reference_outputs.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, "%.2f MB" % (os.path.getsize(path) / 1e6), len(out), "arrays")


if __name__ == "__main__":
    main()
