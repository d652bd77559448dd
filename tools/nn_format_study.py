"""Number-format study of the policy/value tower (CPU only, no kernel involved): which operand formats could hold the
north-star tolerance (logits within 1e-3 of the fp32 forward) on trained-like weights?

VERDICT r1 (next item 2) proposed two ways to close the tolerance on the tensor-core path: (1) per-layer activation scaling
into the fp16 range folded into the BatchNorm scale, (2) a split-fp16 (hi + lo) representation of the residual-block input
only.  This tool evaluates those and the other candidates with the format model of oracle/nn.py: every convolution of the
tower is computed EXACTLY (fp64) on operands rounded the way a format would round them, everything else (folded BatchNorm,
residual stream, heads) in fp32 -- so a row is the floor of what any kernel using that format can reach (tools/nn_diag.py
shows that the tcgen05 kernel sits on its format's floor).

    fp16            both operands rounded to fp16 (what csrc/rz_net_tc.cu does: 1 MMA per product)
    fp16-scaled     activations multiplied by a per-layer power of two that brings their maximum to 2^14 before rounding
                    (proposal 1; fp16 rounding is relative, so nothing changes unless values were subnormal)
    bf16            both operands rounded to bf16
    act-split@res   activations of the first convolution of every block (the residual stream) as hi + lo, 2 MMAs there
                    (proposal 2)
    act-split       all activations as hi + lo (2 MMAs per product)
    w-split         all weights as hi + lo (2 MMAs)
    3-mma           hi*hi + hi*lo + lo*hi (both operands split, the lo*lo term dropped)

Prints max-abs errors over the positions for the tower output, the policy logits and the value logit, for `--new`
random-init weights, perturbed BatchNorm statistics and trained-like (calibrated) weights of the ch5 network.
    python tools/nn_format_study.py > profiles/nn_format_study_r02.txt"""
import os
import sys

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "reversi-alpha-zero_b200"))

MODES = ("fp16", "fp16-scaled", "bf16", "act-split@res", "act-split", "w-split", "3-mma")
MMAS = {"fp16": "1", "fp16-scaled": "1", "bf16": "1", "act-split@res": "1.5", "act-split": "2", "w-split": "2", "3-mma": "3"}


def hi(t, dt=torch.float16):
    return t.to(dt).float()


def lo(t):
    return (t - hi(t)).half().float()


def conv_terms(x, k, mode, first_of_block, exact_input):
    """list of (activation part, weight part) whose exact products are summed"""
    if mode == "bf16":
        return [(hi(x, torch.bfloat16), hi(k, torch.bfloat16))]
    if mode == "fp16-scaled" and not exact_input:
        s = 2.0 ** np.floor(14 - np.log2(max(float(x.abs().max()), 1e-30)))
        return [(hi(x * s) / s, hi(k))]
    split_a = (mode in ("act-split", "3-mma") or (mode == "act-split@res" and first_of_block)) and not exact_input
    split_w = mode in ("w-split", "3-mma")
    terms = [(hi(x), hi(k))]
    if split_a:
        terms.append((lo(x), hi(k)))
    if split_w:
        terms.append((hi(x), lo(k)))
    return terms


@torch.no_grad()
def tower(w, planes, n_res, mode):
    from oracle import nn as onn

    def conv(x, name, first_of_block=False, exact_input=False):
        k = torch.from_numpy(w[f"{name}.kernel"]).permute(3, 2, 0, 1).contiguous()
        s, sh = onn._fold(w, name)
        acc = sum(F.conv2d(a.double(), b.double(), padding=1) for a, b in conv_terms(x, k, mode, first_of_block, exact_input))
        return acc.float() * s + sh

    x = F.relu(conv(torch.from_numpy(np.ascontiguousarray(planes)).float(), "conv0", exact_input=True))
    for i in range(n_res):
        y = F.relu(conv(x, f"res{i}.conv1", first_of_block=True))
        x = F.relu(conv(y, f"res{i}.conv2") + x)
    return onn.heads(w, x)   # policy, value, logits, value logit, tower


def main():
    from oracle import nn as onn
    from reversi_zero_b200.agent import model as M
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_net_gpu import selfplay_positions
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from nn_diag import weights_of
    torch.set_num_threads(max(1, len(os.sched_getaffinity(0))))
    n, R = 48, 10
    planes = onn.planes_from_bitboards(*selfplay_positions(n, 5))
    planes_cal = onn.planes_from_bitboards(*selfplay_positions(256, 11))
    mc = M.ModelConfig(cnn_filter_num=256, res_layer_num=R, value_fc_size=256)
    print(f"ch5 tower (256 filters x {R} blocks), {n} self-play positions, max-abs error against the fp32 forward "
          f"(exact products, fp32 everything else); MMAs = tensor-core passes per product")
    for kind in ("random-init", "perturbed", "calibrated"):
        w = weights_of(kind, mc, 5, planes_cal)
        ref = onn.forward_logits(w, planes, R)
        print(f"\n{kind} weights: |logits| <= {np.abs(ref[2]).max():.2f}, |value logit| <= {np.abs(ref[3]).max():.2f}, tower rms {np.sqrt((ref[4] ** 2).mean()):.3f}")
        print(f"  {'format':14s} {'MMAs':>4s} {'tower':>10s} {'logits':>10s} {'value logit':>12s} {'policy':>10s} {'value':>10s}   logits <= 1e-3")
        for mode in MODES:
            got = tower(w, planes, R, mode)
            e = [float(np.abs(g - r).max()) for g, r in zip(got, ref)]
            print(f"  {mode:14s} {MMAS[mode]:>4s} {e[4]:10.3g} {e[2]:10.3g} {e[3]:12.3g} {e[0]:10.3g} {e[1]:10.3g}   {'yes' if max(e[2], e[3]) <= 1e-3 else 'no'}")


if __name__ == "__main__":
    main()
