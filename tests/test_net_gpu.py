"""GPU parity tests for the network kernels through the C ABI against the fp32 torch oracle
(oracle/nn.py).  Tolerance (BASELINE.json north_star: "policy/value logits ... within 1e-3"): 1e-3 max-abs on the policy
LOGITS (input of the softmax), the value logit (input of the tanh), the softmax probabilities and the tanh value for the
fp16-operand / fp32-accumulate tcgen05 tower on `--new` (random-init) weights, the north-star configuration; 2e-5 for the
fp32 generic kernel on any weights.  For trained-like weights the tower is held to the error of its NUMBER FORMAT
(oracle/nn.py forward_fp16_operands; profiles/nn_diag_r02.*): test_tcgen05_trained_like_weights_format_bound."""
import numpy as np
import pytest

from oracle import nn as onn
from oracle import bitboard as ob
from reversi_zero_b200.agent import model as M
from reversi_zero_b200.agent.api import ReversiModelAPI
from reversi_zero_b200 import net as N

pytestmark = pytest.mark.gpu


def selfplay_positions(n, seed=3):
    """positions from random playouts (side-to-move frame), a few of them dihedral-transformed."""
    rng = np.random.default_rng(seed)
    own, enemy = [], []
    while len(own) < n:
        e = ob.Env().reset()
        while not e.done and len(own) < n:
            o, en = e.own_enemy()
            t = int(rng.integers(8))
            own.append(ob.dihedral(o, t)); enemy.append(ob.dihedral(en, t))
            legal = ob.find_correct_moves(o, en)
            ms = [i for i in range(64) if legal >> i & 1]
            e.step(ms[rng.integers(len(ms))])
    return np.array(own, np.uint64), np.array(enemy, np.uint64)


def run_case(mc, n, impl, seed, perturb, tol, check_tower=False, logit_tol=None):
    import torch
    from reversi_zero_b200 import device as D
    w = M.build_random_weights(mc, seed, perturb_bn=perturb)
    net = N.Net(mc)
    net.load_weights(w)
    own, enemy = selfplay_positions(n, seed)
    planes = onn.planes_from_bitboards(own, enemy)
    p_ref, v_ref, logits_ref, tower_ref = onn.forward(w, planes, mc.res_layer_num, return_tower=True)
    d_own, d_en = D.to_device(own), D.to_device(enemy)
    d_pol, d_val = D.empty(n * 64, np.float32), D.empty(n, np.float32)
    if check_tower:
        d_tow = D.empty(n * 64 * 256, np.float32)
        net.debug_tower_dev(d_own, d_en, d_pol, d_val, d_tow, n)
        torch.cuda.synchronize()
        tower = d_tow.cpu().numpy().reshape(n, 64, 256).transpose(0, 2, 1).reshape(n, 256, 8, 8)
        terr = np.abs(tower - tower_ref).max()
        scale = np.abs(tower_ref).max()
        assert terr <= 4e-3 * max(scale, 1.0), f"tower max-abs err {terr} (scale {scale})"
    elif impl == N.IMPL_TCGEN05:
        # the head outputs BEFORE softmax / tanh: the north-star tolerance is stated on the logits
        d_log, d_vl = D.empty(n * 64, np.float32), D.empty(n, np.float32)
        net.debug_heads_dev(d_own, d_en, d_pol, d_val, d_log, d_vl, n)
        torch.cuda.synchronize()
        _, _, lg_ref, vl_ref, _ = onn.forward_logits(w, planes, mc.res_layer_num)
        lerr = np.abs(d_log.cpu().numpy().reshape(n, 64) - lg_ref).max()
        vlerr = np.abs(d_vl.cpu().numpy() - vl_ref).max()
        lt = logit_tol or tol
        assert lerr <= lt and vlerr <= lt, f"policy-logit err {lerr}, value-logit err {vlerr} (tol {lt})"
        d_pol2, d_val2 = D.empty(n * 64, np.float32), D.empty(n, np.float32)
        net.predict_dev(d_own, d_en, d_pol2, d_val2, n, impl)      # the production entry point gives the same numbers
        torch.cuda.synchronize()
        assert torch.equal(d_pol, d_pol2) and torch.equal(d_val, d_val2)
    else:
        net.predict_dev(d_own, d_en, d_pol, d_val, n, impl)
        torch.cuda.synchronize()
    p = d_pol.cpu().numpy().reshape(n, 64)
    v = d_val.cpu().numpy()
    assert np.isfinite(p).all() and np.isfinite(v).all()
    perr, verr = np.abs(p - p_ref).max(), np.abs(v - v_ref).max()
    assert perr <= tol and verr <= tol, f"policy err {perr}, value err {verr} (tol {tol})"
    # host-buffer path (ReversiModelAPI.predict contract, agent/api.py:30-45)
    api = ReversiModelAPI(None, net, impl)
    k = min(5, n)
    p2, v2 = api.predict(planes[:k])
    assert p2.shape == (k, 64) and v2.shape == (k, 1)
    assert np.abs(p2 - p_ref[:k]).max() <= tol and np.abs(v2[:, 0] - v_ref[:k]).max() <= tol
    p1, v1 = api.predict(planes[0])
    assert p1.shape == (64,) and v1.shape == (1,)
    net.close()
    return perr, verr


MINI = dict(cnn_filter_num=16, res_layer_num=1, value_fc_size=16)
CH5 = dict(cnn_filter_num=256, res_layer_num=10, value_fc_size=256)


@pytest.mark.parametrize("cfg,n", [(MINI, 33), (dict(cnn_filter_num=32, res_layer_num=2, value_fc_size=64), 9),
                                   (dict(cnn_filter_num=256, res_layer_num=1, value_fc_size=256), 5)])
def test_generic_kernel_vs_oracle(cfg, n):
    run_case(M.ModelConfig(**cfg), n, N.IMPL_GENERIC, seed=1, perturb=True, tol=2e-5)


@pytest.mark.parametrize("res_blocks", [0, 1, 2])
def test_tcgen05_small_towers(res_blocks):
    """0 blocks isolates the layer-0 im2col GEMM + heads; 1-2 blocks the shifted-operand convs and the
    TMEM residual."""
    mc = M.ModelConfig(cnn_filter_num=256, res_layer_num=res_blocks, value_fc_size=256)
    run_case(mc, 7, N.IMPL_TCGEN05, seed=2, perturb=True, tol=1e-3, check_tower=True)
    run_case(mc, 7, N.IMPL_TCGEN05, seed=2, perturb=True, tol=1e-3)


@pytest.mark.parametrize("n", [1, 2, 301, 1000])
def test_tcgen05_ch5_vs_oracle(n):
    """ch5 network (256 filters x 10 blocks), random-init as `--new` builds it; n = 1000 > 2 x 148 SMs so
    every CTA processes several tiles."""
    run_case(M.ModelConfig(**CH5), n, N.IMPL_TCGEN05, seed=0, perturb=False, tol=1e-3)


def test_tcgen05_deep_tower_config4():
    """BASELINE config 4: the same kernel with a deeper tower (19 residual blocks = 39 convolutions, the AlphaGo Zero
    depth), random-init as `--new` builds it; same 1e-3 bound on policy probabilities and value; the logits of a tower
    twice as deep as ch5 are held to 4e-3 (fp16 operand rounding compounds with depth and with the growing residual stream:
    measured 5.5e-4 at ch5's 21 convolutions, 2.3e-3 at 39)."""
    run_case(M.ModelConfig(cnn_filter_num=256, res_layer_num=19, value_fc_size=256), 96, N.IMPL_TCGEN05, seed=0, perturb=False, tol=1e-3,
             logit_tol=4e-3)


def _heads_on_device(net, own, enemy, want_tower=True):
    import torch
    from reversi_zero_b200 import device as D
    n = own.size
    d_own, d_en = D.to_device(own), D.to_device(enemy)
    d_pol, d_val, d_log, d_vl = D.empty(n * 64, np.float32), D.empty(n, np.float32), D.empty(n * 64, np.float32), D.empty(n, np.float32)
    d_tow = D.empty(n * 64 * 256, np.float32) if want_tower else None
    net.debug_heads_dev(d_own, d_en, d_pol, d_val, d_log, d_vl, n, tower_t=d_tow)
    torch.cuda.synchronize()
    out = dict(policy=d_pol.cpu().numpy().reshape(n, 64), value=d_val.cpu().numpy(), logits=d_log.cpu().numpy().reshape(n, 64),
               vlogit=d_vl.cpu().numpy())
    if want_tower:
        out["tower"] = d_tow.cpu().numpy().reshape(n, 64, 256).transpose(0, 2, 1).reshape(n, 256, 8, 8)
    return out


@pytest.mark.parametrize("kind", ["perturbed", "calibrated"])
def test_tcgen05_trained_like_weights_format_bound(kind):
    """Weights that are NOT the north-star's `--new` initialisation: `perturbed` = random biases / BatchNorm statistics
    (the round-1 stress case), `calibrated` = BatchNorm statistics of every layer set to the statistics of its own
    pre-activation over 256 self-play positions, random gamma / beta / biases (what a trained network looks like: every
    layer normalised, residual stream growing with depth).  The residual stream reaches rms 1.4 / 3.0 (random-init: 0.17)
    and the logits magnitude 3-4, so one fp16 rounding of an operand (2^-11 relative) is already ~1e-3 absolute: NO
    single-pass fp16-operand evaluation can hold 1e-3 here (profiles/nn_diag_r02.txt: format error 2e-3 / 5e-3 on the
    logits).  What the kernel is held to: it adds nothing to the error of its number format -- its distance to the fp32
    reference is within 1.6 x the distance of the exact fp16-operand model (oracle/nn.py forward_fp16_operands), for the
    tower output, the policy logits and the value logit -- and stays below the stress bounds measured in round 1/2.
    The generic fp32 kernel (net_impl = 1) is the exact path for such weights: <= 2e-5."""
    import torch
    from reversi_zero_b200 import device as D
    mc = M.ModelConfig(cnn_filter_num=256, res_layer_num=10, value_fc_size=256)
    w = M.build_random_weights(mc, 5, perturb_bn=True)
    if kind == "calibrated":
        oc, ec = selfplay_positions(256, 11)
        onn.calibrate_bn(w, onn.planes_from_bitboards(oc, ec), 10)
    n = 64
    own, enemy = selfplay_positions(n, 5)
    planes = onn.planes_from_bitboards(own, enemy)
    net = N.Net(mc)
    net.load_weights(w)
    got = _heads_on_device(net, own, enemy)
    names = ("policy", "value", "logits", "vlogit", "tower")
    ref = dict(zip(names, onn.forward_logits(w, planes, 10)))
    fmt = dict(zip(names, onn.forward_fp16_operands(w, planes, 10)))
    for k, floor in (("tower", 1e-3), ("logits", 3e-4), ("vlogit", 3e-4)):
        kernel_err, format_err = np.abs(got[k] - ref[k]).max(), np.abs(fmt[k] - ref[k]).max()
        assert kernel_err <= 1.6 * format_err + floor, (kind, k, kernel_err, format_err)
    bound = dict(perturbed=4e-3, calibrated=1.2e-2)[kind]      # measured: 1.8e-3 / 6.3e-3 on the logits, 1e-3 / 3.2e-3 on the value logit
    assert np.abs(got["logits"] - ref["logits"]).max() <= bound and np.abs(got["vlogit"] - ref["vlogit"]).max() <= bound
    assert np.abs(got["policy"] - ref["policy"]).max() <= 1e-3      # the probabilities MCTS consumes stay within 1e-3 all the same
    # the exact path for arbitrary weights: generic fp32 kernel
    d_own, d_en = D.to_device(own), D.to_device(enemy)
    d_pol, d_val = D.empty(n * 64, np.float32), D.empty(n, np.float32)
    net.predict_dev(d_own, d_en, d_pol, d_val, n, N.IMPL_GENERIC)
    torch.cuda.synchronize()
    assert np.abs(d_pol.cpu().numpy().reshape(n, 64) - ref["policy"]).max() <= 2e-5
    assert np.abs(d_val.cpu().numpy() - ref["value"]).max() <= 5e-5
    net.close()


def test_tcgen05_matches_generic_on_device():
    """the two CUDA implementations agree with each other (cross-check independent of torch)."""
    import torch
    from reversi_zero_b200 import device as D
    mc = M.ModelConfig(**CH5)
    net = N.Net(mc)
    net.load_weights(M.build_random_weights(mc, 9))
    own, enemy = selfplay_positions(40, 9)
    d_own, d_en = D.to_device(own), D.to_device(enemy)
    outs = []
    for impl in (N.IMPL_GENERIC, N.IMPL_TCGEN05):
        d_pol, d_val = D.empty(40 * 64, np.float32), D.empty(40, np.float32)
        net.predict_dev(d_own, d_en, d_pol, d_val, 40, impl)
        torch.cuda.synchronize()
        outs.append((d_pol.cpu().numpy(), d_val.cpu().numpy()))
    assert np.abs(outs[0][0] - outs[1][0]).max() <= 1e-3 and np.abs(outs[0][1] - outs[1][1]).max() <= 1e-3


def test_tower_kernel_deterministic_vs_oracle():
    """The tcgen05 tower kernel (csrc/rz_net_tc.cu, CTA pairs with the epilogue overlapped) on ch5 `--new` weights and a
    ragged batch: bit-identical over two calls, and within 1e-3 of the fp32 oracle on logits, value logit, probabilities
    and value."""
    mc = M.ModelConfig(**CH5)
    w = M.build_random_weights(mc, 4)
    own, enemy = selfplay_positions(301, 4)
    planes = onn.planes_from_bitboards(own, enemy)
    ref = dict(zip(("policy", "value", "logits", "vlogit", "tower"), onn.forward_logits(w, planes, 10)))
    net = N.Net(mc)
    net.load_weights(w)
    a, b = _heads_on_device(net, own, enemy, want_tower=False), _heads_on_device(net, own, enemy, want_tower=False)
    assert all(np.array_equal(a[k], b[k]) for k in a)
    for k in ("logits", "vlogit", "policy", "value"):
        assert np.abs(a[k] - ref[k]).max() <= 1e-3, (k, np.abs(a[k] - ref[k]).max())
    net.close()
