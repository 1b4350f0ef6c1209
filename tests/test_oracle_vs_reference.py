"""The oracle and the product's parameter tree on fresh seeds, against what the unmodified reference computed for
the same inputs, recorded in tests/golden/oracle_vs_reference.npz (tests/golden/make_golden_oracle_vs_reference.py
says which values are equal to the reference's and which are within its tolerance).  CPU only."""
import ast

import numpy as np
import pytest
import torch

import fixtures_util as FU
import velocity_oracle as O

# Recorded values that stand within 1e-4 (mel) / 5e-5 (logits) of the reference's are matched far tighter, so
# the oracle stays as close to the reference as it was: the oracle is float64 throughout and a re-run differs
# only in summation order; the recorded mel is float32.
MEL_PIN = 1e-6
LOGIT_PIN = 1e-9


def rel(a, b):
    return float(np.abs(np.asarray(a, dtype=np.float64) - b).max() / (np.abs(b).max() + 1e-30))


@pytest.fixture(scope="module")
def g(golden):
    return golden("oracle_vs_reference")


def recorded(g, name):
    return ast.literal_eval(str(g[name]))


def test_mel_and_forward_fresh_seed(g):
    import velocity_asr
    audio = FU.synth_audio(2, 24000, seed=321)
    mel = g["mel"]
    assert np.abs(O.log_mel(audio.numpy()) - mel).max() < MEL_PIN
    for mode in ("sequential", "parallel"):
        torch.manual_seed(5)
        m = velocity_asr.VELOCITYASR(velocity_asr.VelocityASRConfig(scan_mode=mode))
        sd = {k: v.numpy() for k, v in FU.amplify_state_dict(m.state_dict(), seed=9).items()}
        got = O.forward(mel, sd, dict(scan_mode=mode))
        assert rel(got[:, ::8], g[mode + "_logits_sub"]) < LOGIT_PIN
        assert O.ctc_greedy_decode(got) == recorded(g, mode + "_tokens")


def test_product_parameter_tree_draws_reference_weights(g):
    import velocity_asr
    torch.manual_seed(11)
    b = velocity_asr.VELOCITYASR(velocity_asr.VelocityASRConfig()).state_dict()
    assert FU.state_dict_fingerprint(b) == g["tree_seed11"].tolist()


def test_timestamp_decode_matches_reference(g):
    """decode.py:74-125 against the oracle's restatement, on run-heavy random predictions."""
    rs = np.random.RandomState(3)
    for i, (B, L, V) in enumerate([(5, 97, 6), (3, 1, 4), (2, 300, 3), (1, 33, 2)]):
        lg = rs.standard_normal((B, L, V)).astype(np.float32)
        lg[..., 0] += 0.8
        lg = np.repeat(lg, 2, axis=1)[:, :L]
        assert recorded(g, f"timestamps_{i}") == O.ctc_greedy_decode_with_timestamps(lg)


def test_beam_search_matches_reference(g):
    """decode.py:128-217 against the restatement fed with the reference's log-prob table."""
    rs = np.random.RandomState(5)
    for i, (B, L, V, W, blank) in enumerate([(2, 18, 9, 4, 0), (1, 10, 4, 6, 1), (2, 9, 7, 1, 0), (1, 14, 5, 3, 4)]):
        lg = (np.round(rs.standard_normal((B, L, V)) * 3.0) / 3.0).astype(np.float32)
        lp = torch.log_softmax(torch.from_numpy(lg), dim=-1).numpy()
        got = O.ctc_beam_search(lg, W, blank, log_probs=lp)
        assert recorded(g, f"beam_{i}") == got


def test_non_default_local_stack_shapes(g):
    """A config whose LOCAL stack differs from the global one (ssm_kernel_size 3, expand_ratio 1, 3 layers, state 32):
    GlobalSSM keeps expand_ratio 2 / kernel_size 4 whatever the config says (ssm.py:529-538).  The product's parameter
    tree must draw the same tensors as the reference and the oracle (shape-driven) must follow it."""
    import velocity_asr
    kw = dict(ssm_layers=3, ssm_state_dim=32, ssm_expand_ratio=1, ssm_kernel_size=3, scan_mode="sequential")
    torch.manual_seed(21)
    a = velocity_asr.VELOCITYASR(velocity_asr.VelocityASRConfig(**kw)).state_dict()
    assert FU.state_dict_fingerprint(a) == g["tree_nondefault"].tolist()
    assert a["local_ssm.layers.0.conv.weight"].shape[-1] == 3
    assert a["global_context.global_ssm.layers.0.conv.weight"].shape[-1] == 4
    assert a["global_context.global_ssm.layers.0.ssm.in_proj.weight"].shape[0] == 2 * 2 * 192
    sd = FU.amplify_state_dict(a, seed=4)
    audio = FU.synth_audio(2, 12000, seed=8)
    mel = g["nondefault_mel"]
    assert np.abs(O.log_mel(audio.numpy()) - mel).max() < MEL_PIN
    got = O.forward(mel, {k: v.numpy() for k, v in sd.items()}, dict(kw))
    assert rel(got[:, ::8], g["nondefault_logits_sub"]) < LOGIT_PIN
