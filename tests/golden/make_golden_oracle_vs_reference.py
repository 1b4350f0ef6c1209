"""Generate tests/golden/oracle_vs_reference.npz, the expected values of tests/test_oracle_vs_reference.py.

Those checks ran live against the unmodified reference, which is not part of the repository, and skipped
wherever it was not installed.  They passed against it at the commit this file was generated from, with the
oracle and the product's parameter tree the values below were recorded from, so on the same seeded inputs:
  - the parameter trees (sha256 per tensor), greedy token ids, timestamps and beam results are EQUAL to the
    reference's (the live checks used torch.equal / ==);
  - mel is within 1e-4 absolute and logits within 5e-5 relative of the reference's.

    python tests/golden/make_golden_oracle_vs_reference.py

Inputs are regenerated from seeds on the test side; only outputs are stored: mel as float32 (it is the
oracle's input in the tests), logits every 8th frame as float64, ragged results as Python literals.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for p in (os.path.join(ROOT, "velocity-asr_b200"), os.path.join(ROOT, "oracle"), os.path.dirname(HERE)):
    sys.path.insert(0, p)
import fixtures_util as FU  # noqa: E402
import velocity_asr as va  # noqa: E402
import velocity_oracle as O  # noqa: E402

NONDEFAULT = dict(ssm_layers=3, ssm_state_dim=32, ssm_expand_ratio=1, ssm_kernel_size=3, scan_mode="sequential")


def plain(x):
    """numpy scalars -> Python numbers, so that repr() is a literal ast.literal_eval reads back."""
    if isinstance(x, (list, tuple)):
        return type(x)(plain(v) for v in x)
    if isinstance(x, np.integer):
        return int(x)
    if isinstance(x, np.floating):
        return float(x)
    return x


def tree(seed, **kw):
    torch.manual_seed(seed)
    return va.VELOCITYASR(va.VelocityASRConfig(**kw)).state_dict()


out = {}

# ---- test_mel_and_forward_fresh_seed ------------------------------------------------
mel = O.log_mel(FU.synth_audio(2, 24000, seed=321).numpy()).astype(np.float32)
out["mel"] = mel
for mode in ("sequential", "parallel"):
    sd = {k: v.numpy() for k, v in FU.amplify_state_dict(tree(5, scan_mode=mode), seed=9).items()}
    logits = O.forward(mel, sd, dict(scan_mode=mode))
    out[mode + "_logits_sub"] = logits[:, ::8]
    out[mode + "_tokens"] = np.array(repr(plain(O.ctc_greedy_decode(logits))))

# ---- test_product_parameter_tree_draws_reference_weights ----------------------------
out["tree_seed11"] = np.array(FU.state_dict_fingerprint(tree(11)))

# ---- test_timestamp_decode_matches_reference ----------------------------------------
rs = np.random.RandomState(3)
for i, (B, L, V) in enumerate([(5, 97, 6), (3, 1, 4), (2, 300, 3), (1, 33, 2)]):
    lg = rs.standard_normal((B, L, V)).astype(np.float32)
    lg[..., 0] += 0.8
    lg = np.repeat(lg, 2, axis=1)[:, :L]
    out[f"timestamps_{i}"] = np.array(repr(plain(O.ctc_greedy_decode_with_timestamps(lg))))

# ---- test_beam_search_matches_reference ---------------------------------------------
rs = np.random.RandomState(5)
for i, (B, L, V, W, blank) in enumerate([(2, 18, 9, 4, 0), (1, 10, 4, 6, 1), (2, 9, 7, 1, 0), (1, 14, 5, 3, 4)]):
    lg = (np.round(rs.standard_normal((B, L, V)) * 3.0) / 3.0).astype(np.float32)
    lp = torch.log_softmax(torch.from_numpy(lg), dim=-1).numpy()
    out[f"beam_{i}"] = np.array(repr(plain(O.ctc_beam_search(lg, W, blank, log_probs=lp))))

# ---- test_non_default_local_stack_shapes --------------------------------------------
sd_t = tree(21, **NONDEFAULT)
out["tree_nondefault"] = np.array(FU.state_dict_fingerprint(sd_t))
mel = O.log_mel(FU.synth_audio(2, 12000, seed=8).numpy()).astype(np.float32)
out["nondefault_mel"] = mel
sd = {k: v.numpy() for k, v in FU.amplify_state_dict(sd_t, seed=4).items()}
out["nondefault_logits_sub"] = O.forward(mel, sd, dict(NONDEFAULT))[:, ::8]

path = os.path.join(HERE, "oracle_vs_reference.npz")
np.savez_compressed(path, **out)
print(f"oracle_vs_reference.npz  {os.path.getsize(path) / 1024:.0f} KiB")
