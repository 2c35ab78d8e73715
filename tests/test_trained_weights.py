"""Every path against float64 on weights with the statistics of a trained checkpoint.

Every weight set the other tests use has random-init magnitudes.  A trained checkpoint can have sharp attention (large
|q||k|: the single fp16 pass of the default tcgen05 scores loses precision with it), a large key bias (softmax ignores it, but it
makes |k| larger), outlier residual channels, a wide spread of LayerNorm gains and BatchNorm variances near zero.  ``trained_sd``
builds seeded sets with each property on its own and all at once (SETS; its docstring gives the knobs), from
``make_state_dict(stress=True)``.  What each set reaches on the oracle in float64 over the crop-edge table of
test_tracking_edges.py (the CPU test asserts each value within a factor of two; top P: mean top attention probability):

   set            max|logit|  top P   max|resid|  max |A| / |B| of qkv, scores, pv, fc1, fc2, head conv1 .. conv4
   random_init    0.92        0.0036  1.6         3.1/0.14, 0.31/2, 0.0048/2.1, 3.4/0.14, 1.8/0.072, 2.7/0.14, 2.8/0.18, 2.4/0.23, 3.3/0.3
   logit4         4.6         0.0083  1.6         3.1/0.58, 0.88/7.5, 0.021/2.1, 3.4/0.14, 1.8/0.072, 2.7/0.14, 2.8/0.18, 2.4/0.23, 3.3/0.3
   logit16        17          0.11    1.6         3.1/1.2, 1.7/15, 0.6/2.2, 3.4/0.14, 1.8/0.072, 2.7/0.14, 2.8/0.18, 2.5/0.23, 3.3/0.3
   logit64        64          0.63    1.8         3.1/2.3, 3.5/31, 1/2.2, 3.4/0.14, 1.8/0.072, 2.7/0.14, 2.9/0.18, 2.6/0.23, 3.2/0.3
   key_bias       5           0.0036  1.6         3.1/0.14, 0.31/27, 0.0048/2.1, 3.4/0.14, 1.8/0.072, 2.7/0.14, 2.8/0.18, 2.4/0.23, 3.3/0.3
   outliers       0.7         0.0031  30          7.8/0.14, 0.18/1.4, 0.0032/1.5, 6.8/0.14, 1.5/0.072, 5.2/0.14, 2.5/0.18, 2.2/0.23, 1.6/0.3
   ln_spread      1.5         0.0036  2           8.9/0.14, 0.38/2.5, 0.0045/3.1, 5.1/0.14, 1.8/0.072, 6.1/0.14, 4.3/0.18, 4.2/0.23, 3.8/0.3
   bn_var         1.9         0.0059  1.7e+03     4.6/0.14, 0.4/2.5, 0.019/2.7, 4.7/0.14, 2.9/0.072, 4.6/0.14, 5.3/0.18, 5/0.23, 3.9/0.3
   all            19          0.0036  5.1e+04     8.7/0.89, 0.71/61, 0.0051/2.1, 8/0.14, 2/0.072, 2.2/0.14, 2.2/0.18, 1.5/0.23, 1.4/0.3

1. CPU.  Every set reaches its statistics and leaves the fp32 oracle finite.  The single-pass score emulation
   (tools/precision_budget.py) moves the maps at least 10x further from the three-term one on logit16, logit64 and key_bias than
   on random-init weights (1.6e-4, 1.5e-3 and 4.6e-5 against 3.2e-6), so the GPU comparison cannot pass there by accident.  The
   rule by which vt_finalize_weights picks the score pass (vt_api.cu: score_terms, restated in ``score_bound``) keeps every
   random-init seed below 1/16 of its threshold and sends logit16, logit64 and all to the three-term pass.

2. GPU, one run per weight set and implementation (simt, tcgen05, tcgen05_3term, and the generic configurations small and img of
   test_generic_edges.py).  Tight: the crop-edge table stepped once, every track's maps against float64 (q and k rounded to
   fp16 before q k^T where the handle takes the single pass), boxes and detail rows decoded exactly, and Engine.forward(taps=True)
   on three of its crops, each tap as max |err| / RMS of the float64 tap.  Contract: 1024 open-loop 720p tracks against plain
   float64, maps and boxes within 1e-2 abs / 1e-3 rel, the Hann-windowed arg-max equal except for ties below 1e-5.  Never silently
   wrong: every track has status 0 and meets the contract or has VT_TRACK_NUMERIC_RANGE with NaN maps; with the range fallback on,
   flagged tracks give the simt engine's bits and the others keep theirs.  Where the handle takes the three-term pass on tcgen05,
   its bits equal tcgen05_3term's.

   Before vt_finalize_weights chose the score pass, tcgen05 on logit64 put 3 of the 1024 boxes past the contract (maps 4.2e-4 /
   3.4e-4 / 2.9e-3 off float64; the single-pass column of the table next to VT_BLOCKS_TCGEN05 in include/vittrack_b200.h).  No
   set flags a track.  Maximum measured on an NVIDIA B200 at a 1000 W power limit over two runs (the tolerances in TOL are 3x,
   rounded up; the GPU tests of this file take 40 s):

   set            impl            score    size     offset   stem     blocks   | contract: score    size     offset
   random_init    simt            4.1e-07 2.2e-07 3.0e-06 2.8e-06 2.6e-06  |           5.7e-07 3.3e-07 3.3e-06
   random_init    tcgen05         5.4e-07 4.0e-07 8.7e-06 2.5e-06 7.8e-06  |           8.8e-07 7.7e-07 1.4e-05
   random_init    tcgen05_3term   5.5e-07 3.6e-07 8.9e-06 2.5e-06 7.9e-06  |           6.0e-07 4.9e-07 1.0e-05
   random_init    small           1.2e-06 8.9e-07 2.5e-06 2.7e-06 4.6e-06  |           1.4e-06 9.7e-07 3.1e-06
   random_init    img             2.0e-06 2.0e-06 7.4e-06 5.3e-06 1.3e-05  |           2.2e-06 2.3e-06 8.0e-06
   logit4         simt            3.6e-07 2.2e-07 3.7e-06 2.8e-06 2.3e-06  |           5.6e-07 3.7e-07 3.8e-06
   logit4         tcgen05         5.4e-07 4.2e-07 8.5e-06 2.5e-06 9.6e-06  |           3.5e-06 2.3e-06 3.9e-05
   logit4         tcgen05_3term   5.4e-07 4.5e-07 9.0e-06 2.5e-06 8.4e-06  |           6.4e-07 5.4e-07 1.0e-05
   logit4         small           1.3e-06 8.0e-07 2.3e-06 2.7e-06 4.7e-06  |           1.4e-06 9.6e-07 3.2e-06
   logit4         img             2.0e-06 2.2e-06 7.5e-06 5.3e-06 1.3e-05  |           2.4e-06 2.4e-06 8.4e-06
   logit16        simt            4.2e-07 3.5e-07 3.2e-06 2.8e-06 3.4e-06  |           5.5e-07 4.2e-07 3.5e-06
   logit16        tcgen05         6.3e-07 4.9e-07 1.5e-05 2.5e-06 1.1e-05  |           9.0e-07 1.1e-06 1.5e-05
   logit16        tcgen05_3term   6.3e-07 4.9e-07 1.5e-05 2.5e-06 1.1e-05  |           9.0e-07 1.1e-06 1.5e-05
   logit16        small           1.3e-06 9.0e-07 2.4e-06 2.7e-06 4.8e-06  |           1.4e-06 9.9e-07 3.0e-06
   logit16        img             2.4e-06 2.3e-06 8.0e-06 5.3e-06 1.3e-05  |           2.8e-06 2.6e-06 9.1e-06
   logit64        simt            4.2e-07 3.2e-07 3.2e-06 2.8e-06 3.3e-06  |           1.2e-06 6.1e-07 5.1e-06
   logit64        tcgen05         5.2e-07 5.9e-07 9.6e-06 2.5e-06 1.5e-05  |           1.0e-06 1.1e-06 1.3e-05
   logit64        tcgen05_3term   5.2e-07 5.9e-07 9.6e-06 2.5e-06 1.5e-05  |           1.0e-06 1.1e-06 1.3e-05
   logit64        small           1.5e-06 8.7e-07 3.1e-06 2.7e-06 5.3e-06  |           1.5e-06 1.6e-06 6.9e-06
   logit64        img             2.7e-06 2.5e-06 1.0e-05 5.3e-06 1.9e-05  |           3.6e-06 3.9e-06 1.3e-05
   key_bias       simt            4.2e-07 2.1e-07 2.8e-06 2.8e-06 2.4e-06  |           5.5e-07 4.0e-07 3.3e-06
   key_bias       tcgen05         5.3e-07 4.0e-07 8.3e-06 2.5e-06 7.7e-06  |           8.1e-06 5.6e-06 8.1e-05
   key_bias       tcgen05_3term   5.2e-07 4.2e-07 8.6e-06 2.5e-06 7.9e-06  |           6.0e-07 4.9e-07 9.6e-06
   key_bias       small           1.3e-06 8.6e-07 2.6e-06 2.7e-06 4.7e-06  |           1.4e-06 1.0e-06 3.1e-06
   key_bias       img             2.2e-06 2.0e-06 7.3e-06 5.3e-06 1.3e-05  |           2.2e-06 2.4e-06 8.4e-06
   outliers       simt            3.6e-07 2.2e-07 2.2e-06 6.1e-06 5.0e-06  |           4.2e-07 2.9e-07 2.7e-06
   outliers       tcgen05         4.3e-07 1.7e-07 3.0e-06 5.3e-06 4.7e-06  |           5.0e-07 2.0e-07 3.5e-06
   outliers       tcgen05_3term   4.1e-07 1.5e-07 3.0e-06 5.3e-06 4.7e-06  |           5.0e-07 2.0e-07 3.5e-06
   outliers       small           7.1e-07 5.2e-07 2.9e-06 9.1e-07 2.3e-06  |           8.5e-07 6.3e-07 2.9e-06
   outliers       img             2.1e-06 1.2e-06 3.4e-06 1.1e-06 2.7e-06  |           2.3e-06 1.2e-06 3.7e-06
   ln_spread      simt            4.9e-07 5.0e-07 3.2e-06 2.8e-06 3.2e-06  |           6.6e-07 5.9e-07 3.5e-06
   ln_spread      tcgen05         5.7e-07 7.1e-07 3.4e-06 2.5e-06 8.5e-06  |           1.5e-06 1.3e-06 1.2e-05
   ln_spread      tcgen05_3term   4.6e-07 6.7e-07 3.8e-06 2.5e-06 6.3e-06  |           5.5e-07 7.7e-07 3.9e-06
   ln_spread      small           1.2e-06 1.4e-06 5.2e-06 2.7e-06 8.2e-06  |           1.2e-06 1.5e-06 6.7e-06
   ln_spread      img             2.1e-06 2.6e-06 8.5e-06 5.3e-06 1.1e-05  |           2.0e-06 2.6e-06 8.9e-06
   bn_var         simt            5.9e-07 4.2e-07 2.9e-06 2.8e-06 3.2e-06  |           6.6e-07 4.6e-07 4.3e-06
   bn_var         tcgen05         8.1e-07 5.3e-07 6.0e-06 6.9e-06 7.2e-06  |           9.6e-07 6.3e-07 8.0e-06
   bn_var         tcgen05_3term   8.4e-07 5.3e-07 5.7e-06 6.9e-06 7.2e-06  |           9.9e-07 6.2e-07 8.0e-06
   bn_var         small           1.1e-06 1.4e-06 7.3e-06 1.2e-05 1.2e-05  |           1.4e-06 2.1e-06 9.7e-06
   bn_var         img             2.8e-06 2.5e-06 1.4e-05 2.5e-05 2.6e-05  |           3.8e-06 2.9e-06 1.7e-05
   all            simt            2.6e-07 1.6e-07 1.1e-06 5.6e-06 4.8e-06  |           4.2e-07 2.2e-07 1.4e-06
   all            tcgen05         4.2e-07 1.8e-07 1.6e-06 4.3e-06 4.1e-06  |           4.6e-07 2.3e-07 1.8e-06
   all            tcgen05_3term   4.2e-07 1.8e-07 1.6e-06 4.3e-06 4.1e-06  |           4.6e-07 2.3e-07 1.8e-06
   all            small           4.7e-07 7.1e-07 2.8e-06 1.1e-06 1.6e-06  |           6.0e-07 9.5e-07 2.9e-06
   all            img             1.9e-06 2.6e-06 1.2e-05 1.6e-06 2.8e-06  |           2.1e-06 2.8e-06 1.3e-05

   The bn_var and all sets condition the model worse (the stem's BatchNorms normalise near-constant channels), so even simt
   is 1e-4 .. 1e-3 off float64 there.

Mutants (profiles/experiments/trained_weights_mutants.diff): tcgen05_3term built with a single-pass score, and one dropped split
term in the block kernel's qkv or fc2 contraction; each makes tests of this file fail (that diff lists which).
"""
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import vt_oracle as O
from test_generic_edges import CONFIGS, _tap_errors, make_cfg
from test_scale_invariance import Operands
from test_tracking_edges import MAPS, Model64, Tracks, _crops, _frames, _step, _table_specs, assert_decode_exact, exact_decode

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
from precision_budget import SplitModel  # noqa: E402

VT_TRACK_NUMERIC_RANGE = 3
ABS_TOL, REL_TOL = 1e-2, 1e-3          # the parity contract: maps and boxes
TIE_GAP = 1e-5                         # float64 top-1 - top-2 of the Hann-windowed score below this is a tie

# ------------------------------------------------------------------------------------------------
# the weight sets
# ------------------------------------------------------------------------------------------------
OUTLIERS = (200.0, 120.0)              # the two outlier channels' bias, in units of the RMS of the stem's tokens
SETS = {
    "random_init": {},
    "logit4": dict(logit=4.0),
    "logit16": dict(logit=16.0),
    "logit64": dict(logit=64.0),
    "key_bias": dict(key_bias=16.0),
    "outliers": dict(outliers=OUTLIERS),
    "ln_spread": dict(ln_spread=True),
    "bn_var": dict(bn_var=True),
    "all": dict(logit=16.0, key_bias=16.0, outliers=OUTLIERS, ln_spread=True, bn_var=True),
}
# what each set reaches on the oracle in float64 over the crop-edge table (module docstring); asserted within a factor of two
STATS = {
    "random_init": dict(max_logit=0.92, top_prob=0.0036, max_resid=1.6, qkv_A=3.1, qkv_B=0.14, scores_A=0.31, scores_B=2.0, pv_A=0.0048, pv_B=2.1, proj_A=2.0, proj_B=0.14, fc1_A=3.4, fc1_B=0.14, fc2_A=1.8, fc2_B=0.072, conv1_A=2.7, conv1_B=0.14, conv2_A=2.8, conv2_B=0.18, conv3_A=2.4, conv3_B=0.23, conv4_A=3.3, conv4_B=0.3),
    "logit4": dict(max_logit=4.6, top_prob=0.0083, max_resid=1.6, qkv_A=3.1, qkv_B=0.58, scores_A=0.88, scores_B=7.5, pv_A=0.021, pv_B=2.1, proj_A=2.0, proj_B=0.14, fc1_A=3.4, fc1_B=0.14, fc2_A=1.8, fc2_B=0.072, conv1_A=2.7, conv1_B=0.14, conv2_A=2.8, conv2_B=0.18, conv3_A=2.4, conv3_B=0.23, conv4_A=3.3, conv4_B=0.3),
    "logit16": dict(max_logit=17.0, top_prob=0.11, max_resid=1.6, qkv_A=3.1, qkv_B=1.2, scores_A=1.7, scores_B=15.0, pv_A=0.6, pv_B=2.2, proj_A=2.1, proj_B=0.14, fc1_A=3.4, fc1_B=0.14, fc2_A=1.8, fc2_B=0.072, conv1_A=2.7, conv1_B=0.14, conv2_A=2.8, conv2_B=0.18, conv3_A=2.5, conv3_B=0.23, conv4_A=3.3, conv4_B=0.3),
    "logit64": dict(max_logit=64.0, top_prob=0.63, max_resid=1.8, qkv_A=3.1, qkv_B=2.3, scores_A=3.5, scores_B=31.0, pv_A=1.0, pv_B=2.2, proj_A=2.1, proj_B=0.14, fc1_A=3.4, fc1_B=0.14, fc2_A=1.8, fc2_B=0.072, conv1_A=2.7, conv1_B=0.14, conv2_A=2.9, conv2_B=0.18, conv3_A=2.6, conv3_B=0.23, conv4_A=3.2, conv4_B=0.3),
    "key_bias": dict(max_logit=5.0, top_prob=0.0036, max_resid=1.6, qkv_A=3.1, qkv_B=0.14, scores_A=0.31, scores_B=27.0, pv_A=0.0048, pv_B=2.1, proj_A=2.0, proj_B=0.14, fc1_A=3.4, fc1_B=0.14, fc2_A=1.8, fc2_B=0.072, conv1_A=2.7, conv1_B=0.14, conv2_A=2.8, conv2_B=0.18, conv3_A=2.4, conv3_B=0.23, conv4_A=3.3, conv4_B=0.3),
    "outliers": dict(max_logit=0.7, top_prob=0.0031, max_resid=30.0, qkv_A=7.8, qkv_B=0.14, scores_A=0.18, scores_B=1.4, pv_A=0.0032, pv_B=1.5, proj_A=1.5, proj_B=0.14, fc1_A=6.8, fc1_B=0.14, fc2_A=1.5, fc2_B=0.072, conv1_A=5.2, conv1_B=0.14, conv2_A=2.5, conv2_B=0.18, conv3_A=2.2, conv3_B=0.23, conv4_A=1.6, conv4_B=0.3),
    "ln_spread": dict(max_logit=1.5, top_prob=0.0036, max_resid=2.0, qkv_A=8.9, qkv_B=0.14, scores_A=0.38, scores_B=2.5, pv_A=0.0045, pv_B=3.1, proj_A=3.0, proj_B=0.14, fc1_A=5.1, fc1_B=0.14, fc2_A=1.8, fc2_B=0.072, conv1_A=6.1, conv1_B=0.14, conv2_A=4.3, conv2_B=0.18, conv3_A=4.2, conv3_B=0.23, conv4_A=3.8, conv4_B=0.3),
    "bn_var": dict(max_logit=1.9, top_prob=0.0059, max_resid=1700.0, qkv_A=4.6, qkv_B=0.14, scores_A=0.4, scores_B=2.5, pv_A=0.019, pv_B=2.7, proj_A=1.9, proj_B=0.14, fc1_A=4.7, fc1_B=0.14, fc2_A=2.9, fc2_B=0.072, conv1_A=4.6, conv1_B=0.14, conv2_A=5.3, conv2_B=0.18, conv3_A=5.0, conv3_B=0.23, conv4_A=3.9, conv4_B=0.3),
    "all": dict(max_logit=19.0, top_prob=0.0036, max_resid=51000.0, qkv_A=8.7, qkv_B=0.89, scores_A=0.71, scores_B=61.0, pv_A=0.0051, pv_B=2.1, proj_A=2.0, proj_B=0.14, fc1_A=8.0, fc1_B=0.14, fc2_A=2.0, fc2_B=0.072, conv1_A=2.2, conv1_B=0.14, conv2_A=2.2, conv2_B=0.18, conv3_A=1.5, conv3_B=0.23, conv4_A=1.4, conv4_B=0.3),
}

# implementation -> (blocks_impl, generic configuration of test_generic_edges.py or None for vit_48_h32)
IMPLS = {"simt": ("simt", None), "tcgen05": ("tcgen05", None), "tcgen05_3term": ("tcgen05_3term", None),
         "small": ("tcgen05", "small"), "img": ("tcgen05", "img")}
SEED = 17
# max |device - float64| per map, and max |err| / RMS per tap (stem; blocks and final LayerNorm): 3x the measured maximum
TOL = {
    "simt": {
        "random_init": dict(score_map=1.3e-06, size_map=6.7e-07, offset_map=9.1e-06, stem=8.4e-06, blocks=7.9e-06),
        "logit4": dict(score_map=1.1e-06, size_map=6.7e-07, offset_map=1.2e-05, stem=8.4e-06, blocks=6.8e-06),
        "logit16": dict(score_map=1.3e-06, size_map=1.1e-06, offset_map=9.6e-06, stem=8.4e-06, blocks=1.1e-05),
        "logit64": dict(score_map=1.3e-06, size_map=9.8e-07, offset_map=9.7e-06, stem=8.4e-06, blocks=1e-05),
        "key_bias": dict(score_map=1.3e-06, size_map=6.4e-07, offset_map=8.5e-06, stem=8.4e-06, blocks=7.3e-06),
        "outliers": dict(score_map=1.1e-06, size_map=6.8e-07, offset_map=6.6e-06, stem=1.9e-05, blocks=1.6e-05),
        "ln_spread": dict(score_map=1.5e-06, size_map=1.6e-06, offset_map=9.6e-06, stem=8.4e-06, blocks=9.5e-06),
        "bn_var": dict(score_map=1.8e-06, size_map=1.3e-06, offset_map=8.9e-06, stem=8.5e-06, blocks=9.6e-06),
        "all": dict(score_map=8e-07, size_map=4.9e-07, offset_map=3.3e-06, stem=1.7e-05, blocks=1.5e-05),
    },
    "tcgen05": {
        "random_init": dict(score_map=1.7e-06, size_map=1.2e-06, offset_map=2.7e-05, stem=7.4e-06, blocks=2.4e-05),
        "logit4": dict(score_map=1.7e-06, size_map=1.3e-06, offset_map=2.6e-05, stem=7.4e-06, blocks=2.9e-05),
        "logit16": dict(score_map=1.9e-06, size_map=1.5e-06, offset_map=4.4e-05, stem=7.4e-06, blocks=3.4e-05),
        "logit64": dict(score_map=1.6e-06, size_map=1.8e-06, offset_map=2.9e-05, stem=7.4e-06, blocks=4.5e-05),
        "key_bias": dict(score_map=1.6e-06, size_map=1.2e-06, offset_map=2.5e-05, stem=7.4e-06, blocks=2.4e-05),
        "outliers": dict(score_map=1.3e-06, size_map=5.1e-07, offset_map=9e-06, stem=1.6e-05, blocks=1.5e-05),
        "ln_spread": dict(score_map=1.8e-06, size_map=2.2e-06, offset_map=1.1e-05, stem=7.4e-06, blocks=2.6e-05),
        "bn_var": dict(score_map=2.5e-06, size_map=1.6e-06, offset_map=1.8e-05, stem=2.1e-05, blocks=2.2e-05),
        "all": dict(score_map=1.3e-06, size_map=5.5e-07, offset_map=4.8e-06, stem=1.3e-05, blocks=1.3e-05),
    },
    "tcgen05_3term": {
        "random_init": dict(score_map=1.7e-06, size_map=1.1e-06, offset_map=2.7e-05, stem=7.4e-06, blocks=2.4e-05),
        "logit4": dict(score_map=1.7e-06, size_map=1.4e-06, offset_map=2.7e-05, stem=7.4e-06, blocks=2.6e-05),
        "logit16": dict(score_map=1.9e-06, size_map=1.5e-06, offset_map=4.4e-05, stem=7.4e-06, blocks=3.4e-05),
        "logit64": dict(score_map=1.6e-06, size_map=1.8e-06, offset_map=2.9e-05, stem=7.4e-06, blocks=4.5e-05),
        "key_bias": dict(score_map=1.6e-06, size_map=1.3e-06, offset_map=2.6e-05, stem=7.4e-06, blocks=2.4e-05),
        "outliers": dict(score_map=1.3e-06, size_map=4.6e-07, offset_map=8.9e-06, stem=1.6e-05, blocks=1.5e-05),
        "ln_spread": dict(score_map=1.4e-06, size_map=2.1e-06, offset_map=1.2e-05, stem=7.4e-06, blocks=2e-05),
        "bn_var": dict(score_map=2.6e-06, size_map=1.6e-06, offset_map=1.8e-05, stem=2.1e-05, blocks=2.2e-05),
        "all": dict(score_map=1.3e-06, size_map=5.5e-07, offset_map=4.8e-06, stem=1.3e-05, blocks=1.3e-05),
    },
    "small": {
        "random_init": dict(score_map=3.7e-06, size_map=2.7e-06, offset_map=7.6e-06, stem=8.1e-06, blocks=1.4e-05),
        "logit4": dict(score_map=3.8e-06, size_map=2.4e-06, offset_map=7e-06, stem=8.1e-06, blocks=1.4e-05),
        "logit16": dict(score_map=3.9e-06, size_map=2.7e-06, offset_map=7.3e-06, stem=8.1e-06, blocks=1.5e-05),
        "logit64": dict(score_map=4.4e-06, size_map=2.7e-06, offset_map=9.3e-06, stem=8.1e-06, blocks=1.6e-05),
        "key_bias": dict(score_map=3.9e-06, size_map=2.6e-06, offset_map=7.9e-06, stem=8.1e-06, blocks=1.5e-05),
        "outliers": dict(score_map=2.2e-06, size_map=1.6e-06, offset_map=8.8e-06, stem=2.8e-06, blocks=7e-06),
        "ln_spread": dict(score_map=3.6e-06, size_map=4.2e-06, offset_map=1.6e-05, stem=8.1e-06, blocks=2.5e-05),
        "bn_var": dict(score_map=3.3e-06, size_map=4.2e-06, offset_map=2.3e-05, stem=3.7e-05, blocks=3.6e-05),
        "all": dict(score_map=1.5e-06, size_map=2.2e-06, offset_map=8.4e-06, stem=3.4e-06, blocks=4.8e-06),
    },
    "img": {
        "random_init": dict(score_map=6.1e-06, size_map=6.1e-06, offset_map=2.3e-05, stem=1.6e-05, blocks=3.8e-05),
        "logit4": dict(score_map=6.2e-06, size_map=6.5e-06, offset_map=2.3e-05, stem=1.6e-05, blocks=4e-05),
        "logit16": dict(score_map=7.3e-06, size_map=7.1e-06, offset_map=2.5e-05, stem=1.6e-05, blocks=4.1e-05),
        "logit64": dict(score_map=8.1e-06, size_map=7.5e-06, offset_map=3.2e-05, stem=1.6e-05, blocks=5.9e-05),
        "key_bias": dict(score_map=6.6e-06, size_map=6.2e-06, offset_map=2.2e-05, stem=1.6e-05, blocks=3.8e-05),
        "outliers": dict(score_map=6.3e-06, size_map=3.6e-06, offset_map=1.1e-05, stem=3.3e-06, blocks=8.1e-06),
        "ln_spread": dict(score_map=6.3e-06, size_map=7.9e-06, offset_map=2.6e-05, stem=1.6e-05, blocks=3.4e-05),
        "bn_var": dict(score_map=8.5e-06, size_map=7.7e-06, offset_map=4.3e-05, stem=7.7e-05, blocks=7.7e-05),
        "all": dict(score_map=5.7e-06, size_map=7.9e-06, offset_map=3.7e-05, stem=4.8e-06, blocks=8.4e-06),
    },
}


def _shape(gen):
    """(C, heads, depth, head channels) of vit_48_h32 (gen None) or a generic configuration."""
    if gen is None:
        return O.EMBED_DIM, O.NUM_HEADS, O.DEPTH, O.HEAD_CHANNELS
    C, heads, depth, hc, _ = CONFIGS[gen]
    return C, heads, depth, hc


def _calibration_crops():
    """Two fixed (template, search) crop pairs on which the generator measures what it scales."""
    frames = O.synth_frames(2, 360, 640, seed=61, smooth=True)
    boxes = [[300.0, 150.0, 60.0, 40.0], [100.0, 200.0, 80.0, 50.0]]
    z = torch.cat([O.preprocess(O.sample_target_spec(frames[0], b, O.TEMPLATE_FACTOR, O.TEMPLATE_SIZE)[0]) for b in boxes])
    x = torch.cat([O.preprocess(O.sample_target_spec(frames[1], b, O.SEARCH_FACTOR, O.SEARCH_SIZE)[0]) for b in boxes])
    return z, x


class Recorder(Operands):
    """The oracle recording, per block, the operands of every split contraction (Operands) and the LayerNorm input of qkv."""

    def block(self, x, b):
        self.ops[f"resid{b}"] = x
        return super().block(x, b)


def record(sd, gen, z, x, double=True, device="cpu"):
    """Run the oracle (in float64 with ``double``) and return (its maps, its recorder)."""
    C, heads, depth, _ = _shape(gen)
    m = Recorder(sd, depth=depth, num_heads=heads)
    dt = torch.float64 if double else torch.float32
    m.sd = {k: v.to(device, dt) if v.is_floating_point() else v.to(device) for k, v in m.sd.items()}
    out = m.forward(z.to(device, dt), x.to(device, dt))
    return out, m


def bn_inputs(sd, gen, z, x):
    """Every BatchNorm's input on crops z, x: prefix of its conv -> [channels, values] (stem: template and search pooled)."""
    C, heads, depth, _ = _shape(gen)
    m = O.OracleModel(sd, depth=depth, num_heads=heads)
    out = {}
    for img in (z, x):
        t = img
        for i in range(4):
            p = f"patch_embed.net.{2 * i}."
            t = F.conv2d(t, m.sd[p + "c.weight"], None, stride=2, padding=1)
            out.setdefault(p, []).append(t.transpose(0, 1).reshape(t.shape[1], -1))
            t = F.batch_norm(t, m.sd[p + "bn.running_mean"], m.sd[p + "bn.running_var"], m.sd[p + "bn.weight"], m.sd[p + "bn.bias"],
                             False, 0.0, O.BN_EPS)
            t = F.hardswish(t) if i < 3 else t
    taps = {}
    m.forward(z, x, taps)
    feat = taps["tokens_norm"][:, -O.FEAT_SZ ** 2:].transpose(1, 2).reshape(-1, C, O.FEAT_SZ, O.FEAT_SZ)
    for tw in O.TOWERS:
        t = feat
        for i in range(4):
            p = f"box_head.conv{i + 1}_{tw}."
            t = F.conv2d(t, m.sd[p + "0.weight"], m.sd[p + "0.bias"], padding=1)
            out[p] = [t.transpose(0, 1).reshape(t.shape[1], -1)]
            t = F.relu(F.batch_norm(t, m.sd[p + "1.running_mean"], m.sd[p + "1.running_var"], m.sd[p + "1.weight"],
                                    m.sd[p + "1.bias"], False, 0.0, O.BN_EPS))
    return {p: torch.cat(v, 1) for p, v in out.items()}


def trained_sd(name, gen=None, seed=SEED):
    """A seeded weight set with trained-checkpoint statistics: ``make_state_dict(stress=True)`` with the knobs of SETS[name]:
    ln_spread  every LayerNorm gain log-uniform over [2^-6, 4], bias N(0, 0.5);
    bn_var     every stem BatchNorm's running variance log-uniform over [1e-4, 10], its channel's conv weights scaled so that this
               is the variance the channel has on the calibration crops, and the running mean set to the channel's mean there, as in
               a trained checkpoint.  Variances alone, with random-init weights, amplify each stem layer up to 100x: the residual
               reaches 5e5 and even the fp32 oracle's maps leave 1e-2 of float64.  The head's BatchNorms keep their statistics:
               calibrated the same way on two crops, they put raw offsets of 1e3 cells on other crops, where the fp32 oracle's
               boxes are already 1e-2 off float64;
    outliers   (a, b): two residual channels offset by a and b x the RMS of the stem's tokens, through the stem's last BatchNorm
               bias and block 0's projection bias;
    key_bias   b_k of every block set to a random direction with norm key_bias x the median ||W_k h|| (h: norm1's output);
    logit      q and k rows of every block's qkv (weights and bias) scaled together until max |q k^T / sqrt(d)| on the calibration
               crops reaches this value.
    The knobs are applied in this order and each one is calibrated on the model the earlier ones left."""
    knobs = SETS[name]
    C, heads, depth, hc = _shape(gen)
    sd = O.make_state_dict(seed=seed, stress=True, C=C, depth=depth, head_ch=hc)
    g = torch.Generator().manual_seed(seed + 1000)
    if knobs.get("ln_spread"):
        for k in [k for k in sd if k.endswith("norm1.weight") or k.endswith("norm2.weight") or k == "norm.weight"]:
            sd[k] = torch.exp2(torch.rand(sd[k].shape, generator=g) * 8 - 6)
            b = k[:-len("weight")] + "bias"
            sd[b] = torch.randn(sd[b].shape, generator=g) * 0.5
    z, x = _calibration_crops()
    if knobs.get("bn_var"):
        for p, v in bn_inputs(sd, gen, z, x).items():
            if not p.startswith("patch"):
                continue
            bn, conv = (p + "bn.", p + "c.") if p.startswith("patch") else (p + "1.", p + "0.")
            var = 10.0 ** (torch.rand(v.shape[0], generator=g) * 5 - 4)
            s = (var / v.var(dim=1)).sqrt()
            sd[conv + "weight"] = sd[conv + "weight"] * s[:, None, None, None]
            if conv + "bias" in sd:
                sd[conv + "bias"] = sd[conv + "bias"] * s
            sd[bn + "running_mean"] = v.mean(dim=1) * s
            sd[bn + "running_var"] = var
    if knobs.get("outliers"):
        _, m = record(sd, gen, z, x, double=False)
        rms = float(m.ops["resid0"].pow(2).mean().sqrt())
        a, b = knobs["outliers"]
        sd["patch_embed.net.6.bn.bias"][3] += a * rms
        sd["blocks.0.attn.proj.bias"][C - 5] += b * rms
    if knobs.get("key_bias"):
        _, m = record(sd, gen, z, x, double=False)
        for blk in range(depth):
            h = m.ops[f"qkv{blk}"][0]
            wk = sd[f"blocks.{blk}.attn.qkv.weight"][C:2 * C]
            typical = float((h @ wk.t()).norm(dim=-1).median())
            d = torch.randn(C, generator=g)
            sd[f"blocks.{blk}.attn.qkv.bias"][C:2 * C] = d / d.norm() * knobs["key_bias"] * typical
    if knobs.get("logit"):
        _, m = record(sd, gen, z, x, double=False)
        for blk in range(depth):
            q, kt = m.ops[f"scores{blk}"]
            t = (knobs["logit"] / float((q @ kt).abs().max())) ** 0.5
            for k in (f"blocks.{blk}.attn.qkv.weight", f"blocks.{blk}.attn.qkv.bias"):
                sd[k][:2 * C] *= t
    return sd


SHARP_SCORES = 512.0       # vt_api.cu: kSharpScores


def score_bound(sd, C=O.EMBED_DIM, depth=O.DEPTH):
    """vt_api.cu (score_terms), restated: max over blocks of the bound (||W_q||_2 R + ||b_q||)(||W_k||_2 R + ||b_k||) / sqrt(C) on
    |q . k| / sqrt(C), R = sqrt(C) max|gamma| + ||beta|| bounding norm1's output."""
    out = 0.0
    for b in range(depth):
        p = f"blocks.{b}."
        g, beta = sd[p + "norm1.weight"].double(), sd[p + "norm1.bias"].double()
        w, bias = sd[p + "attn.qkv.weight"].double(), sd[p + "attn.qkv.bias"].double()
        R = C ** 0.5 * float(g.abs().max()) + float(beta.norm())
        q = float(torch.linalg.matrix_norm(w[:C], 2)) * R + float(bias[:C].norm())
        k = float(torch.linalg.matrix_norm(w[C:2 * C], 2)) * R + float(bias[C:2 * C].norm())
        out = max(out, q * k / C ** 0.5)
    return out


def single_pass(impl, sd):
    """Whether a handle of ``impl`` computes q k^T as one fp16 pass on these weights (vt_finalize_weights)."""
    return impl == "tcgen05" and score_bound(sd) <= SHARP_SCORES


def statistics(m, depth):
    """What a weight set reaches, from a recorder run: max |logit|, mean top attention probability, max |residual| and the
    max |operand| of every split contraction (A, B) over blocks and towers."""
    st = {"max_logit": 0.0, "top_prob": 0.0, "max_resid": 0.0}
    for b in range(depth):
        q, kt = m.ops[f"scores{b}"]
        st["max_logit"] = max(st["max_logit"], float((q @ kt).abs().max()))
        st["top_prob"] += float(m.ops[f"pv{b}"][0].max(dim=-1).values.mean()) / depth
        st["max_resid"] = max(st["max_resid"], float(m.ops[f"resid{b}"].abs().max()))
    for op in ("qkv", "scores", "pv", "proj", "fc1", "fc2", "conv1", "conv2", "conv3", "conv4"):
        keys = [f"{op}_{t}" for t in O.TOWERS] if op.startswith("conv") else [f"{op}{b}" for b in range(depth)]
        st[f"{op}_A"] = max(float(m.ops[k][0].abs().max()) for k in keys)
        st[f"{op}_B"] = max(float(m.ops[k][1].abs().max()) for k in keys)
    return st


# ------------------------------------------------------------------------------------------------
# fixtures and references
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def frames():
    return _frames()


@pytest.fixture(scope="module")
def table(frames):
    return Tracks(frames, _table_specs())


_SD = {}


def weights(name, gen=None):
    if (name, gen) not in _SD:
        _SD[(name, gen)] = trained_sd(name, gen)
    return _SD[(name, gen)]


def ref64(sd, gen, z, x, fp16_scores=False, taps=None, device="cpu"):
    """The oracle's maps in float64 (``fp16_scores``: q and k rounded to fp16 before q k^T, as the tcgen05 blocks do)."""
    C, heads, depth, _ = _shape(gen)
    if gen is None:
        m = Model64(sd, fp16_scores)
    else:
        m = O.OracleModel(sd, depth=depth, num_heads=heads)
        m.sd = {k: v.double() if v.is_floating_point() else v for k, v in m.sd.items()}
    m.to(device)
    out = m.forward(z.to(device, torch.float64), x.to(device, torch.float64), taps)
    return {k: v.cpu() for k, v in out.items()}


# ------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(SETS))
def test_set_reaches_its_statistics_and_oracle_stays_finite(table, name):
    torch.set_num_threads(16)
    z, x = _crops(table)
    sd = weights(name)
    _, m = record(sd, None, z, x)
    st = statistics(m, O.DEPTH)
    print(f"\n[{name}]", {k: f"{v:.3g}" for k, v in st.items()})
    for k, want in STATS[name].items():
        assert want / 2 <= st[k] <= want * 2, (name, k, st[k], want)
    out = O.OracleModel(sd).forward(z, x)
    for k, v in out.items():
        assert torch.isfinite(v).all(), (name, k)


def test_sharp_scores_rule_separates_random_init_from_sharp_sets():
    """Random-init weights (those of bench.py, smoke() and every other test) keep the single-pass scores; the sets whose
    single-pass error reaches the parity contract (logit64 on a B200: boxes 1e-2 off) take the three-term pass."""
    bounds = {name: score_bound(weights(name)) for name in SETS}
    print("\nscore bound:", {k: f"{v:.0f}" for k, v in bounds.items()})
    for seed in range(8):
        for stress in (False, True):
            assert score_bound(O.make_state_dict(seed=seed, stress=stress)) < SHARP_SCORES / 16, (seed, stress)
    assert bounds["random_init"] < SHARP_SCORES / 16
    assert {n for n, b in bounds.items() if b > SHARP_SCORES} == {"logit16", "logit64", "all"}, bounds


def _split_maps(sd, z, x, drops):
    return SplitModel(sd, drops).forward(z, x)


@pytest.mark.parametrize("name", ["logit16", "logit64", "key_bias"])
def test_single_pass_scores_differ_from_three_terms(table, name):
    """The single-pass score emulation moves the maps at least 10x further from the three-term one than on random-init weights,
    so the GPU comparison of tcgen05 with plain float64 cannot pass on these sets by accident."""
    torch.set_num_threads(16)
    z, x = _crops(table)
    diff = {}
    for s in ("random_init", name):
        sd = weights(s)
        three, one = _split_maps(sd, z, x, {}), _split_maps(sd, z, x, {"scores": "both"})
        diff[s] = max(float((three[k] - one[k]).abs().max()) for k in MAPS)
    print(f"\nsingle-pass - three-term, max over maps: {diff}")
    assert diff[name] >= 10 * diff["random_init"], diff


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
FWD_ROWS = ["c256_identity_top_left", "odd_interior_half", "uhd_interior"]
N_CONTRACT = 1024


def _engine(impl, n):
    from vittracker_b200 import load_cfg
    from vittracker_b200.engine import Engine
    blocks, gen = IMPLS[impl]
    if gen is None:
        return Engine(load_cfg(), max_tracks=n, blocks_impl=blocks)
    C, heads, depth, hc, _ = CONFIGS[gen]
    return Engine(make_cfg(C, heads, hc), max_tracks=n, blocks_impl=blocks, depth=depth)


def _map_errors(maps, want, ok):
    """max |device - float64| per map over the tracks ``ok``: (value, track index)."""
    out = {}
    for k in MAPS:
        err = np.abs(maps[k].astype(np.float64) - want[k].numpy()).reshape(len(ok), -1).max(1)
        err[~ok] = 0.0
        i = int(err.argmax())
        out[k] = (float(err[i]), i)
    return out


def _check_flagged(maps, out, det, ok, tag):
    """Every track is status 0 or VT_TRACK_NUMERIC_RANGE; a flagged one has NaN maps and confidence -1."""
    st = det[:, 6]
    assert np.isin(st, (0, VT_TRACK_NUMERIC_RANGE)).all(), (tag, np.unique(st))
    for k in MAPS:
        assert np.isnan(maps[k][~ok]).all(), (tag, k)
    assert (out[~ok, 4] == -1.0).all(), tag


@pytest.mark.gpu
@pytest.mark.parametrize("impl", list(IMPLS))
@pytest.mark.parametrize("name", list(SETS))
def test_step_and_taps_against_float64(table, name, impl):
    """The crop-edge table stepped once and three of its crops through Engine.forward(taps=True), against float64."""
    blocks, gen = IMPLS[impl]
    sd = weights(name, gen)
    dev = torch.device("cuda")
    e = _engine(impl, table.n)
    e.load_state_dict(sd)
    maps, out, det = _step(e, table.device(e.device), table.n)
    ok = det[:, 6] == 0
    _check_flagged(maps, out, det, ok, (name, impl))
    z, x = _crops(table)
    fp16_scores = single_pass(impl, sd)
    want = ref64(sd, gen, z, x, fp16_scores=fp16_scores, device=dev)
    err = _map_errors(maps, want, ok)
    rows = [table.labels.index(r) for r in FWD_ROWS]
    taps64 = {}
    ref64(sd, gen, z[rows], x[rows], fp16_scores=fp16_scores, taps=taps64, device=dev)
    got = e.forward(z[rows], x[rows], taps=True)
    torch.cuda.synchronize()
    taps = _tap_errors(got["taps"], {k: v.cpu() for k, v in taps64.items()}, _shape(gen)[2]) if ok[rows].all() else {}
    print(f"\nTIGHT {name} {impl} single_pass={fp16_scores} flagged={int((~ok).sum())}/{table.n}",
          {k: f"{v[0]:.2e}" for k, v in err.items()}, {k: f"{v:.2e}" for k, v in taps.items()})
    tol = TOL[impl][name]
    for k in MAPS:
        assert err[k][0] <= tol[k], (name, impl, k, err[k][0], table.labels[err[k][1]])
    for k, v in taps.items():
        assert v <= tol["stem" if k == "stem" else "blocks"], (name, impl, k, v, taps)
    keep = np.flatnonzero(ok)
    assert_decode_exact({k: v[keep] for k, v in maps.items()}, out[keep], det[keep], table, rows=keep, tag=f"{name} {impl}")


@pytest.fixture(scope="module")
def contract_tracks(frames):
    """N_CONTRACT open-loop tracks on the 720p frames: template box on frame 0, search box on frame 1."""
    H, W = 720, 1280
    tb, sb = O.synth_boxes(N_CONTRACT, H, W, seed=71), O.synth_boxes(N_CONTRACT, H, W, seed=72)
    return Tracks(frames, [(f"open{i}", "hd", i % 4, list(tb[i]), list(sb[i])) for i in range(N_CONTRACT)])


_CROPS, _BITS = {}, {}


def _device_crops(e, tr, d):
    """The tracks' oracle crops, cut by vt_crop_normalize (bit-exact with the oracle's: test_gpu_parity.py)."""
    if "c" not in _CROPS:
        z = e.crop_normalize(d.buf, d.off[0], d.hw, d.tbox, O.TEMPLATE_FACTOR, O.TEMPLATE_SIZE)["tensors"]
        x = e.crop_normalize(d.buf, d.off[1], d.hw, d.sbox, O.SEARCH_FACTOR, O.SEARCH_SIZE)["tensors"]
        _CROPS["c"] = (z, x)
    return _CROPS["c"]


def _bits(name, impl, tr):
    """The step of a vit_48_h32 engine of ``impl`` on the tracks (cached)."""
    if (name, impl) not in _BITS:
        e = _engine(impl, tr.n)
        e.load_state_dict(weights(name))
        _BITS[(name, impl)] = _step(e, tr.device(e.device), tr.n)
        del e
    return _BITS[(name, impl)]


def _same_bits(got, want, rows, what):
    (gm, go, gd), (wm, wo, wd) = got, want
    for k in MAPS:
        assert np.array_equal(gm[k][rows].view(np.uint32), wm[k][rows].view(np.uint32)), (what, k)
    assert np.array_equal(go[rows], wo[rows]) and np.array_equal(gd[rows], wd[rows]), what


@pytest.mark.gpu
@pytest.mark.parametrize("impl", list(IMPLS))
@pytest.mark.parametrize("name", list(SETS))
def test_contract_and_never_silently_wrong(contract_tracks, name, impl):
    """Every track has status 0 and meets the parity contract against plain float64 (maps and boxes within 1e-2 abs / 1e-3 rel,
    the Hann-windowed arg-max equal except for ties below 1e-5), or has VT_TRACK_NUMERIC_RANGE with NaN maps.  With the range
    fallback on, a flagged track gives the simt engine's bits."""
    tr = contract_tracks
    blocks, gen = IMPLS[impl]
    sd = weights(name, gen)
    e = _engine(impl, tr.n)
    e.load_state_dict(sd)
    d = tr.device(e.device)
    maps, out, det = _step(e, d, tr.n)
    ok = det[:, 6] == 0
    _check_flagged(maps, out, det, ok, (name, impl))
    z, x = _device_crops(e, tr, d)
    want = ref64(sd, gen, z, x, device=e.device)
    win = O.hann2d(16, 16).double().reshape(1, -1)
    resp = (win * want["score_map"].reshape(tr.n, -1)).numpy()
    top2 = np.sort(resp, axis=1)[:, -2:]
    tie = (top2[:, 1] - top2[:, 0]) < TIE_GAP
    flips, far = [], {}
    for k in MAPS:
        w = want[k].numpy()
        bad = (np.abs(maps[k] - w) > ABS_TOL + REL_TOL * np.abs(w)).reshape(tr.n, -1).any(1) & ok
        if bad.any():
            far[k] = list(np.flatnonzero(bad))
    for i in np.flatnonzero(ok):
        if tie[i]:
            continue
        if int(det[i, 5]) != int(resp[i].argmax()):
            flips.append(i)
            continue
        H, W = (int(v) for v in tr.hw[i])
        wb, _ = exact_decode(want["score_map"][i], want["size_map"][i], want["offset_map"][i], tr.sbox[i], H, W)
        if not np.allclose(out[i, :4], wb[:4], atol=ABS_TOL, rtol=REL_TOL):
            far.setdefault("box", []).append(i)
    err = _map_errors(maps, want, ok)
    print(f"\nCONTRACT {name} {impl} flagged={int((~ok).sum())}/{tr.n} ties={int(tie.sum())} flips={len(flips)}",
          {k: f"{v[0]:.2e}" for k, v in err.items()}, {k: len(v) for k, v in far.items()})
    assert not flips, (name, impl, f"{len(flips)} arg-max flips", flips[:8])
    assert not far, (name, impl, {k: v[:8] for k, v in far.items()})
    if impl == "tcgen05" and not single_pass(impl, sd):
        _same_bits((maps, out, det), _bits(name, "tcgen05_3term", tr), np.arange(tr.n), (name, "sharp scores: tcgen05_3term's bits"))
    if gen is None and blocks != "simt":
        e.set_range_fallback(True)
        got = _step(e, d, tr.n)
        _same_bits(got, _bits(name, "simt", tr), np.flatnonzero(~ok), (name, impl, "fallback: simt bits"))
        _same_bits(got, (maps, out, det), np.flatnonzero(ok), (name, impl, "fallback: unflagged tracks unchanged"))
