"""Host-side checks of the recogniser's vocabulary limit (no GPU needed)."""
import pytest

from aptai_b200 import Wav2Vec2_PR, ops
from aptai_b200.config import W2V2Config


def test_pr_vocab_above_1024_rejected_at_construction():
    """The wide recogniser head holds one row of logits in one warp's registers (32 per lane): 1024 classes at most.
    The limit is checked before the backbone is built, not left to the first kernel launch."""
    assert ops.PR_HEAD_MAX_VOCAB == 1024 and ops.PR_HEAD_NARROW == 48
    cfg = W2V2Config.base(num_hidden_layers=1, vocab_size=1025)
    with pytest.raises(ValueError, match="1024"):
        Wav2Vec2_PR(cfg, None, "mem://never-registered")


def test_pr_vocab_1024_passes_the_check():
    """At the limit construction proceeds to the backbone (which then fails on the unknown checkpoint id)."""
    cfg = W2V2Config.base(num_hidden_layers=1, vocab_size=1024)
    with pytest.raises(FileNotFoundError):
        Wav2Vec2_PR(cfg, None, "mem://never-registered")
