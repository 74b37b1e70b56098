"""CPU checks of the wide top-k configuration (128 < k <= 1024): its workspace query needs no GPU."""
import pytest

# tmf_score_topk_ws_bytes for k <= 128, as the library returned it before the wide configuration existed
NARROW_WS = {(1, 1, 1): 2135296, (300, 5000, 32): 7667200, (138493, 26744, 64): 2297125888,
             (1000000, 1000000, 128): 4957100032}


@pytest.mark.parametrize("shape", sorted(NARROW_WS))
def test_workspace_unchanged_up_to_k128_and_larger_above(shape):
    from teamoflow_b200 import _abi
    n_u, n_i, r = shape
    for k in (1, 10, 100, 128):
        assert _abi.query("tmf_score_topk_ws_bytes", n_u, n_i, r, k) == NARROW_WS[shape]
    wide = [_abi.query("tmf_score_topk_ws_bytes", n_u, n_i, r, k) for k in (129, 500, 1024)]
    assert wide[0] > NARROW_WS[shape] and wide[0] == wide[1] == wide[2]


def test_wide_workspace_stays_bounded():
    # the candidate lists go through in batches of user blocks: the workspace stops growing with n_users
    from teamoflow_b200 import _abi
    a = _abi.query("tmf_score_topk_ws_bytes", 1_000_000, 1000, 64, 1024)
    b = _abi.query("tmf_score_topk_ws_bytes", 2_000_000, 1000, 64, 1024)
    assert a < 6 << 30 and b - a < 1 << 30  # unbatched, the lists alone would grow by 64 GB
