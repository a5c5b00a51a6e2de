"""Window bookkeeping of streaming.StreamSession (host logic, no GPU), and the streaming semantics on the CPU
oracle: provisional logits of frames below T - W plus close's result equal the reference's windowed inference."""
import pytest
import torch

from feature_vs_text_compound_emotion_b200 import streaming as S
from feature_vs_text_compound_emotion_b200 import synthetic, windowing
from oracle import lfan_oracle as O


def _simulate(T, c, W, H):
    """Push a T-frame stream c frames at a time (a partial last chunk) through the session's bookkeeping: for every
    frame, the windows its provisional logit averages; the windows close uses; every step table."""
    n_slots, n_lslots = S.n_window_slots(W, H, c), S.n_logit_slots(W, H, c)
    prov, tables, t, parity = {}, [], 0, 0
    lslot_owner = {}
    while t < T:
        cc = min(c, T - t)
        tab = S.step_table([(5, t, parity)], cc, W, H, n_slots, n_lslots)
        tables.append((t, cc, tab))
        act = tab[tab[:, 6] == 1]
        starts = [int(s) for s in act[:, 3]]
        assert starts == sorted(starts)
        assert len(set(act[:, 1].tolist())) == len(act)          # no two active windows share a TCN slot
        for s, ls in zip(starts, act[:, 2].tolist()):
            lslot_owner.setdefault(ls, [])
            if not lslot_owner[ls] or lslot_owner[ls][-1] != s:
                lslot_owner[ls].append(s)
        for f in range(t, t + cc):
            prov[f] = [s for s in starts if s <= f < s + W]
        t += cc
        parity ^= 1
    return prov, tables, lslot_owner, n_lslots


@pytest.mark.parametrize("W,H", [(300, 200), (100, 50)])
@pytest.mark.parametrize("c", [1, 7, 64, 200, 301])
def test_bookkeeping_agrees_with_window_starts(W, H, c):
    for T in range(1, 1301):
        prov, _, owner, n_lslots = _simulate(T, c, W, H)
        starts = windowing.window_starts(T, W, H)
        first, last = S.close_range(T, W)
        assert (first, last) == (T - min(T, W), T)
        assert S.final_upto(T, W) == max(0, T - W)
        assert first >= S.final_upto(T, W)
        # provisional windows below the close range are exactly the final ones
        for f in range(first):
            assert prov[f] == [s for s in starts if s <= f < s + W], (T, c, f)
        # close: the windows of window_starts(T) that reach the close range, in order, the tail recomputed
        cw = S.close_windows(T, W, H)
        assert [s for s, _ in cw] == [s for s in starts if s + min(W, T) > first and s < T]
        for s, rec in cw:
            grid = T >= W and s % H == 0 and s + W <= T
            assert rec == (not grid)
            if not rec:                 # a kept window's logit slot still holds it: no later window took the slot
                assert owner[(s // H) % n_lslots][-1] == s, (T, c, s)


def test_active_windows_and_slots_small_cases():
    assert S.active_windows(0, 1, 300, 200) == [0]
    assert S.active_windows(199, 2, 300, 200) == [0, 1]
    assert S.active_windows(300, 1, 300, 200) == [1]
    assert S.active_windows(250, 200, 300, 200) == [0, 1, 2]
    assert S.n_window_slots(300, 200, 30) == 2 == S.n_window_slots(300, 200, 101)
    assert S.n_window_slots(300, 200, 102) == 3
    assert S.n_logit_slots(300, 200, 30) == 3
    tab = S.step_table([(3, 390, 1), (7, 0, 0)], 20, 300, 200, 2, 3)
    assert tab.tolist() == [[3, 1, 1, 200, 390, 1, 1, 0], [3, 0, 2, 400, 390, 1, 1, 0],
                            [7, 0, 0, 0, 0, 0, 1, 0], [7, 0, 0, 0, 0, 0, 0, 0]]
    with pytest.raises(ValueError):
        S.step_table([(0, 250, 0)], 200, 300, 200, 2, 3)


def _oracle_stream(sd, feats, mods, T, c, W, H):
    """The session's procedure on the oracle: each active window's head over its prefix, averaged per frame as
    pushed; close recomputes the tail window from the last W inputs and stitches with the kept windows."""
    prov = torch.zeros(T, 7)
    kept = {}
    t = 0
    while t < T:
        cc = min(c, T - t)
        s_ = torch.zeros(cc, 7)
        cnt = torch.zeros(cc, 1)
        for k in S.active_windows(t, cc, W, H):
            s0 = k * H
            y = O.head_forward(sd, {m: v[s0:t + cc].unsqueeze(0) for m, v in feats.items()}, mods)[0]
            kept.setdefault(s0, torch.zeros(W, 7))
            lo = max(t, s0)
            hi = min(t + cc, s0 + W)
            kept[s0][lo - s0:hi - s0] = y[lo - s0:hi - s0]
            s_[lo - t:hi - t] += y[lo - s0:hi - s0]
            cnt[lo - t:hi - t] += 1
        prov[t:t + cc] = s_ / cnt
        t += cc
    first, _ = S.close_range(T, W)
    win = []
    for s0, rec in S.close_windows(T, W, H):
        if rec:
            x = {m: windowing.gather_windows(v[first:T], [0], W) for m, v in feats.items()}
            win.append(O.head_forward(sd, x, mods)[0])
        else:
            win.append(kept[s0])
    out = torch.zeros(W, 7)
    cnt = torch.zeros(W, 1)
    for (s0, _), y in zip(S.close_windows(T, W, H), win):
        rel = s0 - first
        lo, hi = max(0, rel), min(W, rel + W)
        out[lo:hi] += y[lo - rel:hi - rel]
        cnt[lo:hi] += 1
    return torch.cat([prov[:first], (out / cnt)[:T - first]])


@pytest.mark.parametrize("T", [150, 450, 701])
def test_streaming_semantics_on_the_oracle(T):
    mods = ["cnn_res50", "vggish"]
    ch = {"cnn_res50": [64, 64, 32, 32], "vggish": [32, 32, 32, 32]}
    sd = synthetic.head_state_dict(3, mods, tcn_channels=ch, encoder_dim={"cnn_res50": 32, "vggish": 32})
    g = torch.Generator().manual_seed(T)
    feats = {"cnn_res50": torch.nn.functional.normalize(torch.randn(T, 512, generator=g), dim=-1),
             "vggish": torch.randn(T, 128, generator=g)}
    got = _oracle_stream(sd, feats, mods, T, 64, 300, 200)
    X = {"video": feats["cnn_res50"].unsqueeze(0), "vggish": feats["vggish"].view(1, 1, T, 128)}
    want = O.windowed_inference(
        lambda ck: O.head_forward(sd, {"cnn_res50": ck["video"], "vggish": ck["vggish"].squeeze(1)}, mods), X)[0]
    assert got.shape == want.shape == (T, 7)
    torch.testing.assert_close(got, want, rtol=1e-5, atol=1e-5)
