"""The peaky attention cases of tests/kernel_cases.py must reach the online-softmax branches they are written for.

A GPU case that silently stops reaching the O / l rescale would still pass, so this replays, in float64 on the
CPU, the per-row bookkeeping that every attention kernel in csrc/attention.cu does on those inputs: tiles of
64 keys (source 0, then source 1), the running max in log2 units, which moves only when a tile's max beats it by
more than 8 (the redo vote of attn2 / attn3, the alpha != 1 of all three).  Each pattern's claim is then checked,
with a margin from the threshold large enough that the kernels' fp32 logits cannot take the other branch."""
import math

import pytest
import torch

from tests import kernel_cases as K

MARGIN = 0.5  # log2 units between any tile's max growth and the lazy threshold


def _replay(batch, heads, d, nq, n0, n1, pattern, bank_batches):
    q, kv = K.attention_peaky_inputs(batch, heads, d, nq, n0, n1, pattern, bank_batches, device="cpu")
    amp, _, _ = K.peaky_profiles(pattern, batch, nq, n0, n1)
    scale_log2 = d ** -0.5 * math.log2(math.e)
    rows = []
    for b in range(batch):
        kk, _ = K.attention_keys(b, **kv)
        qq = q[b * nq:(b + 1) * nq].double().reshape(nq, heads, d).transpose(0, 1)
        lg = (qq @ kk.double().reshape(-1, heads, d).permute(1, 2, 0)) * scale_log2  # [heads, nq, keys], log2 units
        t0 = -(-n0 // K.ATT_BKV)
        tiles = [(j * K.ATT_BKV, min((j + 1) * K.ATT_BKV, n0)) for j in range(t0)]
        tiles += [(n0 + j * K.ATT_BKV, n0 + min((j + 1) * K.ATT_BKV, n1)) for j in range(-(-n1 // K.ATT_BKV))
                  if n1 and b < bank_batches]
        m_run = torch.full(lg.shape[:2], -math.inf, dtype=torch.float64)
        vote, margin, tmax, pos_arg = [], [], [], []
        for j, (k0, k1) in enumerate(tiles):
            mt = lg[..., k0:k1].amax(-1)
            tmax.append(mt)
            if j == 0:
                m_new = mt
            else:
                grow = mt - m_run
                vote.append(grow > K.ATT_LAZY_LOG2)
                margin.append((grow - K.ATT_LAZY_LOG2).abs().min())
                m_new = torch.where(vote[-1], mt, m_run)
            full = k1 - k0 == K.ATT_BKV
            pos_arg.append((lg[..., k0:k1] - m_new[..., None]).amax(-1) if full else torch.full_like(mt, -math.inf))
            m_run = m_new
        rows.append(dict(
            lg=lg, tiles=tiles, t0=t0, peaky=amp[b].bool(),
            vote=torch.stack(vote, -1) if vote else torch.zeros(*lg.shape[:2], 0, dtype=torch.bool),  # tiles j > 0
            margin=min(margin) if margin else math.inf, tmax=torch.stack(tmax, -1), pos_arg=torch.stack(pos_arg, -1),
            q=qq, kv=kv))
    return rows


def _shapes():
    return [(d,) + s for d in (40, 80, 160) for s in K.PEAKY_SHAPES]


@pytest.mark.parametrize("d,pattern,n0,n1,bb", _shapes(), ids=[f"d{s[0]}-{s[1]}-n0_{s[2]}" for s in _shapes()])
def test_peaky_case_reaches_its_branch(d, pattern, n0, n1, bb):
    batch, heads, nq = 2, 2, 256
    bank_batches = batch if bb is None else bb
    reps = _replay(batch, heads, d, nq, n0, n1, pattern, bank_batches)
    for b, r in enumerate(reps):
        lg, vote, pk = r["lg"], r["vote"], r["peaky"]
        n_tiles = len(r["tiles"])
        assert r["margin"] >= MARGIN, f"batch {b}: a tile's growth is {r['margin']:.3f} from the threshold"
        assert float(lg.abs().max()) <= 150 * math.log2(math.e), "logits beyond 150 natural units"
        rescales = vote.sum(-1)  # [heads, nq]: tiles j > 0 with alpha != 1
        if pattern == "rise":
            assert n_tiles >= 8 and bool((rescales[:, pk] == n_tiles - 1).all())
        elif pattern == "slow_rise":
            assert bool((rescales[:, pk] == (n_tiles - 1) // 2).all()) and (n_tiles - 1) // 2 >= 3
            # lazily accepted tiles: P up to 2^(>4) from the exponentials of a full tile
            assert bool((r["pos_arg"][:, pk].amax(-1) > 4).all())
        elif pattern == "mixed_rows":
            assert bool((rescales[:, pk] == n_tiles - 1).all()) and bool((rescales[:, ~pk] == 0).all())
            warps = vote.reshape(heads, nq // 32, 32, -1)
            lanes_disagree = warps.any(2) & ~warps.all(2)  # [heads, warp, tile]
            assert bool(lanes_disagree.any()), "no warp whose lanes disagree on the vote"
            cta = warps.any(2).reshape(heads, nq // 128, 4, -1)
            assert bool((cta.any(2) & ~cta.all(2)).any()), "no CTA whose warps disagree on the vote"
        elif pattern == "fall":
            tm = r["tmax"][:, pk]
            assert int(rescales.sum()) == 0 and bool((tm.argmax(-1) == 0).all())
            assert bool((tm[..., 1:] <= tm[..., :1] - 30).all())
            assert float((tm[..., -1] - tm[..., 0]).max()) < -126  # past ex2_poly's clamp and ex2.approx's ftz
        elif pattern == "bank_peak":
            if b < bank_batches:
                t0 = r["t0"]
                assert n_tiles > t0 and bool(vote[:, pk, t0 - 1].all())  # vote index t0 - 1 == tile t0
                assert bool((r["tmax"][:, pk].argmax(-1) >= t0).all())
            else:
                assert n_tiles == r["t0"] and int(rescales.sum()) == 0
        elif pattern == "ragged_peak":
            if b == 0:
                k0, k1 = r["tiles"][-1]
                assert k1 - k0 < K.ATT_BKV
                assert bool((r["tmax"][:, pk].argmax(-1) == n_tiles - 1).all()) and bool(vote[:, pk, -1].all())
                # the keys the last tile reads past n0 (the next batch element's) beat every valid logit
                spill = r["kv"]["k0"][n0:n0 + K.ATT_BKV - n0 % K.ATT_BKV].double()
                ls = (r["q"] @ spill.reshape(-1, heads, d).permute(1, 2, 0)) * d ** -0.5 * math.log2(math.e)
                assert float((ls.amax(-1) - lg.amax(-1))[:, pk].min()) > 20
        else:
            raise AssertionError(pattern)


def test_every_attention_kernel_gets_the_rescale_patterns():
    """attn_tc (d=160), attn3 (d=40, 80 on small grids), attn2 (d=40, 80 under ATT2Q) each run every pattern"""
    seen = set()
    for fn, args in K.ALL_CASES:
        tune = None
        if fn is K.case_tuned:
            tune, fn, args = args[0], args[1], args[2:]
        if fn is K.case_attention_peaky:
            seen.add((tune, args[2], args[6]))
    for tune, d in K.PEAKY_KERNELS:
        for pat in K.PEAKY_PATTERNS:
            assert (tune, d, pat) in seen, (tune, d, pat)
