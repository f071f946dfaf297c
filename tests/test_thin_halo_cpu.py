"""Planner side of the compact thin halo (engine.thin_items / setup_halo / setup_halo_s2, CisConv.thin), checked on launch plans built
on CPU tensors (nothing is launched)."""
import pytest

from unsupervised_detection_b200 import engine
from unsupervised_detection_b200.step_graph import CISGraph


def _convs(plan):
    return [a[0]._obj for fn, a, name, fl, lane in plan.ops if name == 'cis_conv_igemm']


def _cover(items, rel, m_chunks):
    """Every tap exactly once, every K half reads the pixel the kernel's descriptor points it at."""
    seen = []
    for a, b, h0, h1 in items:
        for h, (t, c0) in enumerate((h0, h1)):
            if t < 0:
                continue
            if m_chunks == 1:
                assert c0 == 0 and rel[t] == (a, b + h)           # second K half = next pixel
            else:
                assert c0 == 8 * h and rel[t] == (a, b)           # second K half = next 8-channel plane
            seen.append((t, c0))
    assert sorted(seen) == sorted((t, c) for t in range(len(rel)) for c in ((0,) if m_chunks == 1 else (0, 8)))


@pytest.mark.parametrize('k', [1, 2, 3, 4, 5, 7])
def test_thin_items_pair_x_adjacent_taps(k):
    rel = [(r, c) for r in range(k) for c in range(k)]
    items = engine.thin_items(rel, 1)
    _cover(items, rel, 1)
    assert len(items) == k * (-(-k // 2))                         # 5x5: 15 MMAs, 3x3: 6, 7x7: 28
    assert all(b + 1 <= max(k - 1, 1) for _, b, _, _ in items)    # only a one-column kernel needs a wider halo
    items16 = engine.thin_items(rel, 2)
    _cover(items16, rel, 2)
    assert len(items16) == k * k


def test_thin_items_pair_descending_parity_taps():
    # data-gradient / transposed-conv parity sub-problems list their taps in descending order: they still pair
    rel = [(1, 1), (1, 0), (0, 1), (0, 0)]
    items = engine.thin_items(rel, 1)
    _cover(items, rel, 1)
    assert len(items) == 2


def test_thin_items_parity_subsets():
    # stride-2 phases and the parity sub-problems of a stride-2 data gradient: ragged rows pair within their runs
    rel = [(0, 0), (0, 1), (0, 2), (1, 0), (1, 1), (1, 2), (2, 0)]
    items = engine.thin_items(rel, 1)
    _cover(items, rel, 1)
    assert len(items) == 5


@pytest.fixture(scope='module')
def graph():
    return CISGraph(64, 96, 1, device='cpu', global_batch=2)


def test_thin_launches_take_the_compact_halo(graph):
    """Every conv launch whose GEMM input has <= 16 channels runs on the compact thin halo (stride-2 layers included) unless its map is
    too small for the halo kernel's tile-utilisation rule; compact launches satisfy the launcher's rules."""
    nthin = ns2 = 0
    for plan in (graph.fwd, graph.bwd['G'], graph.bwd['R']):
        for d in _convs(plan):
            ch = sum(d.src[i].chunks for i in range(d.nsrc))
            if d.thin:
                assert d.halo and ch <= 2 and d.dil == 1 and d.splits <= 1 and d.sh == 1 and d.sw == 1
                hp = (8 + d.ex) * (16 * d.MT + d.ey)
                assert 2 * ((hp * 16 + 127) // 128 * 128) <= 227 * 1024
                for t in range(d.ntaps):
                    assert 0 <= d.dh[t] <= d.ey and 0 <= d.dw[t] + (1 if ch == 1 else 0) <= d.ex   # second K half inside the halo
                if d.nph > 1:
                    assert d.ph_tap[0] == 0 and d.ph_tap[4] == d.ntaps
                    ns2 += 1
                nthin += 1
            elif ch <= 2:
                # left on the gather kernel: only maps too small to fill a fifth of their 16x8 tiles
                assert not d.halo and d.OH * d.OW < 0.2 * 128 * (-(-d.OH // 16)) * (-(-d.OW // 8)) * 2 or d.OH * d.OW <= 48
    assert nthin > 20 and ns2 >= 4


def test_thin_weight_tiles_are_packed_in_the_compact_layout(graph):
    """Compact launches get their weights from tiled-pack jobs with layout 1: 16 K positions (one K=16 MMA) per tile."""
    from unsupervised_detection_b200._lib import CisParamJob, JOB_PACK_TILED
    import ctypes as C
    layouts = []
    for plan in (graph.pack_gen, graph.pack_rec):
        for fn, a, name, fl, lane in plan.ops:
            if name != 'cis_param_multi':
                continue
            tab = next(t for t in plan.keep if hasattr(t, 'data_ptr') and t.data_ptr() == a[0])
            raw = bytes(tab.cpu().numpy().tobytes())
            for q in range(a[1]):
                j = CisParamJob.from_buffer_copy(raw[q * C.sizeof(CisParamJob):(q + 1) * C.sizeof(CisParamJob)])
                if j.kind == JOB_PACK_TILED:
                    layouts.append(j.i[6])
                    assert j.i[6] in (0, 1) and (j.i[6] == 0 or j.i[0] == 16)
    assert 1 in layouts and 0 in layouts
