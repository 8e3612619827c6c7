"""The shared-memory layout of the default decimator's stage A (decim8_direct_kernel, csrc/sspsd_decim_kernel.cuh),
restated from the kernel's formulas: tile geometry for both tap presets, the run windows read with LDS.128 from the
contiguous staging buffer and the stores into stage B's polyphase planes.  Checks that every window is inside the
staging buffer and holds exactly the samples hbf_stage's definition of each output needs, that the stores cover the
planes once, and counts shared-memory wavefronts per warp instruction: 4 per LDS.128 (the minimum), and the stores'
count, which no phase stride can bring to 1 for lane-consecutive runs."""
import pytest

DEC_P, DEC_NT, OB, DIR_P = 8, 256, 960, 18
PRESETS = {"hbf140": (5, 10, 23), "hbf98": (3, 6, 15)}


def roundup(v, m):
    return (v + m - 1) // m * m


def geometry(ma, mb, mc):
    g = {}
    g["NB"] = roundup(2 * OB + 4 * mc - 2, DEC_P)
    g["NA"] = roundup(2 * g["NB"] + 4 * mb - 2, DEC_P)
    g["NX"] = roundup(2 * g["NA"] + 4 * ma - 2, 8)
    g["SB"] = ((g["NB"] // 2 + DEC_P - 1) // DEC_P + 27) // 32 * 32 + 4
    g["NRUN"] = (g["NA"] + DIR_P - 1) // DIR_P
    g["D"] = g["NRUN"] * DIR_P - g["NA"]
    g["REL0"] = g["NX"] // 2 - g["NA"]
    g["F"] = 2 * (g["REL0"] - 2 * ma + 1 - g["D"]) + 1
    g["XB"] = g["F"] // 4 * 4  # floor
    g["NXS"] = g["NX"] - g["XB"]
    g["NW"] = 2 * ma + DIR_P - 1
    g["W0"] = g["F"] - g["XB"]
    g["C0"] = 2 * (g["REL0"] - ma + 1 - g["D"]) - g["XB"]
    g["WCH"] = (g["W0"] + 2 * (g["NW"] - 1)) // 4 + 1
    g["SA"] = (g["NA"] // 2 // DEC_P + 1 - 3 + 31) // 32 * 32 + 3
    g["SMEM"] = 4 * (2 * g["NXS"] + 2 * DEC_P * (g["SA"] + g["SB"])) + 16
    return g


def lds128_wavefronts(chunks):
    """one warp-wide LDS.128: chunks[lane] = 16-byte chunk index (None: inactive lane); served a quarter warp at a
    time, each quarter needing as many wavefronts as the most distinct chunks in one 4-bank group"""
    n = 0
    for q in range(4):
        groups = {}
        for c in chunks[8 * q:8 * q + 8]:
            if c is not None:
                groups.setdefault(c % 8, set()).add(c)
        n += max((len(v) for v in groups.values()), default=0)
    return n


def sts_wavefronts(words):
    banks = {}
    for a in words:
        if a is not None:
            banks.setdefault(a % 32, set()).add(a)
    return max((len(v) for v in banks.values()), default=0)


def store_word(g, w, q, sa=None):
    """plane ('e'/'o') and float offset in it of stage-A output q of run w, or None for the unstored ones"""
    j = DIR_P * w + q - g["D"]
    if j < 0:
        return None
    r = j >> 1
    return "eo"[j & 1], (r & 7) * (sa or g["SA"]) + (r >> 3)


@pytest.mark.parametrize("preset", PRESETS)
def test_geometry(preset):
    ma, mb, mc = PRESETS[preset]
    g = geometry(ma, mb, mc)
    assert g["NRUN"] <= DEC_NT and g["D"] % 2 == 0 and 0 <= g["D"] < DIR_P
    assert g["NXS"] % 4 == 0 and g["XB"] <= 0 and g["NXS"] - g["NX"] < 32
    # the last run's window ends inside the staging buffer, and the whole buffer is read
    assert (DIR_P // 2) * (g["NRUN"] - 1) + g["WCH"] == g["NXS"] // 4
    assert g["WCH"] <= 14 and g["SA"] >= (g["NA"] // 2 + 7) // 8
    # two CTAs per SM: 228 KB of shared memory per SM, 1 KB of it reserved per CTA
    assert 2 * (g["SMEM"] + 1024) <= 228 * 1024, g["SMEM"]


@pytest.mark.parametrize("preset", PRESETS)
def test_windows_hold_what_each_output_reads(preset):
    """stage-A output j of the tile reads odd input x[2(j + REL0 - 2M + 1 + i) + 1], i < 2M, and even x[2(j + REL0 -
    M + 1)] (hbf_stage, relative to the tile's first sample x_base); in the kernel they are window samples W0 + 2(q + i)
    and C0 + 2q of run w, whose window starts at staging chunk 9 w, and staging sample s is x[XB + s]"""
    ma, _, _ = PRESETS[preset]
    g = geometry(*PRESETS[preset])
    for w in range(g["NRUN"]):
        base = 4 * (DIR_P // 2) * w
        for q in range(DIR_P):
            j = DIR_P * w + q - g["D"]
            for i in range(2 * ma):
                s = g["W0"] + 2 * (q + i)
                assert 0 <= s < 4 * g["WCH"]
                assert g["XB"] + base + s == 2 * (j + g["REL0"] - 2 * ma + 1 + i) + 1
            c = g["C0"] + 2 * q
            assert 0 <= c < 4 * g["WCH"]
            assert g["XB"] + base + c == 2 * (j + g["REL0"] - ma + 1)
            if j >= 0:  # a stored output only reads samples of the tile itself, x_base .. x_base + NX - 1
                assert 2 * (j + g["REL0"] - 2 * ma + 1) + 1 >= 0 and 2 * (j + g["REL0"]) + 1 < g["NX"]


@pytest.mark.parametrize("preset", PRESETS)
def test_window_loads_are_conflict_free(preset):
    g = geometry(*PRESETS[preset])
    for warp in range(DEC_NT // 32):
        runs = [32 * warp + l if 32 * warp + l < g["NRUN"] else None for l in range(32)]
        active = sum(r is not None for r in runs)
        for k in range(g["WCH"]):
            wf = lds128_wavefronts([None if r is None else (DIR_P // 2) * r + k for r in runs])
            assert wf == (active + 7) // 8  # one wavefront per quarter warp: 4 for a full warp


@pytest.mark.parametrize("preset", PRESETS)
def test_stores_cover_stage_b_planes(preset):
    g = geometry(*PRESETS[preset])
    seen = {"e": set(), "o": set()}
    for w in range(g["NRUN"]):
        for q in range(DIR_P):
            s = store_word(g, w, q)
            if s is not None:
                assert s[1] not in seen[s[0]]
                seen[s[0]].add(s[1])
    for p in "eo":
        assert seen[p] == {(r & 7) * g["SA"] + (r >> 3) for r in range(g["NA"] // 2)}


def store_wavefronts(g, sa):
    total = worst = 0
    for warp in range((g["NRUN"] + 31) // 32):
        for q in range(DIR_P):
            words = []
            for l in range(32):
                w = 32 * warp + l
                s = store_word(g, w, q, sa) if w < g["NRUN"] else None
                words.append(None if s is None else s[1])
            n = sts_wavefronts(words)
            total += n
            worst = max(worst, n)
    return total, worst


@pytest.mark.parametrize("preset", PRESETS)
def test_store_wavefronts(preset):
    """runs w, w+8, w+16, w+24 of a warp write one phase at offsets 9 apart, and the phases' offsets differ by one
    where (w + c) wraps past 8, so for every stride some store instruction is 2-way: the kernel's stride (3 mod 32)
    has the fewest of them"""
    g = geometry(*PRESETS[preset])
    total, worst = store_wavefronts(g, g["SA"])
    assert worst == 2
    instrs = ((g["NRUN"] + 31) // 32) * DIR_P
    assert total <= 1.8 * instrs, (total, instrs)
    for s in range(32):
        sa = g["SA"] - 3 + s
        t, wst = store_wavefronts(g, sa)
        assert wst >= 2 and t >= total
