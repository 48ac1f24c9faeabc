"""GPU parity, stage by stage: every C-ABI entry point against the CPU oracle on the same
seeded input.  Tables come from the oracle so that only the kernels are under test here.

Tolerances (floating point; integer results are compared exactly):
  FFT           1e-6 relative to the spectrum maximum
  embed         RMS(out_gpu - out_oracle) < 1e-5         (north star)
  sync quality  |dq| < 2e-4 (quality is ~1 for a real sync, ~0.05 noise floor)
  refine index  within 8 samples (one sync_search_fine step; SURVEY H1), quality 1e-3
  soft bits     1e-3 relative to mean |soft bit|
  Viterbi       decoded bits identical, error metric 1e-5
"""
import numpy as np
import pytest
import scipy.fft

import awm_oracle as O
import awm_testlib as T
from audiowmark_b200 import capi

pytestmark = pytest.mark.gpu

P = O.Params()
KEY = O.Key()


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    T.setup_ctx(c, KEY, P, T.PAYLOAD)
    yield c
    c.close()


@pytest.fixture(scope="module")
def marked():
    """115 s stereo noise watermarked by the ORACLE (limiter on): contains one full A block."""
    x = T.noise(115.0)
    return x, O.embed(x, KEY, T.PAYLOAD, P).samples


# inputs of the *_signals variants of the sync / decode stage tests, 115 s each (one full A block).  White noise (`marked`) has a
# flat spectrum; these put the loudest in-band component far above the quietest (tone: -6 dBFS over a 1 LSB floor; music: tones
# over pink noise), make one channel of a stereo pair silent or 50 dB quieter than the other (the packed two-channel FFT extracts
# it from a sum dominated by the loud one), or leave the stereo paths (mono, 3 channels).  They are 16 bit signals, watermarked by
# the oracle and written back to 16 bit, as a file would be: the silent channel stays exactly zero.
SIGNALS = {
    "tone": lambda: T.tone(115.0),
    "music": lambda: T.music(115.0),
    "r_zero": lambda: T.one_sided(115.0, "zero"),
    "r_m50": lambda: T.one_sided(115.0, "m50"),
    "mono": lambda: T.music(115.0, 1, seed=6),
    "ch3": lambda: T.music(115.0, 3, seed=7),
}


@pytest.fixture(scope="module", params=list(SIGNALS))
def signal_marked(request):
    """(name, watermarked by the ORACLE with the limiter on, on the 16 bit grid)"""
    y = O.embed(SIGNALS[request.param](), KEY, T.PAYLOAD, P).samples
    return request.param, T.to16(y)


def test_fft_roundtrip_and_numpy(ctx):
    rng = np.random.default_rng(0)
    for count in (1, 2, 7, 64):
        x = rng.standard_normal((count, 1024)).astype(np.float32)
        X = ctx.fft_r2c(x)
        ref = np.fft.rfft(x.astype(np.float64), axis=1)
        assert np.abs(X - ref).max() < 1e-6 * np.abs(ref).max() * 4
        back = ctx.fft_c2r(X)
        assert np.abs(back / 1024 - x).max() < 2e-6 * np.abs(x).max() * 4
        # unnormalised c2r of an arbitrary Hermitian spectrum (FFTW semantics)
        S = (rng.standard_normal((count, 513)) + 1j * rng.standard_normal((count, 513))).astype(np.complex64)
        S[:, 0] = S[:, 0].real
        S[:, 512] = S[:, 512].real
        y = ctx.fft_c2r(S)
        yr = np.fft.irfft(S.astype(np.complex128), n=1024, axis=1) * 1024
        assert np.abs(y - yr).max() < 1e-6 * np.abs(yr).max() * 4


@pytest.mark.parametrize("limiter", [True, False])
@pytest.mark.parametrize("seconds,channels", [(12.0, 2), (3.3, 1), (2.0, 3), (0.01, 2)])
def test_embed_vs_oracle(ctx, limiter, seconds, channels):
    x = T.noise(seconds, channels, seed=7, amp=1.0 if limiter else 0.5)
    Pl = O.Params(test_no_limiter=not limiter)
    ref = O.embed(x, KEY, T.PAYLOAD, Pl, keep_wm=True)
    out, (dpow, spow) = ctx.embed(x, limiter_block=44100 if limiter else 0, want_snr=True)
    assert out.shape == x.shape
    d = T.rms(out - ref.samples)
    assert d < 1e-5, d
    assert np.abs(out - ref.samples).max() < 1e-4
    if ref.wm is not None and seconds > 1:
        assert T.rms(ref.wm) > 1e-4          # a watermark was actually added
        snr = 10 * np.log10(spow / dpow)
        assert abs(snr - ref.snr_db) < 1e-3


@pytest.mark.parametrize("seconds,limiter", [(20.0, True), (3.3, False), (0.01, True)])
def test_embed_strip_kernel_equals_tile_kernel(ctx, monkeypatch, seconds, limiter):
    """k_embed_strip (streaming, TMA-fed, neighbours' window tails carried in registers) and k_embed (CTA tiles with a halo frame on
    each side) run the same arithmetic in the same order: identical bits, identical limiter peaks, for whole and ragged lengths"""
    x = T.noise(seconds, 2, seed=21, amp=1.0 if limiter else 0.5)
    monkeypatch.setenv("AWM_EMBED", "tile")
    tile, tile_snr = ctx.embed(x, limiter_block=44100 if limiter else 0, want_snr=True)
    monkeypatch.delenv("AWM_EMBED")
    strip, strip_snr = ctx.embed(x, limiter_block=44100 if limiter else 0, want_snr=True)
    bad = np.nonzero((tile != strip).any(axis=1))[0]
    assert len(bad) == 0, (len(bad), bad[:8], float(np.abs(tile - strip).max()), tile[bad[:3]], strip[bad[:3]])
    assert np.allclose(tile_snr, strip_snr, rtol=1e-12)


def test_embed_device_pointers_match_host_path(ctx):
    torch = pytest.importorskip("torch")
    x = T.noise(5.0, 2, seed=3)
    host = ctx.embed(x)
    xin = torch.from_numpy(x).cuda()
    xout = torch.empty_like(xin)
    torch.cuda.synchronize()
    ctx.embed(xin.data_ptr(), xout.data_ptr(), n_frames=x.shape[0], channels=2)
    ctx.synchronize()
    assert np.array_equal(xout.cpu().numpy(), host)


def oracle_approx(y):
    """the oracle's search_approx on a whole input"""
    sf = O.SyncFinder(P)
    sf.first, sf.last = 0, y.size
    return sf.search_approx(O.get_sync_bits(KEY, O.BLOCK, P), y, O.BLOCK)


@pytest.fixture(scope="module")
def signal_approx(signal_marked):
    return oracle_approx(signal_marked[1])


def check_sync_approx(ctx, name, y, want):
    ctx.pcm_bind(y)
    got = ctx.sync_approx(0, capi.MODE_BLOCK)
    assert len(got) == len(want) > 0
    assert np.array_equal(got["index"], np.array([s.index for s in want], np.uint64))
    dq = np.abs(got["raw_quality"] - np.array([s.raw_quality for s in want]))
    dm = np.abs(got["local_mean"] - np.array([s.local_mean for s in want]))
    print("%s: sync_approx max |dq| %.3g, max |d local_mean| %.3g" % (name, dq.max(), dm.max()))
    assert dq.max() < 2e-4 and dm.max() < 2e-4, (dq.max(), dm.max())
    # the embedded blocks are found where the reference puts them: first A block at sample 256000, the B block one block later
    # (on some inputs the stronger of the two).  A silent channel adds -96 dB to both sides of every up / down ratio: the reference's
    # own qualities on R = 0 are ~0.45 (tests/golden/golden_large.json r_zero130)
    best = got[np.argmax(np.abs(got["raw_quality"] - got["local_mean"]))]
    if name == "noise":
        assert best["index"] == 256000 and best["raw_quality"] > 1.0
    else:
        assert best["index"] in (256000, 256000 + O.frames_per_block(P) * P.frame_size)
        assert abs(best["raw_quality"] - best["local_mean"]) > (0.4 if name == "r_zero" else 1.0)


def test_sync_approx_vs_oracle(ctx, marked):
    _, y = marked
    check_sync_approx(ctx, "noise", y, oracle_approx(y))


def test_sync_approx_vs_oracle_signals(ctx, signal_marked, signal_approx):
    name, y = signal_marked
    check_sync_approx(ctx, name, y, signal_approx)


def check_tensor_core_entry_sums(ctx, name, y, monkeypatch):
    """k_stft_mags_tc (tcgen05.mma on fp16 hi/lo terms of the dB values, fp32 accumulation in TMEM, masks by TMA) against k_stft_mags
    (the same sums on the fp32 pipes): the two differ only by the rounding of the additions -- far below the 2e-4 bar against the
    oracle that test_sync_approx_vs_oracle holds the default path to.  Both tile variants of the kernel are run; for stereo also with
    the frames fetched by global loads instead of bulk copies (AWM_TC_PCM=ldg, the path every other channel count takes)."""
    ctx.pcm_bind(y)
    monkeypatch.setenv("AWM_APPROX", "simt")
    simt = ctx.sync_approx(0, capi.MODE_BLOCK)
    monkeypatch.delenv("AWM_APPROX")
    for pcm in ("tma", "ldg") if y.shape[1] == 2 else ("ldg",):
        if pcm == "ldg":
            monkeypatch.setenv("AWM_TC_PCM", "ldg")
        for variant in ("8x2", "12x1"):
            monkeypatch.setenv("AWM_TC", variant)
            tc = ctx.sync_approx(0, capi.MODE_BLOCK)
            assert np.array_equal(tc["index"], simt["index"])
            d = np.abs(tc["raw_quality"] - simt["raw_quality"]).max()
            dm = np.abs(tc["local_mean"] - simt["local_mean"]).max()
            print("%s %s %s: tensor-core vs fp32 pipes max |dq| %.3g, max |d local_mean| %.3g" % (name, pcm, variant, d, dm))
            assert d < 2e-5, (variant, pcm, d)
            assert dm < 2e-5, (variant, pcm, dm)
    monkeypatch.delenv("AWM_TC")


def test_tensor_core_entry_sums_match_fp32_pipes(ctx, marked, monkeypatch):
    check_tensor_core_entry_sums(ctx, "noise", marked[1], monkeypatch)


def test_tensor_core_entry_sums_match_fp32_pipes_signals(ctx, signal_marked, monkeypatch):
    name, y = signal_marked
    check_tensor_core_entry_sums(ctx, name, y, monkeypatch)


FLOAT64_ARBITER = ("tone", "r_zero", "r_m50")          # inputs on which the refine scores are also held against float64


def refine_candidates(y, approx):
    """what search() hands search_refine, plus a candidate near the start (index < 256) and one whose window runs past the end"""
    sf = O.SyncFinder(P)
    sf.first, sf.last = 0, y.size
    sel = sf.select_threshold_and_n_best(sf.mask_avg_false_positives(sf.select_local_maxima(approx)), P.sync_threshold2 * 0.75)
    sel = sel + [O.SearchScore(128, 0.01, 0.0), O.SearchScore(approx[-1].index, approx[-1].raw_quality, approx[-1].local_mean)]
    inp = np.zeros(len(sel), capi.SEARCH_SCORE)
    inp["index"] = [s.index for s in sel]
    inp["raw_quality"] = [s.raw_quality for s in sel]
    inp["local_mean"] = [s.local_mean for s in sel]
    return sf, sel, inp


def check_sync_refine(ctx, name, y, approx):
    ctx.pcm_bind(y)
    sb = O.get_sync_bits(KEY, O.BLOCK, P)
    sf, sel, inp = refine_candidates(y, approx)
    S, vs = ctx.sync_refine_offsets(inp, exact=False)
    E, ve = ctx.sync_refine_offsets(inp, exact=True)
    if y.shape[1] <= 2:
        print("%s: max |S - E| %.3g over %d candidates" % (name, np.abs(S - E)[vs].max(), len(sel)))
    if name in FLOAT64_ARBITER:
        check_refine_vs_float64(name, y, sb, sf, sel, S, E, ve)
    want = sf.search_refine(y, O.BLOCK, sel, sb, KEY)
    got = np.sort(ctx.sync_refine(inp, 0, capi.MODE_BLOCK), order="index")
    assert len(got) == len(want)
    for g, w in zip(got, want):
        assert int(g["index"]) == w.index, (g, w)               # sync positions are exact, not "within one fine step"
        assert abs(g["raw_quality"] - w.raw_quality) < 2e-4
        assert g["local_mean"] == w.local_mean
    # error bound behind the exactness claim (awm_capi.cu: kVerifyMargin = 1e-3): the sliding-DFT ranking S and the exact scores E
    # of all 65 offsets differ by less than a quarter of the margin, so the exact arg-max is always among the re-scored offsets.
    # More than two channels take the exact kernel for the ranking as well (no sliding DFT): S is E there.
    assert np.array_equal(vs, ve) and vs.sum() > 60 * (len(sel) - 2)
    if y.shape[1] <= 2:
        assert np.abs(S - E)[vs].max() < 1e-3 / 4, np.abs(S - E)[vs].max()
    # the result is the exact kernel's: the reference rule (start from the approx index, replace on strictly larger |q - mean|,
    # offsets ascending) applied to E alone gives the indices awm_sync_refine returns
    unsorted = ctx.sync_refine(inp, 0, capi.MODE_BLOCK)
    for k, (i, m) in enumerate(zip(inp["index"], inp["local_mean"])):
        start = max(int(i) - 256, 0)
        o_self = (int(i) - start) // 8
        if not ve[k][o_self]:
            continue
        best_o, best_v = o_self, abs(E[k][o_self] - m)
        for o in range(65):
            if ve[k][o] and abs(E[k][o] - m) > best_v:
                best_o, best_v = o, abs(E[k][o] - m)
        assert int(unsorted[k]["index"]) == start + 8 * best_o, (k, int(unsorted[k]["index"]), start + 8 * best_o)
        assert abs(abs(unsorted[k]["raw_quality"] - m) - best_v) < 1e-12


def test_sync_refine_vs_oracle(ctx, marked):
    _, y = marked
    check_sync_refine(ctx, "noise", y, oracle_approx(y))


def test_sync_refine_vs_oracle_signals(ctx, signal_marked, signal_approx):
    """on the tone and one-sided inputs the scores are also held against float64 (check_refine_vs_float64)"""
    name, y = signal_marked
    check_sync_refine(ctx, name, y, signal_approx)


def q64_offsets(y, sb, start, n_off):
    """search_refine's per-offset sync quality in float64 throughout: rfft of the Hann-windowed sync frames, 10 log10 |X|^2
    (-96 for an exact zero, as db_from_complex does), dB summed over channels, sync_decode's formula in double.  nan where the
    block does not fit."""
    n = P.frame_size
    i = np.arange(n, dtype=np.float64)
    win = O.window_cos((i - n / 2) / (n / 2))
    win *= 2.0 / win.sum()
    total = O.frames_per_block(P)
    frames = np.unique(sb.frame)
    yy = y.astype(np.float64)
    up = sb.up.reshape(len(sb.frame), -1)
    down = sb.down.reshape(len(sb.frame), -1)
    q = np.full(n_off, np.nan)
    for o in range(n_off):
        pos = start + 8 * o
        if pos + total * n > len(y):
            continue
        seg = yy[pos + frames[:, None] * n + np.arange(n)]                        # [frames][n][ch]
        X = scipy.fft.rfft(seg * win[None, :, None], axis=1, workers=-1)[:, P.min_band:P.max_band + 1]
        a2 = X.real ** 2 + X.imag ** 2
        dbv = np.where(a2 > 0, 10 * np.log10(np.where(a2 > 0, a2, 1.0)), -96.0).sum(axis=2)
        dbe = dbv[np.searchsorted(frames, sb.frame)]                                # [entries][bands]
        umag = np.add.reduceat(np.take_along_axis(dbe, up, 1).sum(axis=1), sb.off[:-1])
        dmag = np.add.reduceat(np.take_along_axis(dbe, down, 1).sum(axis=1), sb.off[:-1])
        quality, count = 0.0, 0
        for bit in range(P.sync_bits):
            u, d = umag[bit], dmag[bit]
            raw = 0.0 if u == 0 or d == 0 else (1 - u / d if u < d else d / u - 1)
            n_e = int(sb.off[bit + 1] - sb.off[bit])
            quality += (raw if bit & 1 else -raw) * n_e
            count += n_e
        q[o] = quality / count / min(P.water_delta, 0.080) / 2.9
    return q


def check_refine_vs_float64(name, y, sb, sf, sel, S, E, ve):
    """float64 as the arbiter of the refine scores on the inputs with the widest in-band dynamic range (a -6 dBFS tone over a 1 LSB
    floor; a silent or -50 dB channel beside a loud one): per candidate, the GPU's exact re-score E of every offset is no further
    from the float64 quality Q64 than twice the reference's own float32 error (the oracle: same transforms, same order of additions
    as the reference) plus 1e-5.  Prints max |S - E| of the sliding-DFT ranking S and the errors, so that a disagreement between
    GPU and oracle shows which side is off."""
    want = np.zeros(O.frames_per_block(P), np.int8)
    bpg = O.BitPosGen(KEY, P)
    for f in range(O.mark_sync_frame_count(P)):
        want[bpg.sync_frame(f)] = 1
    worst = []
    for k, sc in enumerate(sel):
        start = max(int(sc.index) - 256, 0)
        n_off = (int(sc.index) + 256 - start) // 8 + 1
        q64 = q64_offsets(y, sb, start, n_off)
        orc = np.full(n_off, np.nan)
        for o in range(n_off):
            db, have = sf.sync_fft(y, start + 8 * o, O.frames_per_block(P), want)
            if db is not None:
                orc[o] = sf.sync_decode(sb, [0], db, have)[0]
        ok = ~np.isnan(q64)
        assert np.array_equal(ok, ve[k][:n_off]) and not ve[k][n_off:].any(), k
        if not ok.any():
            continue
        e_err = np.abs(E[k][:n_off] - q64)[ok].max()
        o_err = np.abs(orc - q64)[ok].max()
        worst.append((e_err, o_err, np.abs(S[k] - E[k])[ve[k]].max(), k, int(sc.index)))
    w = np.array(worst)
    print("%s: max |E - Q64| %.3g, max |oracle - Q64| %.3g, max |S - E| %.3g over %d candidates" % (name, *w[:, :3].max(axis=0), len(w)))
    for e_err, o_err, _, k, index in worst:
        assert e_err <= 2 * o_err + 1e-5, (k, index, e_err, o_err)


def raw_bits_float64(y, index):
    """raw_bits_for_block from the float64 spectrum (numpy rfft of the frames, float64 Hann window), rounded to float32 once: the
    soft bits without the rounding error of a float transform"""
    n, fpb = P.frame_size, O.frames_per_block(P)
    if index + fpb * n > len(y):
        return None
    i = np.arange(n, dtype=np.float64)
    win = O.window_cos((i - n / 2) / (n / 2))
    win *= 2.0 / win.sum()
    seg = y.astype(np.float64)[index + np.arange(fpb)[:, None] * n + np.arange(n)]          # [frames][n][ch]
    X = scipy.fft.rfft(seg * win[None, :, None], axis=1, workers=-1).transpose(0, 2, 1)     # [frames][ch][n/2+1]
    sp = np.empty((fpb * y.shape[1], n + 2), np.float32)
    sp[:, 0::2] = X.real.reshape(-1, n // 2 + 1)
    sp[:, 1::2] = X.imag.reshape(-1, n // 2 + 1)
    raw = O.mix_decode(KEY, sp, y.shape[1], P)
    return np.array(O.randomize_bit_order(KEY, list(raw), False), dtype=np.float32)


def check_decode_blocks(ctx, name, y):
    """soft bits within 1e-3 of their mean magnitude of the oracle's.  Where they are not, float64 decides: the GPU is no further
    from the soft bits of the float64 spectrum than twice the oracle is.  On the tone the oracle is the less accurate side (bins far
    below the tone carry the float transforms' rounding relative to it; measured on a B200 at the A block: |gpu - oracle| 0.98 at a
    mean of 428, |gpu - f64| 4.1, |oracle - f64| 4.5).  R at -50 dB is the exception: the packed two-channel FFT extracts R from a
    transform dominated by L, and its soft bits at sample 100 (no block there) are 1.02e-3 of the mean from the oracle's and ~100x further from float64 than the
    oracle's (0.118 vs 0.001 at a mean of 115); they are held to 2e-3 (DESIGN.md section 6).  Whole documents and sync positions
    on this input are identical to the reference's (test_gpu_large_golden.py)."""
    ctx.pcm_bind(y)
    n_coded = O.conv_code_size(O.A, P.payload_size)
    idx = [256000, 256008, 100, y.shape[0] - 100]
    raw, valid = ctx.decode_blocks(idx, n_coded)
    assert list(valid) == [1, 1, 1, 0]
    for i in range(3):
        want = O.raw_bits_for_block(KEY, y, idx[i], P)
        scale = np.abs(want).mean()
        err = np.abs(raw[i] - want).max()
        print("%s: block at %d: soft bits max |gpu - oracle| %.3g (%.3g of the mean)" % (name, idx[i], err, err / scale))
        if name == "r_m50":
            assert err < 2e-3 * scale, i
        elif name == "noise" or err < 1e-3 * scale:
            assert err < 1e-3 * scale, i
        else:
            r64 = raw_bits_float64(y, idx[i])
            e_gpu, e_orc = np.abs(raw[i] - r64).max(), np.abs(want - r64).max()
            print("    |gpu - f64| %.3g, |oracle - f64| %.3g" % (e_gpu, e_orc))
            assert e_gpu <= 2 * e_orc, (i, e_gpu, e_orc)
    # and the payload comes out
    bits, err = ctx.viterbi(raw[:1], [capi.BLOCK_A])
    assert O.bit_vec_to_str(list(bits[0])) == T.PAYLOAD


def test_decode_blocks_vs_oracle(ctx, marked):
    check_decode_blocks(ctx, "noise", marked[1])


def test_decode_blocks_vs_oracle_signals(ctx, signal_marked):
    name, y = signal_marked
    check_decode_blocks(ctx, name, y)


@pytest.mark.parametrize("variant", ["single", "pair"])
def test_viterbi_vs_oracle(ctx, monkeypatch, variant):
    """k_viterbi (one CTA per code word, the default) and k_viterbi_pair (a 2-CTA cluster per word, metrics exchanged through
    distributed shared memory; AWM_VITERBI=pair) against the oracle: identical bits, error within 1e-5"""
    monkeypatch.setenv("AWM_VITERBI", variant)
    rng = np.random.default_rng(5)
    msg = [int(b) for b in rng.integers(0, 2, 128)]
    for bt, cbt in ((O.A, capi.BLOCK_A), (O.B, capi.BLOCK_B), (O.AB, capi.BLOCK_AB)):
        coded = np.array(O.conv_encode(bt, msg), np.float32)
        jobs = []
        for noise in (0.0, 0.6, 1.5, 4.0):
            jobs.append(((coded * 2 - 1) + noise * rng.standard_normal(len(coded))).astype(np.float32))
        bits, err = ctx.viterbi(jobs, [cbt] * len(jobs))
        hbits, herr = ctx.viterbi(jobs, [cbt] * len(jobs), hard=True)
        for j in range(len(jobs)):
            wb, we = O.conv_decode_soft(bt, O.normalize_soft_bits(jobs[j], P))
            assert list(bits[j]) == wb, (bt, j)
            assert abs(err[j] - we) < 1e-5 * max(1.0, we)
            Ph = O.Params(hard=True)
            wb, we = O.conv_decode_soft(bt, O.normalize_soft_bits(jobs[j], Ph))
            assert list(hbits[j]) == wb
        assert list(bits[0]) == msg


def test_clip_mode_approx_with_silence(ctx):
    """CLIP tables + zero padding: frames in digital silence are skipped (have = 0) like sync_fft :583-588."""
    x = T.noise(20.0, 2, seed=11)
    y = O.embed(x, KEY, T.PAYLOAD, P).samples
    fpb = O.frames_per_block(P)
    npad = (fpb + 5) * 1024
    pad_start = npad + (npad - y.shape[0])
    ctx.pcm_bind(y, pad_start=pad_start, pad_end=npad)
    ext = np.concatenate([np.zeros((pad_start, 2), np.float32), y, np.zeros((npad, 2), np.float32)])
    flat = ext.reshape(-1)
    nz = np.nonzero(flat)[0]
    first, last = int(nz[0]), int(nz[-1]) + 1
    got = ctx.sync_approx(0, capi.MODE_CLIP, first, last)
    sf = O.SyncFinder(P)
    sf.first, sf.last = first, last
    want = sf.search_approx(O.get_sync_bits(KEY, O.CLIP, P), ext, O.CLIP)
    assert len(got) == len(want) > 0
    dq = np.abs(got["raw_quality"] - np.array([s.raw_quality for s in want]))
    assert dq.max() < 2e-4, dq.max()
