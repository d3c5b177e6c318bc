"""The two-frames-per-warp synthesis kernel with the register-resident DCT-IV (synth_pair_kernel, dct_iv_pair).

At nf = 480 (48 and 44.1 kHz, 10 ms) synth mode 0 runs synth_pair_kernel for every launch of at least
2 x SMs x 5 CTAs x 8 frames rows (80 x SMs; 11 840 on a 148-SM B200): two frames per warp, one per half warp, with the
FFT's stages in registers.  Synth mode 1 runs synth_classic_kernel at every size: one frame per warp, with the
shared-memory Stockham stages of dct_iv_warp.  Both compute every butterfly with the same inputs, twiddles and
instruction sequence, so their PCM must be identical bit for bit.  Every case below is sized above that threshold, from
the device's SM count, and test_cases_reach_the_pair_kernel shows with the profiler that mode 0 launches
synth_pair_kernel there and mode 1 synth_classic_kernel.  The cases aim at what the pairing can get wrong:
- odd row counts: the last warp has one frame, and its second half warp has no frame to transform;
- a good and a concealed frame in one warp;
- subset calls, the IDS instantiation, whose rows map to streams in random order;
- split calls: sub-batches of the pair kernel whose last one has an odd row count;
- streams whose post filter is active (x_hat goes to ltpf_kernel), and the min_nbytes promise that keeps no history.
"""
import numpy as np
import pytest

from common import corpus, gpu_decode

pytestmark = pytest.mark.gpu

GEOMETRIES = [(48000, 150), (44100, 130)]       # every (fs, 10 ms) whose synthesis kernel pairs frames: nf = 480


def _pair_min_rows():
    """The smallest launch that runs synth_pair_kernel (plan_synth: 2 x SMs x SYN_PAIR_CTAS x SYN_WARPS x 2)."""
    import torch
    return 2 * torch.cuda.get_device_properties(0).multi_processor_count * 5 * 4 * 2


def _split4_rows(t):
    """An odd row count whose four sub-batches (lc3b_decode_frames: part = ceil(n / 4) rounded up to 128 rows) are all at
    least t rows, the last one odd."""
    n = 4 * t + 1
    while True:
        part = ((n + 3) // 4 + 127) & ~127
        last = n - 3 * part
        if last >= t and last % 2 == 1:
            return n, part, last
        n += 2


def _tiled(fs, nb, S, F, seed, lossy=True):
    """S streams x F frames tiled from a small oracle-encoded corpus, with lost (length 0) and garbage frames mixed in."""
    _, base = corpus(fs, 10, nb, 64, F)
    frames = np.tile(base, ((S + base.shape[0] - 1) // base.shape[0], 1, 1))[:S].copy()
    lens = np.full((S, F), nb, np.int32)
    if lossy:
        rng = np.random.default_rng(seed)
        lens[rng.random((S, F)) < 0.15] = 0
        bad = rng.random((S, F)) < 0.1
        frames[bad] = rng.integers(0, 256, (int(bad.sum()), nb), dtype=np.uint8)
    return frames, lens


def _both_modes(fs, frames, lens, trace=False, **kw):
    """Decode with the default kernel choice (pairs above the threshold) and with one frame per warp forced."""
    a = gpu_decode(fs, 10, frames, lens, trace=trace, synth_mode=0, **kw)
    b = gpu_decode(fs, 10, frames, lens, trace=trace, synth_mode=1, **kw)
    return a, b


def _decoder(fs, S, nb, synth_mode, split=None, graph=None):
    import torch

    import lc3_codec_b200 as L
    sf, fd = L.SamplingFrequency.from_hz(fs), L.FrameDuration.from_ms(10)
    ws = torch.empty(L.Lc3BatchDecoder.calc_working_buffer_lengths(S, fd, sf, nb), dtype=torch.uint8, device="cuda:0")
    dec = L.Lc3BatchDecoder(S, fd, sf, ws, nb)
    dec.set_synth_mode(synth_mode)
    if split is not None:
        dec.set_split(split)
    if graph is not None:
        dec.set_graph_mode(graph)
    return dec


def _subset_call(dec, ids, frames, lens):
    import torch
    n = len(ids)
    out = torch.full((n, 480), 12345, dtype=torch.int16, device="cuda:0")
    st = torch.full((n,), 7, dtype=torch.int32, device="cuda:0")
    dec.decode_frames_subset(16, ids, torch.from_numpy(np.ascontiguousarray(frames)).cuda(), out,
                             torch.from_numpy(np.ascontiguousarray(lens)).cuda(), status_out=st)
    return out.cpu().numpy(), st.cpu().numpy()


@pytest.mark.parametrize("fs,nb", GEOMETRIES)
@pytest.mark.parametrize("extra", [1, 449])
def test_odd_row_counts_equal_single_frame_kernel(fs, nb, extra):
    """T + 1 and T + 449 rows (T = the pair threshold): the last warp has one frame."""
    S = _pair_min_rows() + extra
    frames, lens = _tiled(fs, nb, S, 4, seed=extra)
    a, b = _both_modes(fs, frames, lens)
    assert np.array_equal(a[0], b[0]), (fs, S)
    assert np.array_equal(a[4], b[4])
    assert (a[4] == 1).any() and (a[4] == 0).any()             # concealed and decoded frames side by side


@pytest.mark.parametrize("fs,nb", GEOMETRIES)
def test_good_and_concealed_frame_in_one_warp(fs, nb):
    """Rows alternate good / lost and good / garbage, so every warp holds one decoded and one concealed frame; the last
    row (odd count) is lost in some frames."""
    S, F = _pair_min_rows() + 3, 6
    frames, lens = _tiled(fs, nb, S, F, seed=0, lossy=False)
    lens[1::4, 2:] = 0
    frames[3::4, 2:] = np.random.default_rng(5).integers(0, 256, (len(range(3, S, 4)), F - 2, nb), dtype=np.uint8)
    lens[::2, 4] = 0                                            # and a frame where the first row of each pair is lost
    lens[-1, 1::2] = 0
    a, b = _both_modes(fs, frames, lens)
    assert np.array_equal(a[0], b[0])
    assert (a[4][1::4, 2:] == 1).all()


def test_split_calls_with_an_odd_last_sub_batch():
    n, part, last = _split4_rows(_pair_min_rows())
    frames, lens = _tiled(48000, 150, n, 3, seed=7)
    a, b = _both_modes(48000, frames, lens, split=4)
    assert np.array_equal(a[0], b[0]), (n, part, last)
    assert np.array_equal(a[4], b[4])
    c = gpu_decode(48000, 10, frames, lens, trace=False, synth_mode=0, split=1)
    assert np.array_equal(a[0], c[0])                          # and the same as one launch over all rows


@pytest.mark.parametrize("fs,nb", GEOMETRIES)
def test_subset_calls_with_ids_in_random_order(fs, nb):
    t = _pair_min_rows()
    S = t + 501
    P = 5
    frames, lens = _tiled(fs, nb, S, P, seed=3)
    rng = np.random.default_rng(9)
    decs = [_decoder(fs, S, nb, m) for m in (0, 1)]
    for p, n in enumerate([t + 1, S, t + 37, t + 1, S]):        # odd row counts at or above the threshold
        ids = rng.permutation(S)[:n].astype(np.int32)
        got = [_subset_call(dec, ids, frames[ids, p], lens[ids, p]) for dec in decs]
        assert np.array_equal(got[0][0], got[1][0]), f"call {p}, {n} rows"
        assert np.array_equal(got[0][1], got[1][1])


def test_full_size_batch():
    """262 144 streams at 48 kHz / 150 B, the benchmark's batch (four sub-batches by default), with lost and garbage
    frames."""
    frames, lens = _tiled(48000, 150, 262144, 3, seed=11)
    a, b = _both_modes(48000, frames, lens)
    assert np.array_equal(a[0], b[0])
    assert np.array_equal(a[4], b[4])


@pytest.mark.parametrize("nb,promise", [(60, 0), (150, 150)])
def test_post_filter_streams_and_the_min_nbytes_promise(nb, promise):
    """60 B frames and no promise, so the post filter really filters (the synthesis kernel hands x_hat to ltpf_kernel);
    150 B frames under min_nbytes = 150, where the synthesis kernel keeps no post-filter history."""
    S = _pair_min_rows() + 1
    frames, lens = _tiled(48000, nb, S, 8, seed=nb)
    a, b = _both_modes(48000, frames, lens, trace=promise == 0, min_nbytes=promise)
    assert np.array_equal(a[0], b[0]), (nb, promise)
    assert np.array_equal(a[4], b[4])
    if promise == 0:
        assert a[1][..., 18].mean() > 0.1                      # LTPF-active frames (trace word 18, as assert_parity reads it)


def _synth_kernels(fn):
    """Names of the synthesis kernels fn() launches (torch.profiler sees every kernel of the process)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = [e.key for e in prof.key_averages()]
    forms = {"synth_pair_kernel<480, true, false>": "17synth_pair_kernelILi480ELb1ELb0E",   # demangled / mangled
             "synth_pair_kernel<480, true, true>": "17synth_pair_kernelILi480ELb1ELb1E",
             "synth_classic_kernel": "20synth_classic_kernel"}
    return {k for k, m in forms.items() if any(k in nm or m in nm for nm in names)}


def test_cases_reach_the_pair_kernel():
    """The sizes above launch synth_pair_kernel (full calls, split calls and subset calls), one row fewer does not, and
    synth mode 1 launches synth_classic_kernel at the same sizes: the reference really is the other kernel."""
    import torch
    t = _pair_min_rows()
    n_split, _, _ = _split4_rows(t)
    for S, split, mode, want in ((t + 1, None, 0, "synth_pair_kernel<480, true, false>"), (n_split, 4, 0, "synth_pair_kernel<480, true, false>"),
                                 (t - 1, None, 0, "synth_classic_kernel"), (t + 1, None, 1, "synth_classic_kernel")):
        frames, lens = _tiled(48000, 150, S, 1, seed=1)
        dec = _decoder(48000, S, 150, mode, split=split, graph=False)
        fr, ln = torch.from_numpy(frames[:, 0].copy()).cuda(), torch.from_numpy(lens[:, 0].copy()).cuda()
        out = torch.zeros((S, 480), dtype=torch.int16, device="cuda:0")
        assert _synth_kernels(lambda: dec.decode_frames(16, fr, out, ln)) == {want}, (S, split, mode)
    S = t + 501
    frames, lens = _tiled(48000, 150, S, 1, seed=2)
    dec = _decoder(48000, S, 150, 0, graph=False)
    ids = np.random.default_rng(4).permutation(S)[:t + 1].astype(np.int32)
    assert _synth_kernels(lambda: _subset_call(dec, ids, frames[ids, 0], lens[ids, 0])) == {"synth_pair_kernel<480, true, true>"}
