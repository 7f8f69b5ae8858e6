"""Bag-of-words vectors from the frame pipeline: a frame handle (or a sequence) with a vocabulary computes, for every frame, what
Frame::ComputeBoW (reference src/Frame.cc:1692-1699) computes, transform(mDescriptors, mBowVec, mFeatVec, levelsup), on the device right
after the descriptors.

  CPU: the binding mirrors the header's hvo_frame_bow_outputs; the drop-in hvo_shim::fill (shim/ORBVocabularyGPU.h) builds from fabricated
       rows the maps FrameFrontEnd.bow() returns, and hvo_shim::VocabularyArrays reads a vocabulary object's tree
  GPU: frame f's BoW rows == oracle.bow_transform on desc[f, :kp_counts[f]] (doubles compared by their bytes) == ORBVocabulary.transform_batch
       (hvo_bow_transform, pinned to the executed DBoW2 in test_bow.py), through every call path; every other output is byte-identical to a
       handle without a vocabulary."""
import ctypes as C
import os
import re
import struct
import subprocess

import numpy as np
import pytest

import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, 'a-low-texture-robust-hybrid-feature-based-visual-odometry_b200')
BOW_KEYS = ('bow_counts', 'bow_words', 'bow_values', 'fv_order', 'fv_counts', 'node_of', 'word_of')


def _fixture_vocabulary():
    """K = 10, L = 4, built by DBoW2's own create() (tests/golden/bow_ref.npz)."""
    g = np.load(os.path.join(ROOT, 'tests', 'golden', 'bow_ref.npz'))
    voc = {k[4:]: g[k] for k in g.files if k.startswith('voc_')}
    voc['L'] = int(voc['L'])
    return voc


def _random_vocabulary(seed, kmin, kmax, levels, p_inner=0.8, p_stopped=0.15):
    """A tree of uneven depth (a node above the last level has children with probability p_inner, the root always), kmin..kmax children
    per inner node, random node descriptors, leaf weights with a share of stopped words (weight 0)."""
    rng = np.random.default_rng(seed)
    children, depth = [[]], [0]
    frontier = [0]
    while frontier:
        nxt = []
        for i in frontier:
            if depth[i] < levels and (i == 0 or rng.random() < p_inner):
                for _ in range(int(rng.integers(kmin, kmax + 1))):
                    children[i].append(len(children))
                    children.append([]); depth.append(depth[i] + 1)
                    nxt.append(children[i][-1])
        frontier = nxt
    n = len(children)
    leaf = np.array([not c for c in children])
    leaf[0] = False
    word = np.full(n, -1, np.int32)
    word[leaf] = np.arange(int(leaf.sum()), dtype=np.int32)
    weight = np.where(leaf, rng.uniform(0.1, 5.0, n), 0.0)
    weight[leaf & (rng.random(n) < p_stopped)] = 0.0
    desc = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    desc[0] = 0
    return dict(child_start=np.concatenate([[0], np.cumsum([len(c) for c in children])]).astype(np.int32),
                child_ids=np.array([j for c in children for j in c], np.int32), node_desc=desc, node_weight=weight, node_word=word,
                L=int(max(depth)))


def _same_bow(got, want):
    (gw, gv), gfv = got
    (ww, wv), wfv = want
    assert np.array_equal(gw, ww)
    assert np.asarray(gv, np.float64).tobytes() == np.asarray(wv, np.float64).tobytes()
    assert gfv == wfv


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_bow_outputs_binding_mirrors_the_header(hvo):
    src = open(os.path.join(ROOT, 'include', 'hvo_capi.h')).read()
    body = re.search(r'typedef struct hvo_frame_bow_outputs \{(.*?)\} hvo_frame_bow_outputs;', src, re.S).group(1)
    body = re.sub(r'/\*.*?\*/', '', body, flags=re.S)
    names = re.findall(r'\*\s*(\w+)\s*;', body)
    assert names == [f[0] for f in hvo._FrameBowOutputs._fields_] == hvo.FrameFrontEnd.BOW_FIELDS == list(BOW_KEYS)
    for name in ('hvo_frame_set_vocabulary', 'hvo_frame_extract_batch_bow', 'hvo_frame_extract_batch_async_bow', 'hvo_frame_extract_batch_device_bow',
                 'hvo_seq_set_vocabulary', 'hvo_seq_extract_bow'):
        assert name in hvo.ABI
    assert hvo.FrameFrontEnd.FIELDS[-1] == 'kps_un' and len(hvo.FrameFrontEnd.FIELDS) == 17   # the frame outputs struct is unchanged


def _fabricated_rows(cap=40, seed=5):
    """BoW rows of four frames as a frame call lays them out: an empty frame, one with stopped words (features missing from fv_order),
    one with several features per node, and a full one."""
    rng = np.random.default_rng(seed)
    nf = 4
    out = dict(bow_counts=np.zeros(nf, np.int32), fv_counts=np.zeros(nf, np.int32), bow_words=np.full((nf, cap), -7, np.int32),
               bow_values=np.full((nf, cap), np.nan), fv_order=np.full((nf, cap), -7, np.int32), node_of=np.full((nf, cap), -7, np.int32))
    for f, (n, nodes, stopped) in enumerate(((0, 1, 0.0), (12, 6, 0.4), (30, 3, 0.0), (cap, 25, 0.1))):
        node = rng.integers(0, nodes, n).astype(np.int32) * 1000 + 17
        word = rng.integers(0, 10 * n + 1, n).astype(np.int32)
        word[rng.random(n) < stopped] = -1
        keep = np.nonzero(word >= 0)[0]
        order = keep[np.lexsort((keep, node[keep]))].astype(np.int32)
        words = np.unique(word[keep])
        values = rng.random(len(words))
        values /= values.sum()
        out['bow_counts'][f], out['fv_counts'][f] = len(words), len(order)
        out['bow_words'][f, :len(words)], out['bow_values'][f, :len(words)] = words, values
        out['fv_order'][f, :len(order)], out['node_of'][f, :n] = order, node
    return out


def _parse_fill(raw, nf):
    pos, res = 0, []
    for _ in range(nf):
        (nw,) = struct.unpack_from('<i', raw, pos); pos += 4
        words, values = [], []
        for _ in range(nw):
            w, v = struct.unpack_from('<Id', raw, pos); pos += 12
            words.append(w); values.append(v)
        (nn,) = struct.unpack_from('<i', raw, pos); pos += 4
        fv = {}
        for _ in range(nn):
            node, k = struct.unpack_from('<Ii', raw, pos); pos += 8
            fv[node] = list(struct.unpack_from(f'<{k}I', raw, pos)); pos += 4 * k
        res.append(((np.array(words, np.int32), np.array(values, np.float64)), fv))
    return res, pos


def test_shim_fill_equals_frame_front_end_bow(hvo, tmp_path):
    exe = str(tmp_path / 'shim_bow_fill')
    subprocess.check_call(['g++', '-O2', '-std=c++14', '-Wall', '-I' + os.path.join(ROOT, 'oracle', 'cvshim'), '-I' + os.path.join(ROOT, 'tests', 'cpp', 'standins'),
                           '-I' + os.path.join(PKG, 'shim'), '-I' + os.path.join(ROOT, 'include'), os.path.join(ROOT, 'tests', 'cpp', 'shim_bow_fill_main.cpp'),
                           '-o', exe])
    out = _fabricated_rows()
    nf, cap = out['bow_words'].shape
    fi, fo = str(tmp_path / 'in.bin'), str(tmp_path / 'out.bin')
    with open(fi, 'wb') as f:
        f.write(struct.pack('<3i', 0x46424f57, nf, cap) + np.stack([out['bow_counts'], out['fv_counts']], 1).astype(np.int32).tobytes()
                + out['bow_words'].tobytes() + out['bow_values'].tobytes() + out['fv_order'].tobytes() + out['node_of'].tobytes())
    subprocess.check_call([exe, fi, fo])
    raw = open(fo, 'rb').read()
    got, pos = _parse_fill(raw, nf)
    for f in range(nf):
        _same_bow(got[f], hvo.FrameFrontEnd.bow(out, f))
    assert got[0][1] == {} and len(got[0][0][0]) == 0                                             # empty frame: both maps cleared
    assert out['fv_counts'][1] < 12 and max(len(v) for v in got[2][1].values()) > 3               # stopped words; several features per node
    # VocabularyArrays on the driver's fixed tree: root -> {1, 2}, 1 -> {3, 4, 5}, leaves 2..5 = words 0..3, node 4 stopped
    n, L = struct.unpack_from('<2i', raw, pos); pos += 8
    cs = np.frombuffer(raw, np.int32, n + 1, pos); pos += 4 * (n + 1)
    (nc,) = struct.unpack_from('<i', raw, pos); pos += 4
    ci = np.frombuffer(raw, np.int32, nc, pos); pos += 4 * nc
    word = np.frombuffer(raw, np.int32, n, pos); pos += 4 * n
    weight = np.frombuffer(raw, np.float64, n, pos); pos += 8 * n
    desc = np.frombuffer(raw, np.uint8, 32 * n, pos).reshape(n, 32); pos += 32 * n
    assert pos == len(raw) and (n, L) == (6, 2)
    assert cs.tolist() == [0, 2, 5, 5, 5, 5, 5] and ci.tolist() == [1, 2, 3, 4, 5]
    assert word.tolist() == [-1, -1, 0, 1, 2, 3] and weight.tolist() == [0.0, 0.25, 0.5, 0.75, 0.0, 1.25]
    assert not desc[0].any() and desc[3].tolist() == [(21 + b) & 255 for b in range(32)]


# ---------------------------------------------------------------------------------------------------------------- GPU
def _cam(synth):
    c = synth.CONFIGS['S1']
    return c['fx'], c['fy'], c['cx'], c['cy'], 1.0 / c['factor']


def _frames(synth):
    """S1 frames, S2 (low-texture) frames and a constant image (no keypoints)."""
    g1, d1 = synth.sequence('S1', 2, start=31)
    g2, d2 = synth.sequence('S2', 2, start=9)
    return np.concatenate([g1, g2, np.full_like(g1[:1], 128)]), np.concatenate([d1, d2, d1[:1]])


def _fe(hvo, synth, **kw):
    return hvo.FrameFrontEnd(640, 480, *_cam(synth), bf=40.0, **kw)


def _check_parity(hvo, voc, out, levelsup, nframes, transformer=None):
    """Frame f's BoW rows == oracle.bow_transform on its descriptor rows (and == hvo_bow_transform when `transformer` is given)."""
    descs = [out['desc'][f, :int(out['kp_counts'][f])] for f in range(nframes)]
    bt = transformer.transform_batch(descs, levelsup) if transformer is not None else None
    for f, d in enumerate(descs):
        n = len(d)
        o = oracle.bow_transform(voc, d, levelsup)
        got = hvo.FrameFrontEnd.bow(out, f)
        _same_bow(got, o[:2])
        assert np.array_equal(out['word_of'][f, :n], o[2]) and np.array_equal(out['node_of'][f, :n], o[3])
        assert int(out['fv_counts'][f]) == int((o[2] >= 0).sum())
        if bt is not None:
            _same_bow(got, bt[f][:2])
            assert np.array_equal(out['word_of'][f, :n], bt[f][2]) and np.array_equal(out['node_of'][f, :n], bt[f][3])


def _check_same_as_plain(d, p, nframes):
    """Every output of a handle without a vocabulary, byte for byte, in the rows a frame owns."""
    for f in range(nframes):
        n, nl, npl = int(p['kp_counts'][f]), int(p['line_counts'][f]), int(p['n_planes'][f])
        assert (n, nl, npl) == (int(d['kp_counts'][f]), int(d['line_counts'][f]), int(d['n_planes'][f]))
        for k in ('kps', 'desc', 'kp_depth', 'kp_uright', 'kps_un'):
            if k in p:
                assert d[k][f, :n].tobytes() == p[k][f, :n].tobytes(), k
        for k in ('keylines', 'line_desc', 'linevec3'):
            assert d[k][f, :nl].tobytes() == p[k][f, :nl].tobytes(), k
        assert d['planes7'][f, :npl].tobytes() == p['planes7'][f, :npl].tobytes()
        for k in ('membership', 'membership8', 'membership4', 'normals8', 'normals3'):
            if k in p:
                assert d[k][f].tobytes() == p[k][f].tobytes(), k


@pytest.mark.gpu
def test_gpu_frame_bow_equals_oracle_and_hvo_bow_transform(hvo, synth):
    voc = _fixture_vocabulary()
    gray, depth = _frames(synth)
    nf = len(gray)
    plain = _fe(hvo, synth, max_batch=nf)
    p = plain.extract_batch(gray, depth)
    launches = plain.last_launches()
    plain.close()
    assert int(p['kp_counts'][-1]) == 0 and min(p['kp_counts'][:-1]) > 100
    bt = hvo.ORBVocabulary(voc)
    fe = _fe(hvo, synth, max_batch=nf, vocabulary=voc, levelsup=2)
    for lu in (2, 4, voc['L'], voc['L'] + 2):
        fe.set_vocabulary(voc, lu)                         # re-attaching replaces the vocabulary
        assert fe.output_shapes(nf)['bow_values'] == ((nf, fe.orb_capacity), np.float64)
        d = fe.extract_batch(gray, depth)
        assert fe.last_launches() == launches + 2
        _check_same_as_plain(d, p, nf)
        _check_parity(hvo, voc, d, lu, nf, bt)
        assert int(d['bow_counts'][-1]) == 0 and int(d['fv_counts'][-1]) == 0
        if lu >= voc['L']:                                 # the FeatureVector's node is the root
            for f in range(nf):
                assert not d['node_of'][f, :int(d['kp_counts'][f])].any()
        else:
            assert len(hvo.FrameFrontEnd.bow(d, 0)[1]) > 5
    bt.close()
    # detaching restores the plain handle
    fe.set_vocabulary(None)
    assert not set(BOW_KEYS) & set(fe.output_shapes(nf))
    d = fe.extract_batch(gray, depth)
    assert fe.last_launches() == launches
    _check_same_as_plain(d, p, nf)
    fe.close()


@pytest.mark.gpu
def test_gpu_frame_bow_through_every_call_path(hvo, synth):
    """Blocking, two queued wait=False calls, the device-resident call, several chunks through two lanes, two serial chunks of 2048 frames
    (device-resident), FrameSequence and the undistorting TUM1 handle: the same BoW rows as the blocking call."""
    import torch
    voc = _fixture_vocabulary()
    gray, depth = _frames(synth)
    nf = len(gray)
    ref = _fe(hvo, synth, max_batch=nf, lanes=1, vocabulary=voc)
    r = ref.extract_batch(gray, depth)
    ref.close()
    _check_parity(hvo, voc, r, 4, nf)

    def same(o, n, frames=None):
        for f in range(n):
            g = f if frames is None else frames[f]
            k = int(r['kp_counts'][g])
            assert k == int(o['kp_counts'][f]) and o['desc'][f, :k].tobytes() == r['desc'][g, :k].tobytes()
            _same_bow(hvo.FrameFrontEnd.bow(o, f), hvo.FrameFrontEnd.bow(r, g))
            assert o['word_of'][f, :k].tobytes() == r['word_of'][g, :k].tobytes() and o['node_of'][f, :k].tobytes() == r['node_of'][g, :k].tobytes()

    fe = _fe(hvo, synth, max_batch=4, lanes=2, vocabulary=voc)
    assert fe.chunk == 2
    same(fe.extract_batch(gray, depth), nf)               # three chunks through two lanes (side by side)
    outs = [fe.alloc_host(nf) for _ in range(2)]
    for o in outs:
        fe.extract_batch(gray, depth, out=o, wait=False)
    fe.sync()
    for o in outs:
        same(o, nf)
    bad = fe.alloc_host(nf)
    bad['fv_order'] = np.empty((nf, fe.orb_capacity - 1), np.int32)
    with pytest.raises(hvo.HvoError):
        fe.extract_batch(gray, depth, out=bad)
    # optional host arrays: without word_of / fv_order / fv_counts / node_of the rest is still written
    part = {k: v for k, v in fe.alloc_host(nf).items() if k not in ('word_of', 'fv_order', 'fv_counts', 'node_of')}
    ptrs = {k: v.ctypes.data for k, v in part.items()}
    hvo._check(hvo.lib().hvo_frame_extract_batch_bow(fe._h, hvo._np_ptr(gray), hvo._np_ptr(depth), nf, C.byref(fe._outputs(ptrs)), fe._bow_outputs(ptrs)))
    for f in range(nf):
        w = int(r['bow_counts'][f])
        assert int(part['bow_counts'][f]) == w and part['bow_values'][f, :w].tobytes() == r['bow_values'][f, :w].tobytes()
    # device-resident, on torch tensors
    dev = torch.device('cuda', 0)
    shapes = fe.output_shapes(4)
    d = {k: torch.empty(int(np.prod(s)) * np.dtype(dt).itemsize, dtype=torch.uint8, device=dev) for k, (s, dt) in shapes.items()}
    g, dp = torch.from_numpy(gray[:4].copy()).to(dev), torch.from_numpy(depth[:4].copy()).to(dev)
    torch.cuda.synchronize()
    fe.extract_batch_device(g.data_ptr(), dp.data_ptr(), 4, {k: v.data_ptr() for k, v in d.items()})
    fe.sync()
    same({k: d[k].cpu().numpy().view(dt).reshape(s) for k, (s, dt) in shapes.items()}, 4)
    fe.close()
    del d

    # 4096 frames device-resident through two lanes: two chunks of 2048, each running its pipelines one after the other
    big = _fe(hvo, synth, max_batch=4096, lanes=2, vocabulary=voc, membership='u8', normals='n8')
    assert big.chunk == 2048
    n = 4096
    pick = np.arange(n) % nf
    g = torch.from_numpy(gray).to(dev)[torch.from_numpy(pick).to(dev)].contiguous()
    dp = torch.from_numpy(depth.view(np.int16)).to(dev)[torch.from_numpy(pick).to(dev)].contiguous()   # (no uint16 indexing on the device)
    shapes = big.output_shapes(n)
    d = {k: torch.empty(int(np.prod(s)) * np.dtype(dt).itemsize, dtype=torch.uint8, device=dev) for k, (s, dt) in shapes.items()}
    torch.cuda.synchronize()
    big.extract_batch_device(g.data_ptr(), dp.data_ptr(), n, {k: v.data_ptr() for k, v in d.items()})
    big.sync()
    keys = ('kp_counts', 'desc') + BOW_KEYS
    same({k: d[k].cpu().numpy().view(shapes[k][1]).reshape(shapes[k][0]) for k in keys}, n, pick)
    big.close()
    del d, g, dp
    torch.cuda.empty_cache()

    # FrameSequence: two handles (the device list names cuda:0 twice), queued calls of two frames
    seq = hvo.FrameSequence(640, 480, *_cam(synth), [0, 0], frames_per_call=2, bf=40.0, vocabulary=voc)
    assert set(BOW_KEYS) <= set(seq.output_shapes(nf, device=False))
    same(seq.extract(gray, depth), nf)
    bad = seq.alloc_host(nf)
    bad['bow_values'] = np.empty((nf, seq.orb_capacity), np.float32)
    with pytest.raises(hvo.HvoError):
        seq.extract(gray, depth, out=bad)
    seq.close()

    # the undistorting TUM1 handle: the descriptors do not depend on the undistortion, neither does the BoW
    dist = np.array([0.262383, -0.953104, -0.005358, 0.002628, 1.163314], np.float32)
    tum = _fe(hvo, synth, max_batch=nf, vocabulary=voc, dist=dist)
    o = tum.extract_batch(gray, depth)
    assert 'kps_un' in o
    same(o, nf)
    tum.close()


@pytest.mark.gpu
@pytest.mark.parametrize('kmin,kmax,levels,levelsup', [(2, 8, 5, 2), (2, 40, 3, 1), (9, 16, 3, 5)])
def test_gpu_frame_bow_on_random_vocabularies(hvo, synth, kmin, kmax, levels, levelsup):
    """Uneven depth, 2..40 children (more than 32: the child scan loops), stopped words; the tile width follows the largest branching."""
    voc = _random_vocabulary(1000 + kmax, kmin, kmax, levels)
    assert (voc['node_weight'][voc['node_word'] >= 0] == 0).any()
    nch = np.diff(voc['child_start'])
    assert nch.max() > 32 if kmax > 32 else nch.max() <= kmax
    gray, depth = _frames(synth)
    fe = _fe(hvo, synth, max_batch=len(gray), stages=hvo.STAGE_ORB, vocabulary=voc, levelsup=levelsup)
    out = fe.extract_batch(gray, depth)
    fe.close()
    _check_parity(hvo, voc, out, levelsup, len(gray))


@pytest.mark.gpu
def test_gpu_frame_bow_argument_errors(hvo, synth):
    voc = _fixture_vocabulary()
    gray, depth = _frames(synth)
    gray, depth = gray[:1], depth[:1]
    lines = _fe(hvo, synth, stages=hvo.STAGE_LINES)
    with pytest.raises(hvo.HvoError) as e:
        lines.set_vocabulary(voc)
    assert e.value.status == hvo.HVO_ERR_ARG
    lines.close()
    wide = _fe(hvo, synth, stages=hvo.STAGE_ORB, nfeatures=5000)
    assert wide.orb_capacity > 4096
    with pytest.raises(hvo.HvoError) as e:
        wide.set_vocabulary(voc)
    assert e.value.status == hvo.HVO_ERR_ARG
    wide.close()

    fe = _fe(hvo, synth, stages=hvo.STAGE_ORB)
    out = fe.alloc_host(1)
    bow = {k: np.zeros((1, fe.orb_capacity), np.float64 if k == 'bow_values' else np.int32) for k in BOW_KEYS}
    ptrs = {k: v.ctypes.data for k, v in list(out.items()) + list(bow.items())}
    bo = hvo._FrameBowOutputs(*[ptrs[k] for k in BOW_KEYS])

    def call(b):
        return hvo.lib().hvo_frame_extract_batch_bow(fe._h, hvo._np_ptr(gray), hvo._np_ptr(depth), 1, C.byref(fe._outputs(ptrs)), C.byref(b))
    assert call(bo) == hvo.HVO_ERR_ARG                                    # no vocabulary attached
    fe.set_vocabulary(voc)
    assert call(bo) == hvo.HVO_OK
    no_node = hvo._FrameBowOutputs(*[None if k == 'node_of' else ptrs[k] for k in BOW_KEYS])
    assert call(no_node) == hvo.HVO_ERR_ARG                               # fv_order without node_of
    import torch
    dev = torch.device('cuda', 0)
    shapes = fe.output_shapes(1)
    d = {k: torch.empty(int(np.prod(s)) * np.dtype(dt).itemsize, dtype=torch.uint8, device=dev) for k, (s, dt) in shapes.items()}
    g, dp = torch.from_numpy(gray.copy()).to(dev), torch.from_numpy(depth.copy()).to(dev)
    dptr = {k: v.data_ptr() for k, v in d.items()}
    for missing in ('word_of', 'fv_counts'):                             # optional on the host, required on the device
        b = hvo._FrameBowOutputs(*[None if k == missing else dptr[k] for k in BOW_KEYS])
        st = hvo.lib().hvo_frame_extract_batch_device_bow(fe._h, g.data_ptr(), dp.data_ptr(), 1, C.byref(fe._outputs(dptr)), C.byref(b))
        assert st == hvo.HVO_ERR_ARG, missing
    fe.extract_batch_device(g.data_ptr(), dp.data_ptr(), 1, dptr)
    fe.sync()
    fe.close()
