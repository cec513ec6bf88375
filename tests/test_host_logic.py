"""CPU: host-side logic of the product (no GPU, no compute through the ABI)."""
import ctypes
import io
import os
import re

import numpy as np
import pytest

from inaspeechsegmenter_b200 import _lib, export_funcs, models
from inaspeechsegmenter_b200 import io as iss_io
from inaspeechsegmenter_b200.segmenter import _rle
from inaspeechsegmenter_b200.sidekit_mfcc import trfbank_htk24

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _csv_rows(path):
    rows = []
    with open(path) as f:
        next(f)
        for line in f:
            lab, a, b = line.rstrip('\n').split('\t')
            rows.append((lab, float(a), float(b)))
    return rows


def test_abi_exports_every_declared_symbol():
    """The C-ABI library loads and exports every function include/iss_b200.h declares."""
    hdr = open(os.path.join(ROOT, 'include', 'iss_b200.h')).read()
    hdr = re.sub(r'/\*.*?\*/', '', hdr, flags=re.S)
    declared = set(re.findall(r'\b(iss_[a-z0-9_]+)\s*\(', hdr))
    assert len(declared) >= 15
    lib = ctypes.CDLL(_lib.lib_path()) if os.path.exists(_lib.lib_path()) else _lib.load()
    for name in sorted(declared):
        assert hasattr(lib, name), 'libiss_b200.so does not export %s' % name
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    assert _lib.load().iss_version() == _lib.ABI_VERSION
    assert _lib.load().iss_sidekit_num_frames(1192367) == 7450      # musanmix.wav (SURVEY section 4)
    assert _lib.load().iss_sidekit_num_frames(399) == 0


def test_layer_desc_abi_layout():
    assert ctypes.sizeof(_lib.LayerDesc) == 12 * 4 + 6 * 8


def test_filterbank_table_matches_reference(golden):
    assert np.array_equal(trfbank_htk24(), golden['fbank'])


def test_csv_export_bytes(media, tmp_path):
    for name in ('musanmix-smn-gender.csv', 'musanmix-sm-gender.csv', '0021-smn-gender.csv', 'silence2sec-smn-gender.csv'):
        ref = os.path.join(media, name)
        rows = _csv_rows(ref)
        out = tmp_path / name
        export_funcs.seg2csv(rows, str(out))
        assert out.read_bytes() == open(ref, 'rb').read()
    # the doubles the reference prints come from start_sec + idx * .02 (segmenter.py:276)
    assert export_funcs.seg2csv([('noEnergy', 0 + 1124 * .02, 0 + 1454 * .02)]).split('\n')[1] == 'noEnergy\t22.48\t29.080000000000002'


def test_csv_export_matches_pandas():
    pd = pytest.importorskip('pandas')
    lseg = [('music', 0 + i * .02, 0 + (i + 7) * .02) for i in range(0, 4000, 7)] + [('male', 0, 0.66)]
    df = pd.DataFrame.from_records(lseg, columns=['labels', 'start', 'stop'])
    assert df.to_csv(None, sep='\t', index=False) == export_funcs.seg2csv(lseg)


def test_textgrid_export_bytes(media, tmp_path):
    rows = _csv_rows(os.path.join(media, 'musanmix-smn-gender.csv'))
    out = tmp_path / 'x.TextGrid'
    export_funcs.seg2textgrid(rows, str(out))
    assert out.read_bytes() == open(os.path.join(media, 'musanmix-smn-gender.TextGrid'), 'rb').read()


def test_rle():
    assert _rle(np.array([5] * 5 + [7] * 10 + [1] * 5)) == [(5, 0, 5), (7, 5, 15), (1, 15, 20)]
    assert _rle(np.array([3])) == [(3, 0, 1)]


def test_wav_reader(media):
    s16 = iss_io.media2sig16kmono(os.path.join(media, 'musanmix.wav'), ffmpeg=None, dtype='float32')
    assert s16.dtype == np.float32 and len(s16) == 1192367
    raw = iss_io.media2sig16kmono(os.path.join(media, 'musanmix.wav'), ffmpeg=None, dtype='float32', return_int16=True)
    assert raw.dtype == np.int16 and np.array_equal(raw.astype(np.float32) / np.float32(32768), s16)
    f32 = iss_io.media2sig16kmono(os.path.join(media, 'lamartine.wav'), ffmpeg=None, dtype='float64')
    assert f32.dtype == np.float64 and len(f32) == 234282
    with pytest.raises(NotImplementedError):
        iss_io.media2sig16kmono('x.wav', start_sec=1, ffmpeg=None)
    with pytest.raises(NotImplementedError):
        iss_io.media2sig16kmono('http://x/y.wav', ffmpeg=None)


def test_lowering_fuses_bn_relu(synth_models):
    cfg, w = synth_models['smn']
    low = models.lower_keras_model(cfg, w, 68, 21)
    kinds = [d['kind'] for d in low.descs]
    assert kinds == [1, 1, 3, 1, 1, 3, 2, 2, 2]
    conv = low.descs[0]
    assert conv['flags'] == _lib.F_BIAS | _lib.F_AFFINE_PRE | _lib.F_RELU and (conv['kh'], conv['kw'], conv['cout']) == (4, 5, 64)
    assert low.descs[-1]['flags'] & _lib.F_SOFTMAX and low.n_classes == 3
    assert all(d['w_off'] % 4 == 0 for d in low.descs if d['kind'] != 3)
    nparam = sum(v.size for k, v in w.items())
    assert 1.0e6 < nparam < 2.0e6


def test_lowering_rejects_unknown_layer(synth_models):
    cfg, w = synth_models['sm']
    bad = {'class_name': 'Sequential', 'config': {'layers': cfg['config']['layers'] + [{'class_name': 'LSTM', 'config': {'name': 'l'}}]}}
    with pytest.raises(NotImplementedError):
        models.lower_keras_model(bad, w, 68, 21)


def test_npz_roundtrip(tmp_path, synth_models):
    cfg, w = synth_models['gender']
    p = str(tmp_path / 'm.npz')
    models.save_npz(p, cfg, w)
    cfg2, w2 = models.load_npz(p)
    assert cfg2 == cfg and set(w2) == set(w) and all(np.array_equal(w[k], w2[k]) for k in w)


def test_product_never_imports_oracle():
    """Only tests/, __graft_entry__.smoke() and bench.py's CPU legs may touch oracle/."""
    for sub in ('inaspeechsegmenter_b200', 'scripts', 'tools'):
        for dirpath, _, files in os.walk(os.path.join(ROOT, sub)):
            for f in files:
                if f.endswith(('.py', '.cu', '.cuh')):
                    src = open(os.path.join(dirpath, f)).read()
                    assert 'import oracle' not in src and 'from oracle' not in src, f


def test_segmenter_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip('GPU present')
    from inaspeechsegmenter_b200 import Segmenter
    with pytest.raises(_lib.IssError):
        Segmenter(ffmpeg=None, models={})


def test_hdf5_reader_on_reference_fixture(media):
    """The pure-Python reader parses the reference's genuine h5py-written media/test.h5
    (the fixture of run_test.py:189-195) and finds both datasets at the offsets SURVEY section 4 lists."""
    from inaspeechsegmenter_b200 import keras_hdf5 as kh
    path = os.path.join(media, 'test.h5')
    f = kh.H5File(path)
    mel, emb = f.read_dataset(f.get('lamartinemelbands')), f.read_dataset(f.get('lamartineonnx'))
    raw = open(path, 'rb').read()
    assert mel.shape == (144, 64) and emb.shape == (256,) and mel.dtype == np.float32
    assert np.array_equal(mel, np.frombuffer(raw[2048:2048 + 144 * 64 * 4], '<f4').reshape(144, 64))
    assert np.array_equal(emb, np.frombuffer(raw[40960:40960 + 1024], '<f4'))


def test_keras_hdf5_roundtrip_and_model_lookup(tmp_path, synth_models, monkeypatch):
    from inaspeechsegmenter_b200 import keras_hdf5 as kh
    cfg, w = synth_models['gender']
    p = tmp_path / 'keras_male_female_cnn.hdf5'
    kh.write_keras_hdf5(str(p), cfg, w)
    cfg2, w2 = kh.load_keras_hdf5(str(p))
    assert cfg2 == cfg and set(w2) == set(w) and all(np.array_equal(w[k], w2[k]) for k in w)
    monkeypatch.setenv(models.MODEL_DIR_ENV, str(tmp_path))
    assert models.find_model_file('keras_male_female_cnn.hdf5') == str(p)
    cfg3, w3 = models.load_model_file(models.find_model_file('keras_male_female_cnn.hdf5'))
    low = models.lower_keras_model(cfg3, w3, 68, 24)
    assert low.n_classes == 2 and len(low.descs) == 9
    assert models.find_model_file('keras_speech_music_cnn.hdf5') is None


def test_cli_parser_matches_reference_flags():
    from inaspeechsegmenter_b200 import cli
    a = cli.build_parser().parse_args(['-i', 'x.wav', '-o', '/tmp', '-d', 'sm', '-g', 'false', '-b', 'None', '-e', 'textgrid', '-r', '0.05', '-s', '1024'])
    assert (a.vad_engine, a.detect_gender, a.ffmpeg_binary, a.export_format, a.energy_ratio, a.batch_size) == ('sm', 'false', 'None', 'textgrid', 0.05, 1024)


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the CPU port of the reference path) prints ONE JSON line with the contract keys."""
    import json
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '1',
                          '--cpu-chunk-sec', '6'], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = [l for l in out.stdout.splitlines() if l.startswith('{')][-1]
    d = json.loads(line)
    for k in ('impl', 'metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
              'vs_baseline', 'dtype', 'data', 'config', 'cpu_baseline', 'e2e'):
        assert k in d, k
    assert d['impl'] == 'reference' and d['value'] > 0 and d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['cores'] >= 1
    assert d['e2e']['h2d_bytes_per_step'] == 0 and d['e2e']['value'] == d['value']


def test_bench_dump_outputs_and_argument_checks(tmp_path):
    """`bench.py --dump-outputs DIR` stores the segment list losslessly as float64 (label code, start, stop) rows;
    a run without timed steps, or a dump from the CPU arm, is refused before anything runs."""
    import subprocess
    import sys
    import bench
    segs = [('noEnergy', 0.0, 1.98), ('female', 1.98, 3.5), ('music', 3.5, 29.080000000000002), ('noise', 29.080000000000002, 30.0)]
    bench.dump_outputs(str(tmp_path / 'out'), segs)
    got = np.load(tmp_path / 'out' / 'segments.npy')
    assert got.dtype == np.float64 and got.shape == (4, 3)
    assert [(bench.SEGMENT_LABELS[int(c)], a, b) for c, a, b in got] == segs
    for extra in (['--steps', '0'], ['--impl', 'reference', '--dump-outputs', str(tmp_path / 'ref')]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + extra, stdout=subprocess.PIPE,
                             stderr=subprocess.PIPE, text=True, timeout=120)
        assert out.returncode == 2 and 'usage:' in out.stderr, extra
    assert not (tmp_path / 'ref').exists()


def test_ffmpeg_branch_with_stand_in_binary(media, tmp_path):
    """The ffmpeg subprocess branch of media2sig16kmono (reference io.py:60-79): no ffmpeg exists in any of the
    boxes, so a stand-in executable checks the argv the reference builds (-i <media> -f wav -acodec pcm_s16le
    -ar 16000 -ac 1 [-ss a] [-to b] pipe:1), cuts the 16 kHz WAV like ffmpeg would and pipes it with the
    0xFFFFFFFF chunk sizes ffmpeg writes on a pipe; a failing binary must surface its stderr as the exception."""
    import stat
    import sys
    fake = tmp_path / 'ffmpeg'
    fake.write_text('''#!%s
import struct, sys
a = sys.argv[1:]
assert a[0] == '-i' and a[2:10] == ['-f', 'wav', '-acodec', 'pcm_s16le', '-ar', '16000', '-ac', '1'] and a[-1] == 'pipe:1', a
if a[1].endswith('broken.wav'):
    sys.stderr.write('broken.wav: Invalid data found when processing input')
    sys.exit(1)
rest = a[10:-1]
ss = float(rest[rest.index('-ss') + 1]) if '-ss' in rest else 0.0
to = float(rest[rest.index('-to') + 1]) if '-to' in rest else None
raw = open(a[1], 'rb').read()
p = raw.index(b'data') + 8
pcm = raw[p:]
pcm = pcm[2 * int(round(ss * 16000)):(2 * int(round(to * 16000)) if to is not None else None)]
hdr = b'RIFF' + struct.pack('<I', 0xFFFFFFFF) + b'WAVEfmt ' + struct.pack('<IHHIIHH', 16, 1, 1, 16000, 32000, 2, 16)
sys.stdout.buffer.write(hdr + b'data' + struct.pack('<I', 0xFFFFFFFF) + pcm)
''' % sys.executable)
    fake.chmod(fake.stat().st_mode | stat.S_IXUSR)
    wav = os.path.join(media, 'musanmix.wav')
    direct = iss_io.media2sig16kmono(wav, ffmpeg=None, dtype='float32')
    piped = iss_io.media2sig16kmono(wav, ffmpeg=str(fake), dtype='float32')
    assert piped.dtype == np.float32 and np.array_equal(piped, direct)
    cut = iss_io.media2sig16kmono(wav, start_sec=1.5, stop_sec=4.25, ffmpeg=str(fake), dtype='float64')
    assert cut.dtype == np.float64 and np.array_equal(cut, direct[24000:68000].astype(np.float64))
    raw16 = iss_io.media2sig16kmono(wav, stop_sec=2.0, ffmpeg=str(fake), return_int16=True)
    assert raw16.dtype == np.int16 and len(raw16) == 32000
    with pytest.raises(Exception, match='Invalid data found'):
        iss_io.media2sig16kmono(str(tmp_path / 'broken.wav'), ffmpeg=str(fake))


def test_kernel_source_stamp_ignores_comments_only():
    """bench.py quotes roofline.traffic from a committed ncu summary only when the summary's stamp equals the hash of the
    kernel's CODE: comments and white space must not change the stamp, code must."""
    import bench
    a = 'int f(int x) { return x + 1; }  // adds one\n/* block\n   comment */ const char *s = "a // b /* c */";\n'
    b = 'int f(int x)\n{\n    return x + 1;\n}\nconst char *s = "a // b /* c */";   // moved\n'
    c = 'int f(int x) { return x + 2; }\nconst char *s = "a // b /* c */";\n'
    assert bench._strip_cxx_comments(a) == bench._strip_cxx_comments(b) != bench._strip_cxx_comments(c)
    assert '"a//b/*c*/"' in bench._strip_cxx_comments(a)                  # comment markers inside a literal are not comments
    assert 'addsone' not in bench._strip_cxx_comments(a) and 'moved' not in bench._strip_cxx_comments(b)
    assert len(bench.kernel_source_hash()) == 64
