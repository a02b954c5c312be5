"""Host-side logic of the section-8f components that needs no GPU: state_dict layout of the speaker encoder, batch grouping
of the evaluation driver, and the torch criterion against the loss oracle."""
import json
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

from oracle import loss_oracle
from voicesplit_b200 import evaluate, losses, synth
from voicesplit_b200.speaker_encoder import SpeakerEncoder


def test_speaker_encoder_state_dict_layout():
    enc = SpeakerEncoder()
    want = {}
    for l in range(3):
        want[f"lstm.weight_ih_l{l}"] = (3072, 40 if l == 0 else 768)
        want[f"lstm.weight_hh_l{l}"] = (3072, 768)
        want[f"lstm.bias_ih_l{l}"] = (3072,)
        want[f"lstm.bias_hh_l{l}"] = (3072,)
    want["proj.linear_layer.weight"] = (256, 768)
    want["proj.linear_layer.bias"] = (256,)
    got = {k: tuple(v.shape) for k, v in enc.state_dict().items()}
    assert got == want
    # the synthetic weights used by the parity tests follow the same layout
    assert {k: tuple(v.shape) for k, v in synth.make_encoder_state_dict(0).items()} == want
    enc.load_state_dict({k: torch.from_numpy(v) for k, v in synth.make_encoder_state_dict(0).items()}, strict=True)


def test_speaker_encoder_loads_the_reference_checkpoint_unchanged():
    # key / shape / dtype of every tensor in the reference's GE2E checkpoint (notebooks/embedder.pt, 48 MB), recorded by
    # tests/golden/make_reference_checks_golden.py; a strict load checks exactly these
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_layouts.json")) as f:
        layout = json.load(f)["embedder_checkpoint"]
    ckpt = {k: torch.zeros(shape, dtype=getattr(torch, dtype)) for k, shape, dtype in layout}
    enc = SpeakerEncoder(40, 3, 768, 80, 40)                      # the notebook's positional arguments (:88)
    missing = enc.load_state_dict(ckpt, strict=True)
    assert not missing.missing_keys and not missing.unexpected_keys


def test_speaker_encoder_without_engine_fails_loudly():
    with pytest.raises(RuntimeError):
        SpeakerEncoder()(torch.zeros(40, 100))                    # CPU tensor: no silent fallback


def test_eval_batches_group_by_shape_and_keep_every_item():
    def item(T, L, tag):
        return [(tag, None, np.zeros((T, 5), np.float32), np.zeros(L, np.float32), None, None, None)]
    loader = [item(10, 100, 0), item(10, 100, 1), item(12, 100, 2), item(10, 100, 3), item(10, 90, 4), item(10, 100, 5), item(10, 100, 6)]
    batches = list(evaluate._batches(loader, 3))
    tags = sorted(it[0] for b in batches for it in b)
    assert tags == list(range(7))
    for b in batches:
        assert len(b) <= 3
        assert len({(it[2].shape, it[3].shape) for it in b}) == 1      # one spectrogram / waveform shape per batch
    assert [it[0] for it in batches[0]] == [0, 1, 3]                     # a full group is emitted as soon as it fills up


def test_torch_criterion_matches_loss_oracle_for_one_source():
    rng = np.random.Generator(np.random.PCG64(3))
    est, tgt = rng.standard_normal((4, 500)), rng.standard_normal((4, 500))
    est = 0.6 * tgt + 0.4 * est
    lens = torch.tensor([500, 321, 500, 77])
    a = losses.si_snr_with_pit(torch.from_numpy(est)[:, None], torch.from_numpy(tgt)[:, None], lens)
    b, _ = loss_oracle.si_snr_c1(torch.from_numpy(est), torch.from_numpy(tgt), lens)
    assert abs(float(a) - float(b)) < 1e-9


def test_sdr_workspace_is_a_pure_host_query():
    from voicesplit_b200 import _cabi
    lib = _cabi.load()
    a, b, c = (int(lib.vs_sdr_workspace_bytes(B, L)) for B, L in ((1, 48000), (8, 48000), (8, 96000)))
    assert 0 < a < b < c
    assert int(lib.vs_sdr_workspace_bytes(0, 48000)) == 0 and int(lib.vs_sdr_workspace_bytes(4, 0)) == 0


@pytest.mark.skipif(shutil.which("gcc") is None, reason="no C compiler")
def test_public_header_is_plain_c_and_cxx():
    hdr = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "voicesplit_b200.h")
    for args in (["gcc", "-std=c99", "-pedantic", "-Werror", "-fsyntax-only", "-x", "c"], ["g++", "-std=c++17", "-Werror", "-fsyntax-only", "-x", "c++"]):
        if shutil.which(args[0]) is None:
            continue
        r = subprocess.run(args + [hdr], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the driver's reference arm: the reference's CPU path, oracle/torch_port.py) prints ONE JSON line
    with the keys of the bench contract; run at a tiny shape so that it takes seconds."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--frames", "41", "--freq", "33"], capture_output=True, text=True, timeout=600, cwd=root)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "e2e", "cpu_baseline"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "utterances/s" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["value"] > 0 and d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and "sample" in d["cpu_baseline"]
    assert d["config"]["frames"] == 41 and d["config"]["freq_bins"] == 33


@pytest.mark.skipif(shutil.which("gcc") is None, reason="no C compiler")
def test_ctypes_structs_and_constants_match_the_public_header(tmp_path):
    """The Python binding (voicesplit_b200/_cabi.py) restates the header's structs and enum values by hand: a C probe compiled
    against include/voicesplit_b200.h prints sizeof / offsetof of every field and the VS_* constants, which must equal what
    ctypes lays out - a silent drift here would hand the library mis-aligned pointers."""
    import ctypes
    from voicesplit_b200 import _cabi
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    structs = {"vs_dims": _cabi.VsDims, "vs_params": _cabi.VsParams, "vs_train_state": _cabi.VsTrainState, "vs_grads": _cabi.VsGrads,
               "vs_audio_params": _cabi.VsAudioParams, "vs_loss_params": _cabi.VsLossParams, "vs_encoder_dims": _cabi.VsEncoderDims,
               "vs_encoder_params": _cabi.VsEncoderParams}
    consts = {"VS_OK": _cabi.VS_OK, "VS_ACT_MISH": _cabi.ACT_MISH, "VS_ACT_RELU": _cabi.ACT_RELU,
              "VS_ISTFT_Q1": 0, "VS_ISTFT_CORRECTED": 1,
              **{"VS_PREC_" + k.upper(): v for k, v in _cabi.PRECISIONS.items()}}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "voicesplit_b200.h"', 'int main(void) {']
    for cname, cls in structs.items():
        lines.append(f'  printf("{cname} %zu\\n", sizeof({cname}));')
        for fname, _ in cls._fields_:
            lines.append(f'  printf("{cname}.{fname} %zu\\n", offsetof({cname}, {fname}));')
    for k in consts:
        lines.append(f'  printf("{k} %d\\n", (int)({k}));')
    lines += ['  return 0;', '}']
    src, exe = tmp_path / "probe.c", tmp_path / "probe"
    src.write_text("\n".join(lines))
    r = subprocess.run(["gcc", "-std=c99", "-I", os.path.join(root, "include"), str(src), "-o", str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = dict(l.rsplit(" ", 1) for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    for cname, cls in structs.items():
        assert int(got[cname]) == ctypes.sizeof(cls), cname
        for fname, _ in cls._fields_:
            assert int(got[f"{cname}.{fname}"]) == getattr(cls, fname).offset, (cname, fname)
    for k, v in consts.items():
        assert int(got[k]) == v, k
    # the engine's string -> enum tables are the same numbers
    from voicesplit_b200.engine import MaskEngine
    assert MaskEngine.PHASE_MODES == {"q1": int(got["VS_ISTFT_Q1"]), "corrected": int(got["VS_ISTFT_CORRECTED"])}


@pytest.mark.skipif(shutil.which("g++") is None, reason="no C++ compiler")
def test_ctypes_signatures_match_the_header_prototypes(tmp_path):
    """Arity and argument class (pointer / 32-bit int / 64-bit int / float / double) of every prototype in the public header, taken
    from the C++ type system, against the argtypes / restype voicesplit_b200/_cabi.py binds."""
    import ctypes
    from voicesplit_b200 import _cabi
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    probe = r'''
#include <cstdio>
#include <type_traits>
#include "voicesplit_b200.h"
template <class T> constexpr char cls() {
    return std::is_pointer<T>::value ? 'p' : std::is_same<T, float>::value ? 'f' : std::is_same<T, double>::value ? 'd'
           : (std::is_integral<T>::value && sizeof(T) == 4) ? 'i' : (std::is_integral<T>::value && sizeof(T) == 8) ? 'l' : '?';
}
template <class F> struct Sig;
template <class R, class... A> struct Sig<R (*)(A...)> {      // decltype(&fn) is unevaluated: nothing to link against
    static void show(const char* name) {
        const char s[] = {cls<A>()..., 0};
        std::printf("%s %c %s\n", name, cls<R>(), s);
    }
};
int main() {
%s
    return 0;
}
'''
    body = "\n".join(f'    Sig<decltype(&{n})>::show("{n}");' for n in _cabi.SIGNATURES)
    src, exe = tmp_path / "sig.cpp", tmp_path / "sig"
    src.write_text(probe.replace("%s\n    return 0;", body + "\n    return 0;"))
    r = subprocess.run(["g++", "-std=c++17", "-I", os.path.join(root, "include"), str(src), "-o", str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    got = {}
    for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines():
        parts = line.split(" ")
        got[parts[0]] = (parts[1], parts[2] if len(parts) > 2 else "")

    def c(t):
        if t is None:
            return "v"
        if t in (ctypes.c_void_p, ctypes.c_char_p) or hasattr(t, "contents") or issubclass(t, ctypes._CFuncPtr):
            return "p"
        if t is ctypes.c_float:
            return "f"
        if t is ctypes.c_double:
            return "d"
        return "i" if ctypes.sizeof(t) == 4 else "l"
    for name, (res, args) in _cabi.SIGNATURES.items():
        assert got[name] == (c(res), "".join(c(a) for a in args)), (name, got[name])


def test_every_entry_point_rejects_a_null_engine_without_crashing():
    """'integer status return, no exceptions across the boundary' (SURVEY 8b): each entry point called with a NULL engine and NULL
    buffers answers with an error code (size queries with 0) - on a host without a GPU too."""
    import ctypes
    from voicesplit_b200 import _cabi
    lib = _cabi.load()
    N = ctypes.c_void_p(0)
    no_sync, no_hook = ctypes.cast(None, _cabi.STAT_ALLREDUCE_FN), ctypes.cast(None, _cabi.BACKWARD_HOOK_FN)
    failing = [
        lambda: lib.vs_engine_load_params(N, None, N), lambda: lib.vs_forward(N, N, N, N, N, 1, 1, 0, N, 0, N),
        lambda: lib.vs_forward_host(N, N, N, N, N, 1, 1, 0, N), lambda: lib.vs_forward_host_submit(N, 0, N, N, N, N, 1, 1, 0),
        lambda: lib.vs_forward_host_wait(N, 0), lambda: lib.vs_forward_host_reserve(N, 1, 1, 0),
        lambda: lib.vs_conv_stack(N, N, N, 1, 1, 0, N, 0, N),
        lambda: lib.vs_train_forward(N, None, N, N, N, 1, 1, N, 0, N), lambda: lib.vs_train_backward(N, N, N, N, N, None, N, N, 1, 1, N, 0, N),
        lambda: lib.vs_engine_set_train_tensor_cores(N, 1), lambda: lib.vs_engine_set_sync_bn(N, no_sync, N, 1),
        lambda: lib.vs_engine_set_backward_hook(N, no_hook, N),
        lambda: lib.vs_audio_configure(N, None, N), lambda: lib.vs_wav2spec(N, N, N, N, 1, 1, N, 0, N), lambda: lib.vs_spec2wav(N, N, N, N, 1, 2, N, 0, N),
        lambda: lib.vs_loss_configure(N, None, N), lambda: lib.vs_loss_spec2wav(N, N, N, N, 1, 2, N, 0, N),
        lambda: lib.vs_loss_spec2wav_backward(N, N, N, N, N, 1, 2, N, 0, N), lambda: lib.vs_sisnr_loss(N, N, N, N, N, N, N, N, 1, 2, N, 0, N),
        lambda: lib.vs_sisnr_wav(N, N, N, N, N, N, 1, 1, N), lambda: lib.vs_sdr(N, N, N, N, 1, 1, N, 0, N),
        lambda: lib.vs_encoder_configure(N, None, N), lambda: lib.vs_encoder_load_params(N, None, N),
        lambda: lib.vs_encoder_mel(N, N, N, 1, 1, N, 0, N), lambda: lib.vs_encoder_forward(N, N, N, 1, 1, N, 0, N),
        lambda: lib.vs_encoder_dvector(N, N, N, 1, 1, N, 0, N),
        lambda: lib.vs_engine_set_profiling(N, 1), lambda: lib.vs_debug_conv_layer(N, 0, N, N, 1, 1, 0, N),
        lambda: lib.vs_debug_lstm_head(N, N, N, N, N, N, 1, 1, 0, N), lambda: lib.vs_debug_lstm_timing(N, None),
    ]
    for i, call in enumerate(failing):
        assert call() < 0, i
    assert lib.vs_last_error()
    for size in (lib.vs_workspace_bytes(N, 1, 1, 0), lib.vs_train_workspace_bytes(N, 1, 1), lib.vs_audio_workspace_bytes(N, 1, 1),
                 lib.vs_loss_workspace_bytes(N, 1, 2), lib.vs_encoder_workspace_bytes(N, 1, 1, 1)):
        assert size == 0
    assert lib.vs_engine_destroy(N) == 0 and lib.vs_last_launch_count(N) == 0 and lib.vs_profile_read(N, 0, None, None) == 0


def test_bench_algorithmic_flops_are_the_survey_figures():
    """roofline.achieved is algorithmic FLOPs / time: the per-utterance figures bench.py uses are SURVEY.md 8(d)'s (2 x MAC, forward),
    with the d-vector folded into a per-utterance gate bias (the smaller of the survey's two input-projection figures)."""
    import importlib.util
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(root, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    want = {(301, 601): dict(conv=195.96, conv5x5_layer=37.049, lstm_input_proj=9.26, lstm_recurrence=0.771, fc=0.506, total=(206.4, 207.0)),
            (601, 257): dict(conv=167.32, conv5x5_layer=31.63, lstm_input_proj=7.91, lstm_recurrence=1.54, fc=0.762, total=(177.5, 178.51))}
    for (T, F), w in want.items():
        f = b.flops_per_utt(T, F)
        for k, v in w.items():
            if k == "total":
                assert v[0] <= f[k] / 1e9 <= v[1], (T, F, k, f[k])
            else:
                assert abs(f[k] / 1e9 - v) <= 0.006 * v, (T, F, k, f[k])
        assert f["total"] == f["conv"] + f["lstm"] + f["fc"] and f["lstm"] == f["lstm_input_proj"] + f["lstm_recurrence"]
    assert b.padded_f(257) == 264 and b.padded_f(601) == 608


def test_product_fails_loudly_without_the_cuda_library(monkeypatch, tmp_path):
    """No CPU or PyTorch fallback: with libvoicesplit_sm100.so absent the engine cannot be constructed at all."""
    from voicesplit_b200 import _cabi
    from voicesplit_b200.engine import MaskEngine
    monkeypatch.setattr(_cabi, "_lib", None)
    monkeypatch.setattr(_cabi, "LIB_PATH", str(tmp_path / "libvoicesplit_sm100.so"))
    with pytest.raises(ImportError, match="no CPU or PyTorch fallback"):
        MaskEngine(33, 16, 24, 40, 33)


def test_product_code_never_touches_the_oracle():
    """oracle/ is test infrastructure: only tests/, __graft_entry__.smoke()/build() and bench.py's baseline / parity legs may import
    it.  Checked on the source of everything under voicesplit_b200/ and models/ (Python and CUDA / C++), and on bench.py's timed arm:
    every oracle import there sits inside one of the named baseline / evidence functions."""
    import ast
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    offenders = []
    for top in ("voicesplit_b200", "models", "include"):
        for dirpath, _dirs, files in os.walk(os.path.join(root, top)):
            if "_build" in dirpath or "__pycache__" in dirpath:
                continue
            for f in files:
                if not f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                    continue
                text = open(os.path.join(dirpath, f), errors="replace").read()
                if f.endswith(".py"):
                    for node in ast.walk(ast.parse(text)):
                        names = [a.name for a in node.names] if isinstance(node, ast.Import) else \
                                [node.module or ""] if isinstance(node, ast.ImportFrom) else []
                        if any(n == "oracle" or n.startswith("oracle.") or n in ("ref_import", "torch_port") for n in names):
                            offenders.append(os.path.join(dirpath, f))
                elif _includes_oracle(text):
                    offenders.append(os.path.join(dirpath, f))
    assert not offenders, offenders
    tree = ast.parse(open(os.path.join(root, "bench.py")).read())
    allowed = {"cpu_reference_throughput", "stock_torch_gpu_baseline", "config2_conv_stack", "main", "extra_measurements"}
    for fn in [n for n in ast.walk(tree) if isinstance(n, ast.FunctionDef)]:
        for node in ast.walk(fn):
            if isinstance(node, ast.ImportFrom) and (node.module or "").split(".")[0] == "oracle":
                assert fn.name in allowed, fn.name
    assert not any(isinstance(n, (ast.Import, ast.ImportFrom)) and "oracle" in ast.dump(n) for n in tree.body)     # nothing at module level


def _includes_oracle(text):
    import re
    return re.search(r'#include\s+["<][^">]*oracle', text) is not None


def test_bench_reference_arm_under_torchrun_prints_one_line_from_rank_0():
    """Launched the way the driver launches N > 1 (torch.distributed.run, one process per GPU slot): rank 0 alone measures and prints,
    the other ranks exit 0 without work."""
    import json
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    port = 29500 + os.getpid() % 400
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", str(port), os.path.join(root, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                        "--warmup", "0", "--frames", "41", "--freq", "33"], capture_output=True, text=True, timeout=600, cwd=root)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, r.stdout[-2000:]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 2 and d["value"] > 0 and d["cpu_baseline"]["cores"] >= 1
