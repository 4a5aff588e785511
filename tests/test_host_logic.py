"""CPU tests of the host side: the C ABI loads and exports every declared symbol, argument validation mirrors the
reference's error behaviour, and the product never falls back to the CPU."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from speechbrain_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "sbk.h")).read()
    declared = set(re.findall(r"\b(sbk_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    L = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(L, name), f"{name} declared in include/sbk.h but not exported by libsbk.so"
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    assert _lib.lib().sbk_version() >= 100


def test_no_cpu_fallback():
    from speechbrain_b200.lobes.features import Fbank
    from speechbrain_b200.processing.features import InputNormalization
    with pytest.raises(RuntimeError, match="CUDA"):
        Fbank(n_fft=400, n_mels=80)(torch.zeros(1, 1600))
    n = InputNormalization(norm_type="sentence").eval()
    with pytest.raises(RuntimeError, match="CUDA"):
        n(torch.zeros(1, 4, 8))


def test_product_does_not_import_oracle():
    for dp, _, files in os.walk(os.path.join(ROOT, "speechbrain_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dp, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f"{f} references oracle/"


def test_constructor_validation_mirrors_reference():
    from speechbrain_b200.lobes.features import Fbank
    from speechbrain_b200.lobes.models.transformer.TransformerASR import TransformerASR
    from speechbrain_b200.processing.features import InputNormalization
    with pytest.raises(ValueError):
        InputNormalization(mean_norm=False)  # processing/features.py:1374-1375
    with pytest.raises(ValueError):
        InputNormalization(norm_type="speaker")
    with pytest.raises(ValueError):
        InputNormalization(avg_factor=0.1)
    with pytest.raises(AssertionError):
        TransformerASR(tgt_vocab=10, input_size=640, attention_type="nope")  # Transformer.py:141-147
    with pytest.raises(AssertionError):
        TransformerASR(tgt_vocab=10, input_size=640, encoder_module="conformer", attention_type="RoPEMHA",
                       normalize_before=False, causal=False)
    with pytest.raises(NotImplementedError):
        Fbank(deltas=True)
    f = Fbank(n_fft=512, n_mels=80, win_length=32)
    assert (f.win_length, f.hop_length) == (512, 160)  # ms -> samples (processing/features.py:132-137)
    assert list(f.state_dict().keys()) == ["compute_deltas.kernel"]


def test_input_norm_checkpoint_roundtrip(tmp_path):
    from speechbrain_b200.processing.features import InputNormalization
    n = InputNormalization(norm_type="global")
    n.glob_mean, n.glob_std, n.count = torch.arange(4.0), torch.ones(4) * 2, 7
    p = str(tmp_path / "normalizer.ckpt")
    n._save(p)
    stats = torch.load(p)
    assert set(stats) == {"count", "glob_mean", "glob_std"}  # processing/features.py:1488-1495
    m = InputNormalization(norm_type="global")
    m._load(p)
    assert m.count == 7 and torch.equal(m.glob_mean, n.glob_mean)


def test_greedy_outputs_match_reference_postprocessing():
    from speechbrain_b200.decoders.seq2seq import greedy_outputs
    pred = torch.tensor([[5, 6, 2, 2], [7, 8, 9, 10]], dtype=torch.int32)
    hyps, lens, scores, lp = greedy_outputs(pred, torch.zeros(2, 4), None, eos_index=2)
    assert hyps == [[5, 6], [7, 8, 9, 10]]  # decoders/seq2seq.py:306-310 + undo_padding
    assert torch.allclose(lens.flatten(), torch.tensor([0.5, 1.0]))
    assert scores.shape == (2, 1, 4)


def test_seeded_weights_are_order_independent():
    from speechbrain_b200.utils.seeded_init import seeded_tensor
    a = seeded_tensor(0, "Transformer.encoder.layers.3.norm1.norm.weight", (512,))
    b = seeded_tensor(0, "Transformer.encoder.layers.3.norm1.norm.weight", (512,))
    assert torch.equal(a, b) and abs(float(a.mean()) - 1.0) < 0.05


def test_scorer_builder_mirrors_reference_validation():
    """ScorerBuilder / CTCScorer / beam searcher argument checks raise like the reference (scorer.py:1186-1218,1317-1341;
    seq2seq.py:785-804) or with NotImplementedError for what is not built -- never a silent fallback."""
    import pytest
    import torch

    from speechbrain_b200.decoders.scorer import CTCScorer, ScorerBuilder, TransformerLMScorer
    from speechbrain_b200.decoders.seq2seq import S2STransformerBeamSearcher
    from speechbrain_b200.lobes.models.transformer.TransformerLM import TransformerLM
    from speechbrain_b200.nnet.linear import Linear
    ctc = CTCScorer(ctc_fc=Linear(input_size=16, n_neurons=8), blank_index=0, eos_index=2)
    with pytest.raises(AssertionError):  # "Weights and scorers are not matched."
        ScorerBuilder(full_scorers=[ctc], weights={})
    with pytest.raises(ValueError):
        ScorerBuilder(full_scorers=[ctc], weights={"transformerlm": 1.0})
    with pytest.raises(NotImplementedError):
        ScorerBuilder(full_scorers=[], partial_scorers=[ctc], weights={"ctc": 1.0})
    with pytest.raises(NotImplementedError):
        CTCScorer(ctc_fc=None, blank_index=0, eos_index=2, ctc_window_size=10)
    with pytest.raises(NotImplementedError):  # post-norm LM only (the recipe's), head_dim 64
        TransformerLM(vocab=100, d_model=128, nhead=4, num_encoder_layers=1, d_ffn=256, normalize_before=True)
    sb = ScorerBuilder(full_scorers=[ctc], weights={"ctc": 0.4})
    assert sb.weights["ctc"] == 0.4 and sb.weights["transformerlm"] == 0.0 and sb.weights["length"] == 0.0
    # blank / bos / eos must differ for joint CTC/attention decoding (seq2seq.py:797-801)
    with pytest.raises(ValueError):
        S2STransformerBeamSearcher(modules=[torch.nn.Identity(), Linear(input_size=16, n_neurons=8)], bos_index=0, eos_index=2,
                                   beam_size=2, scorer=sb)
    with pytest.raises(ValueError):
        S2STransformerBeamSearcher(modules=[torch.nn.Identity(), Linear(input_size=16, n_neurons=8)], bos_index=1, eos_index=2,
                                   beam_size=2, topk=3)
    lm = TransformerLM(vocab=100, d_model=128, nhead=2, num_encoder_layers=2, d_ffn=256, activation=torch.nn.GELU)
    keys = set(lm.state_dict().keys())
    assert "custom_src_module.emb.Embedding.weight" in keys and "output_proj.layers.2.w.bias" in keys
    assert "encoder.layers.1.self_att.att.in_proj_weight" in keys and "positional_encoding.pe" in keys
    TransformerLMScorer(language_model=lm, temperature=1.15)


def test_bench_dump_outputs(tmp_path, monkeypatch):
    """bench.py --dump-outputs: token ids land as exact float64, activations as float32; a dump over the limit is refused."""
    import numpy as np

    import bench
    ids = torch.tensor([[5, 4999, -1], [7, 8, 2]], dtype=torch.int32)
    enc = torch.randn(2, 3, 4).half()
    bench.dump_outputs(str(tmp_path / "out"), {"token_ids": ids, "encoder_out": enc})
    a, e = np.load(tmp_path / "out" / "token_ids.npy"), np.load(tmp_path / "out" / "encoder_out.npy")
    assert a.dtype == np.float64 and np.array_equal(a, ids.numpy())
    assert e.dtype == np.float32 and np.array_equal(e, enc.float().numpy())
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 16)
    with pytest.raises(SystemExit):
        bench.dump_outputs(str(tmp_path / "big"), {"x": torch.zeros(5)})
    assert not (tmp_path / "big").exists()


def test_no_undefined_names_in_package():
    """Static check (the GPU-only code paths cannot run on the CPU box): every name loaded in speechbrain_b200/*.py, bench.py
    and __graft_entry__.py is defined somewhere in its module (imports, defs, assignments, arguments, comprehensions)."""
    import ast
    import builtins
    import glob
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    files = glob.glob(os.path.join(root, "speechbrain_b200", "**", "*.py"), recursive=True)
    files += [os.path.join(root, "bench.py"), os.path.join(root, "__graft_entry__.py")]
    bad = {}
    for f in files:
        tree = ast.parse(open(f).read())
        defined = set(dir(builtins)) | {"__file__", "__name__"}
        for n in ast.walk(tree):
            if isinstance(n, (ast.Import, ast.ImportFrom)):
                defined.update((a.asname or a.name).split(".")[0] for a in n.names)
            elif isinstance(n, (ast.FunctionDef, ast.ClassDef, ast.AsyncFunctionDef)):
                defined.add(n.name)
            elif isinstance(n, ast.Name) and isinstance(n.ctx, (ast.Store, ast.Del)):
                defined.add(n.id)
            elif isinstance(n, ast.arg):
                defined.add(n.arg)
            elif isinstance(n, ast.ExceptHandler) and n.name:
                defined.add(n.name)
        und = {n.id for n in ast.walk(tree) if isinstance(n, ast.Name) and isinstance(n.ctx, ast.Load) and n.id not in defined}
        if und:
            bad[os.path.relpath(f, root)] = sorted(und)
    assert not bad, bad
