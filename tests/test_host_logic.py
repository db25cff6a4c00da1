"""CPU: host-side logic of the drop-in modules that needs no GPU -- data preparation
(reference utils.py quirks), config parsing, metrics, start block, module surfaces."""
import json
import os

import numpy as np
import pytest

import cases


def test_utils_match_reference(golden_dir):
    import utils
    g = np.load(os.path.join(golden_dir, 'utils.npz'))
    split = cases.raw_split()
    pos = utils.add_positional_embeddings({'pos_embed_dim': 4}, split['covarep'].copy())
    np.testing.assert_array_equal(pos, g['pos'])
    # the quirk: only the first pos_embed_dim data points get sin/cos, the rest raw positions
    np.testing.assert_array_equal(pos[5, :, -1], np.arange(pos.shape[1]))
    norm, masks = utils.normalize_data({k: v.copy() for k, v in split.items()})
    np.testing.assert_array_equal(norm['covarep'], g['covarep'])
    np.testing.assert_array_equal(norm['facet'], g['facet'])
    np.testing.assert_array_equal(masks['covarep'], g['m_covarep'])
    np.testing.assert_array_equal(masks['facet'], g['m_facet'])
    assert norm['covarep'].shape[-1] == split['covarep'].shape[-1] - 1       # constant feature dropped


def test_start_block_is_sklearns():
    import sif_functions
    from oracle import sif_oracle as so
    np.testing.assert_array_equal(sif_functions.start_block(300, 1), so.start_block(300, 1))
    assert sif_functions.start_block(40, 3).shape == (40, 13)


def test_module_surface_matches_reference_imports():
    """The names the reference imports from each module (SURVEY.md §8b) exist here."""
    import sif_functions, sif, losses, models, simplesif, utils, sentiment_model  # noqa: E401
    for mod, names in (
        (sif_functions, 'Params seq2weight SIF_embedding get_weighted_average compute_pc remove_pc'),
        (sif, 'load_weights get_sentence_embeddings get_sentence_word_weights get_word_weights'),
        (losses, 'get_log_prob_matrix get_word_log_prob_angular get_word_log_prob_dot_prod '
                 'get_word_log_prob_angular2 get_normal_log_prob full_loss iemocap_loss pom_loss'),
        (models, 'AudioVisualGeneratorConcat AudioVisualGenerator AudioVisualGeneratorMultimodal'),
        (simplesif, 'optimize_latents update_masks update_masks_vect read_config parse_arguments main'),
        (utils, 'load_data normalize_data MMData MMDataExtra add_positional_embeddings'),
        (sentiment_model, 'SentimentData SentimentModel train_sentiment_for_latents'),
    ):
        for n in names.split():
            assert hasattr(mod, n), (mod.__name__, n)


def test_generator_module_layout():
    import models
    m = models.AudioVisualGeneratorMultimodal(300, 76, 49, norm='layer_norm', frozen_weights=False)
    assert list(m.embed2out.keys()) == ['audio', 'visual', 'audiovisual', 'textaudio', 'textvisual',
                                        'textaudiovisual']
    assert m.embed2out['textaudiovisual']['mu'].weight.shape == (425, 300)
    assert sum(p.numel() for p in m.parameters()) == 843400            # SURVEY.md §8a A6
    m1 = models.AudioVisualGeneratorMultimodal(300, 76, 49, unimodal=True)
    assert sum(p.numel() for p in m1.parameters()) == 75250
    assert not any(p.requires_grad for p in m1.embed2out.parameters())   # frozen by default
    with pytest.raises(NotImplementedError):
        models.AudioVisualGeneratorMultimodal(8, 2, 2, norm='group_norm')


def test_parse_arguments_merges_config(tmp_path):
    import simplesif
    cfg = {'config_num': 3, 'lr': 0.01, 'n_epochs': 100, 'optimizer': 'adam', 'norm': 'layer_norm', 'e2e': True,
           'pos_embed_dim': 2, 'n_sentiment_epochs': 50}
    f = tmp_path / 'cfg' / 'config_3.json'
    f.parent.mkdir()
    f.write_text(json.dumps(cfg))
    args = simplesif.parse_arguments([str(f), 'mosi', '--unimodal', '--pos_embed_dim', '4', '--e2e', 'n',
                                      '--sentiment_epochs', '7'])
    assert args['dataset'] == 'mosi' and args['unimodal'] is True
    assert args['optimizer'] == 'adam'            # the JSON wins over the flag default (reference 228-229)
    assert args['pos_embed_dim'] == 4 and args['e2e'] is False and args['n_sentiment_epochs'] == 7


def test_update_masks():
    import simplesif
    ids = np.array([[3, 0, 5], [0, 0, 1]])
    m = {}
    simplesif.update_masks(m, ids, 4)
    assert m['text'].shape == (2, 3, 4)
    np.testing.assert_array_equal(m['text'][:, :, 0], (ids != 0).astype(int))
    x = np.ones((2, 3, 2))
    x[0, 1, 1] = 0
    simplesif.update_masks_vect(m, x, 'text_align')
    np.testing.assert_array_equal(m['text_align'][:, :, 0], [[1, 0, 1], [1, 1, 1]])


def test_metrics_keys():
    import losses
    rng = np.random.default_rng(0)
    y = rng.uniform(-3, 3, 50)
    r = losses.full_loss(y + 0.1 * rng.standard_normal(50), y)
    assert set(r) == {'mae', 'accuracy', 'corr', 'mult_acc', 'f_score', 'confusion_matrix', 'class_report'}
    r = losses.pom_loss(rng.uniform(1, 7, (20, 3)), rng.uniform(1, 7, (20, 3)))
    assert set(r) == {'mae', 'corr', 'mult_acc', 'f_score'} and len(r['mae']) == 3


def test_sweep_grid_matches_reference_generator():
    """sweep.make_grid is the 2^9 grid of reference configs/make_configs.py:16-32 in product order."""
    import sweep
    grid = sweep.make_grid()
    assert len(grid) == 512 and [c['config_num'] for c in grid] == list(range(512))
    varied = [k for k, v in sweep.GRID.items() if len(v) == 2]
    assert sorted(varied) == sorted(['sentiment_hidden_size', 'lr', 'sentiment_lr', 'n_epochs', 'word_loss_weight',
                                     'likelihood_weight', 'pos_embed_dim', 'norm', 'optimizer'])
    assert len({tuple(c[k] for k in varied) for c in grid}) == 512
    assert all(c['e2e'] is True and c['n_sentiment_epochs'] == 400 and c['seq_len'] == 20 for c in grid)
    We, weights, splits = sweep.synthetic_mosi(sizes=(30, 10, 12))
    assert We.shape == (3016, 300) and weights.shape == (3016,) and weights[0] == 1.0
    assert [s['text'].shape for s in splits] == [(30, 20), (10, 20), (12, 20)]
    assert all((s['covarep'][s['text'] == 0] == 0).all() for s in splits)


@pytest.mark.parametrize('tag', sorted(cases.SENTIMENT_CASES))
def test_sentiment_regressor_matches_reference(golden_dir, tag, tmp_path, capsys):
    """The downstream regressor is plain torch and 'unchanged' by the task's scope: on the CPU it must
    reproduce the reference's sentiment_model.train_sentiment_for_latents -- metrics, validation curve,
    files, and the state it leaves torch's global generator in (shuffles of later runs depend on it)."""
    import torch
    import sentiment_model
    g = np.load(os.path.join(golden_dir, 'sentiment.npz'))
    cfg = cases.SENTIMENT_CASES[tag]
    args, lat, labs = cases.sentiment_inputs(**cfg)
    torch.manual_seed(cfg['seed'])
    results, (_, valid_losses) = sentiment_model.train_sentiment_for_latents(
        args, tuple(torch.tensor(x) for x in lat), tuple(labs), torch.device('cpu'), model_save_path=str(tmp_path))
    next_draw = torch.rand(1).numpy()
    capsys.readouterr()
    for k in ('mae', 'corr', 'mult_acc', 'f_score', 'accuracy'):
        if k in results:
            np.testing.assert_allclose(np.asarray(results[k], dtype=np.float64), g['%s_after_%s' % (tag, k)],
                                       rtol=0, atol=2e-6, err_msg=k)
    np.testing.assert_allclose(valid_losses, g[tag + '_valid_losses'], rtol=1e-6)
    np.testing.assert_array_equal(next_draw, g[tag + '_next_draw'])
    before = json.load(open(tmp_path / 'test_results_before.json'))
    np.testing.assert_allclose(np.asarray(before['mae'], dtype=np.float64), g[tag + '_before_mae'], atol=2e-6)
    for name in ('test_results_after.json', 'senti_train_loss.txt', 'senti_valid_loss.txt', 'senti.bin'):
        assert (tmp_path / name).exists(), name


def test_bench_reference_arm_prints_one_json_line():
    """bench.py --impl reference (the CPU arm the driver runs beside the GPU arm): stdout is exactly one
    JSON line with the contract's keys, whatever the libraries print (fd 1 is pointed at stderr)."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, MMB_REF_SAMPLE='300', MMB_BENCH_V='5000')
    r = subprocess.run([sys.executable, os.path.join(root, 'bench.py'), '--impl', 'reference', '--steps', '1',
                        '--warmup', '0'], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout[:500]
    line = json.loads(lines[0])
    assert line['impl'] == 'reference' and line['unit'] == 'utterances/s' and line['higher_is_better'] is True
    assert line['value'] > 0 and line['cpu_baseline']['kind'] in ('port', 'reference') and line['cpu_baseline']['cores'] >= 1
    assert line['e2e'] == {'value': line['value'], 'unit': line['unit'], 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
    assert line['gpu_launches'] == 0 and 'workload' in line['config']


def test_bench_gpu_arm_refuses_to_run_without_cuda():
    """No CPU fallback: without a CUDA device the GPU arm exits non-zero and prints no result line."""
    import subprocess
    import sys
    import torch
    if torch.cuda.is_available():
        pytest.skip('CUDA device present')
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, 'bench.py'), '--steps', '1', '--warmup', '0'],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode != 0
    assert not [l for l in r.stdout.splitlines() if l.strip().startswith('{')]


def test_epoch_index_helpers_draw_like_the_dataloader():
    """The graph-replay loops never iterate the DataLoader; they take its index batches from the batch sampler.
    That is only equivalent if the helpers consume torch's global generator exactly as `for x in loader` does
    (one base-seed draw per iterator, then the RandomSampler's seed) -- batch order and the generator state
    afterwards must match, for shuffled and unshuffled loaders, over several epochs."""
    import torch
    from torch.utils.data import DataLoader, TensorDataset
    import simplesif
    import sentiment_model

    class Rows(TensorDataset):
        def __getitem__(self, i):
            return i, self.tensors[0][i]

    ds = Rows(torch.arange(23.))
    for shuffle in (True, False):
        for helper in (lambda l: [b.tolist() for b in simplesif._epoch_index_batches(l, 'cpu')],
                       lambda l: [b.tolist() for b in sentiment_model._index_batches(l, 'cpu')],
                       lambda l: (lambda f, s: [f[sum(s[:k]):sum(s[:k + 1])].tolist() for k in range(len(s))])(
                           *simplesif._epoch_indices(l, 'cpu')),
                       lambda l: (lambda f, s: [f[sum(s[:k]):sum(s[:k + 1])].tolist() for k in range(len(s))])(
                           *sentiment_model._epoch_indices(l, 'cpu'))):
            loader = DataLoader(ds, batch_size=5, shuffle=shuffle)
            torch.manual_seed(11)
            want = [[j.tolist() for j, _ in loader] for _ in range(3)]
            want_next = torch.rand(1)
            torch.manual_seed(11)
            got = [helper(loader) for _ in range(3)]
            got_next = torch.rand(1)
            assert got == want, (shuffle, got[0], want[0])
            assert torch.equal(got_next, want_next)
    assert sorted(sum(want[0], [])) == list(range(23)) and [len(b) for b in want[0]] == [5, 5, 5, 5, 3]


def test_id_dataset_and_moment_batches_keep_the_reference_tuple_layout():
    """Host wiring of the two step-side extensions (SURVEY.md 8f N3, section 7 H6): `MMDataIds` returns the
    reference's tuple positions (utils.py:231-233) with ids in the text slot, `_batch_dicts` wraps them as
    TokenIds and builds the six MMB2 modalities from base parts, and `_with_moments` swaps the Gaussian inputs
    for per-utterance moments without touching the word term's inputs."""
    import torch
    import losses
    import simplesif
    import utils
    N, L, d, A, Vd, V = 6, 4, 8, 3, 2, 10
    g = torch.Generator().manual_seed(0)
    table = torch.randn(V, d, generator=g)
    ids = torch.randint(0, V, (N, L), generator=g)
    aud, vis = torch.randn(N, L, A, generator=g), torch.randn(N, L, Vd, generator=g)
    masks = {'covarep': torch.ones(N, L, A), 'facet': torch.ones(N, L, Vd)}
    ds = utils.MMDataIds(ids, aud, vis, masks, torch.rand(V, generator=g), table, 'cpu')
    assert len(ds) == N and ds.text_mask.shape == (N, L) and ds.text_weights.shape == (N, L)
    j = torch.tensor([4, 1, 2])
    x = ds[j]
    assert len(x) == 8 and x[1].dtype == torch.int64 and torch.equal(x[1], ids[j])
    args = {'dataset': 'mosi', 'unimodal': False}
    _, data, bmasks = simplesif._batch_dicts(args, x, ds.table)
    assert isinstance(data['text'], losses.TokenIds) and data['text'].shape == (3, L, d)
    assert torch.equal(data['text'].materialize(), table[ids[j]])
    assert set(data) == {'text', 'audio', 'visual', 'text_weights', 'audiovisual', 'textaudio', 'textvisual',
                         'textaudiovisual'}
    assert [type(p).__name__ for p in data['textaudiovisual'].parts] == ['TokenIds', 'Tensor', 'Tensor']
    assert torch.equal(bmasks['text'], (ids[j] != 0).float())
    # moments: the Gaussian slots become MomentStats rows, masks None, the word term's inputs stay
    mom = {k: losses.MomentStats(torch.zeros(N, 3, F)) for k, F in (('audio', A), ('visual', Vd), ('text_gauss', d))}
    xm = simplesif._with_moments(args, x, mom)
    _, data, bmasks = simplesif._batch_dicts(args, xm, ds.table)
    assert isinstance(data['audio'], losses.MomentStats) and data['audio'].stats.shape == (3, 3, A)
    assert bmasks['audio'] is None and isinstance(data['text'], losses.TokenIds)
    assert [type(p).__name__ for p in data['textaudiovisual'].parts] == ['MomentStats'] * 3
    assert [s.shape[-1] for s in losses._segments(data['textaudiovisual'], bmasks['textaudiovisual'])] == [d, A, Vd]
    # POM layout: aligned text in slots 8 / 9
    dse = utils.MMDataExtraIds(ids, aud, vis, dict(masks, text_align=torch.ones(N, L, d)), torch.rand(V), table,
                               torch.randn(N, L, d), 'cpu')
    xe = simplesif._with_moments({'dataset': 'pom', 'unimodal': False}, dse[j], mom)
    assert len(xe) == 10 and isinstance(xe[8], losses.MomentStats) and xe[9] is None
    _, data, _ = simplesif._batch_dicts({'dataset': 'pom', 'unimodal': False}, xe, dse.table)
    assert isinstance(data['text'], losses.TokenIds) and isinstance(data['textaudio'].parts[0], losses.MomentStats)


def test_loaders_read_the_reference_file_layout(tmp_path, monkeypatch, golden_dir):
    """utils.load_data and its parts (reference utils.py:10-128): the id / vocabulary / table files by their
    reference paths, the h5 splits through h5py (a stand-in module here: the image has no h5py), and the real
    POM id matrices (kept in tests/golden/sif_pom_full.npz) laid out as the reference ships them."""
    import pickle
    import sys
    import types
    import utils
    root = tmp_path
    (root / 'pom').mkdir()
    (root / 'mosi').mkdir()
    (root / 'data').mkdir()
    rng = np.random.default_rng(0)
    ids = {s: rng.integers(0, 50, size=(n, 9)).astype(np.int64) for s, n in (('train', 5), ('valid', 3), ('test', 4))}
    for s, a in ids.items():
        np.save(root / 'pom' / ('pom_%s_ids.npy' % s), a)
    table = rng.standard_normal((50, 8)).astype(np.float32)
    np.save(root / 'pom' / 'glove.pom.npy', table)
    np.save(root / 'mosi' / 'glove_300_mosi.npy', table)
    json.dump({'a': 1, '##b': 0}, open(root / 'pom' / 'glove_mappings.pom.json', 'w'))
    pickle.dump({'the': 3}, open(root / 'mosi' / 'word2ix_300_mosi.pkl', 'wb'))
    store = {}
    for name in ('pom_data.h5', 'mosi_data.h5'):
        store[str(root / 'data' / name)] = {
            sp: {k: rng.standard_normal((n, 2)) for k in ('facet', 'covarep', 'text', 'label', 'lengths', 'id')}
            for sp, n in (('train', 5), ('valid', 3), ('test', 4))}

    class FakeFile(object):
        def __init__(self, path, mode):
            if path not in store:
                raise FileNotFoundError(path)
            self.d = store[path]

        def __enter__(self):
            return self.d

        def __exit__(self, *a):
            return False
    monkeypatch.setitem(sys.modules, 'h5py', types.SimpleNamespace(File=FakeFile))
    w2i, We, (tr, va, te) = utils.load_data({'dataset': 'pom', 'data_root': str(root)})
    assert w2i == {'a': 1, '##b': 0}
    np.testing.assert_array_equal(We, table)
    np.testing.assert_array_equal(tr['text_id'], ids['train'])
    np.testing.assert_array_equal(te['text_id'], ids['test'])
    assert set(va) == {'facet', 'covarep', 'text', 'label', 'text_id'} and va['covarep'].shape == (3, 2)
    w2i, We, (tr, va, te) = utils.load_data({'dataset': 'mosi', 'data_root': str(root)})
    assert w2i == {'the': 3} and set(tr) == {'facet', 'covarep', 'text', 'lengths', 'label', 'id'}
    with pytest.raises(ValueError):
        utils.load_data({'dataset': 'nope'})
    with pytest.raises(FileNotFoundError):
        utils.load_data({'dataset': 'iemocap', 'emotion': 'happy', 'data_root': str(root)})
    g = np.load(os.path.join(golden_dir, 'sif_pom_full.npz'))
    real = tmp_path / 'real'
    (real / 'pom').mkdir(parents=True)
    for s in ('valid', 'test'):
        np.save(real / 'pom' / ('pom_%s_ids.npy' % s), g[s + '_ids'].astype(np.int64))
    v, t = utils.load_text_ids('pom', str(real), ('valid', 'test'))
    assert v.shape == (100, 1089) and t.shape == (203, 1357) and t.dtype == np.int64
    np.testing.assert_array_equal(v, g['valid_ids'])
    np.testing.assert_array_equal(t, g['test_ids'])


def test_batched_regressors_equal_sequential_ones(capsys):
    """SURVEY 8f N4: K grid points' downstream regressors trained as ONE batched model (sentiment_batched) give the
    metrics, loss curves and random-stream position of K sequential train_sentiment_for_latents runs -- same
    initialisation and shuffles per config (the generator is replayed from where each run would start), different
    step sizes per config.  CPU here (plain torch both ways); the GPU test repeats it with graph replay."""
    import torch
    import sentiment_model
    import sentiment_batched
    jobs, want = [], []
    for k, (seed, lr) in enumerate([(11, 0.1), (12, 0.01), (13, 0.05)]):
        args, lat, labs = cases.sentiment_inputs(dataset='mosi', n_out=1, early_stopping=False, seed=81 + k)
        args = dict(args, sentiment_lr=lr, n_sentiment_epochs=25)
        lat_t = tuple(torch.tensor(x) for x in lat)
        torch.manual_seed(seed)
        torch.rand(3)                                          # the stream is somewhere in the middle, as after latent loops
        state = torch.get_rng_state()
        res, (tl, vl) = sentiment_model.train_sentiment_for_latents(args, lat_t, tuple(labs), torch.device('cpu'))
        want.append((res, tl, vl, torch.get_rng_state()))
        jobs.append(sentiment_batched.RegressorJob(args, lat_t, tuple(labs), rng_state=state))
    assert all(sentiment_batched.can_batch(j.args, j.labels) for j in jobs)
    sentiment_batched.run_jobs(jobs, torch.device('cpu'))
    capsys.readouterr()
    for job, (res, tl, vl, final_state) in zip(jobs, want):
        for k in ('mae', 'corr', 'mult_acc', 'f_score', 'accuracy'):
            np.testing.assert_allclose(np.asarray(job.results[k], dtype=np.float64), np.asarray(res[k], dtype=np.float64),
                                       rtol=0, atol=1e-5, err_msg=k)
        np.testing.assert_allclose(job.train_losses, tl, rtol=1e-5)
        np.testing.assert_allclose(job.valid_losses, vl, rtol=1e-5)
        assert torch.equal(job.final_rng_state, final_state)   # exactly the draws the sequential run makes
    # (N, 1) labels and early stopping stay with the sequential module
    args, lat, labs = cases.sentiment_inputs(**cases.SENTIMENT_CASES['mosi_column_labels'])
    assert not sentiment_batched.can_batch(args, labs)
    args, lat, labs = cases.sentiment_inputs(**cases.SENTIMENT_CASES['mosi_early_stopping'])
    assert not sentiment_batched.can_batch(args, labs)
    args, lat, labs = cases.sentiment_inputs(**cases.SENTIMENT_CASES['pom'])
    assert sentiment_batched.can_batch(args, labs)


def test_bench_refuses_a_stale_ncu_record(tmp_path, monkeypatch):
    """VERDICT r1: roofline.traffic was multiplied out of an ncu capture of a DIFFERENT kernel instantiation.
    bench.py now takes the kernel name from the library's dispatch and uses the committed capture only when ncu
    saw the same instantiation (template arguments included, whatever the spelling)."""
    import importlib
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    bench = importlib.import_module('bench')
    n = bench.norm_kernel_name
    assert n('void mmb::sif_embed_warp_kernel<3, 0, 2, 4, 0>(const float4 *, int, int)') == \
        n('sif_embed_warp_kernel<3,false,2,4,false>') == 'sif_embed_warp_kernel<3,0,2,4,0>'
    assert n('void sif_embed_prescaled_kernel<3, 2, 4>(const float4 *, int, int, const int *)') == \
        n('sif_embed_prescaled_kernel<3,2,4>')
    assert n('sif_embed_prescaled_kernel<3,2,4>') != n('sif_embed_warp_prefetch_kernel<3,2,4>')
    (tmp_path / 'profiles').mkdir()
    rec = {'zipf': {'ncu_kernel_name': 'void sif_embed_warp_kernel<3, 0, 2, 4, 0>(const float4 *)',
                    'dram_bytes_per_utterance': 7458.0, 'source': 'x'}}
    json.dump(rec, open(tmp_path / 'profiles' / 'embed_traffic.json', 'w'))
    monkeypatch.setattr(bench, 'ROOT', str(tmp_path))
    got, why = bench.load_ncu_record('sif_embed_prescaled_kernel<3,2,4>', 'zipf')
    assert got is None and 'stale capture' in why
    got, why = bench.load_ncu_record('sif_embed_warp_kernel<3,false,2,4,false>', 'zipf')
    assert got is not None and got['dram_bytes_per_utterance'] == 7458.0
    got, why = bench.load_ncu_record('sif_embed_warp_kernel<3,false,2,4,false>', 'uniform')
    assert got is None and 'no uniform record' in why
    # the committed record matches the kernel the library dispatches for the bench workload
    monkeypatch.setattr(bench, 'ROOT', root)
    got, why = bench.load_ncu_record('sif_embed_prescaled_kernel<3,2,4>', 'zipf')
    assert got is not None, why


def test_graph_capture_keeps_the_collector_out(monkeypatch):
    """graph_capture.capture: Python's cyclic collector is off for the whole capture (a dead cycle owning an
    earlier CUDAGraph, collected inside a capture, invalidates it) and back in its previous state afterwards,
    also when the body raises."""
    import contextlib
    import gc
    import torch
    import graph_capture
    seen = []

    @contextlib.contextmanager
    def fake_graph(graph, **kwargs):
        seen.append(('enter', gc.isenabled(), graph, kwargs))
        yield
        seen.append(('exit', gc.isenabled()))

    monkeypatch.setattr(torch.cuda, 'graph', fake_graph)
    assert gc.isenabled()
    with graph_capture.capture('g', pool=None):
        seen.append(('body', gc.isenabled()))
    assert seen == [('enter', False, 'g', {'pool': None}), ('body', False), ('exit', False)]
    assert gc.isenabled()
    with pytest.raises(RuntimeError):
        with graph_capture.capture('g'):
            raise RuntimeError('boom')
    assert gc.isenabled()
    gc.disable()
    try:
        with graph_capture.capture('g'):
            pass
        assert not gc.isenabled()                       # was off before: stays off
    finally:
        gc.enable()
