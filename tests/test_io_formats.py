"""SURVEY 8f rank 3: the data_dir / tsv_dir file formats.  `test_save_read_file` is the port of the reference's own
tests/test_helpers.py (same cases, same assertions) against dae_rnn_news_recommendation_b200.io_formats; the second test checks
the CLI's cache: what --restore_previous_data reads is what the preparation step wrote (main_autoencoder.py:161-244)."""
import os
import sys

import numpy as np
import pandas as pd
import pytest
import scipy.sparse as sparse

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from dae_rnn_news_recommendation_b200.io_formats import save_file, read_file  # noqa: E402


def test_save_read_file(tmp_path):
    for data in (np.array([0, 2, 3, 4]), np.array([[0, 2], [2.3, 0]])):
        for name in ('test.csv', 'test.tsv', 'test.npy'):
            save_file(data, path=tmp_path / name)
            assert (data == read_file(tmp_path / name, data_type='numpy')).all()
            os.remove(tmp_path / name)

    for data in (sparse.csr_matrix([0, 0, 0, 0]), sparse.csr_matrix([[0, 0, 0, 0], [0, 0, 0, 0]]), sparse.csr_matrix([1, 2.2, 0, 0]),
                 sparse.csr_matrix([[1, 2.2, 0, 0], [1, 2.2, 5.12312313, 0]])):
        for name in ('test.csv', 'test.tsv', 'test.npz'):
            save_file(data, path=tmp_path / name)
            back = read_file(tmp_path / name, data_type='scipy')
            assert back.shape[-1] == data.shape[-1] and (data != back.reshape(data.shape)).nnz == 0
            os.remove(tmp_path / name)

    for data in (pd.DataFrame([0, 1, 2], index=[5, 3, 2], columns=['dummy']),
                 pd.DataFrame([[0, 1, 2], [2, 3, 4]], index=['apple', 'boy'], columns=['dummy', 'd2', 'd3']),
                 pd.DataFrame(['apple', 'boy', 'cat'], index=[5, 3, 2], columns=['dummy']),
                 pd.DataFrame([['apple', 'boy', 'cat'], ['apple1', 'boy1', 'cat1']], index=['apple', 'boy'], columns=['dummy', 'd2', 'd3'])):
        for name in ('test.csv', 'test.tsv', 'test.parquet', 'test.pkl'):
            save_file(data, path=tmp_path / name)
            assert data.equals(read_file(tmp_path / name, data_type='pandas_df')), name
            os.remove(tmp_path / name)

    for data in (pd.Series([0, 1, 2], index=[5, 4, 3]), pd.Series(['a', 'b', 'c'])):
        for name in ('test.csv', 'test.tsv', 'test.pkl'):
            save_file(data, path=tmp_path / name)
            assert data.equals(read_file(tmp_path / name, data_type='pandas_series')), name
            os.remove(tmp_path / name)


def test_format_and_type_errors(tmp_path):
    with pytest.raises(AssertionError):
        save_file(np.zeros(3), tmp_path / 'a.npz')             # ndarray has no npz writer (helpers.py:196)
    with pytest.raises(AssertionError):
        save_file(pd.Series([1]), tmp_path / 'a.parquet')
    with pytest.raises(AssertionError):
        read_file(tmp_path / 'missing.npy')                    # '[Error] ... is not a file'
    save_file(sparse.eye(3, format='csr'), tmp_path / 'm.npz')
    assert sparse.issparse(read_file(tmp_path / 'm.npz'))      # type inferred from the extension
    save_file(np.eye(2), tmp_path / 'e.npy')
    assert isinstance(read_file(tmp_path / 'e.npy'), np.ndarray)


class _Dirs:
    def __init__(self, root):
        self.data_dir, self.tsv_dir = str(root) + '/data/', str(root) + '/tsv/'
        os.makedirs(self.data_dir), os.makedirs(self.tsv_dir)


def _tiny_corpus(path, n=60, seed=0):
    rng = np.random.RandomState(seed)
    vocab = ['w%03d' % i for i in range(120)]
    cats = ['business', 'health', 'science', 'entertainment']
    rows = []
    for i in range(n):
        c = int(rng.randint(4))
        words = rng.choice(vocab[c * 20:c * 20 + 50], size=int(rng.randint(15, 40)))
        rows.append({'article_id': 1000 + 3 * i, 'title': 't%d' % i, 'story': 's%d' % (i % 11), 'category_publish_name': cats[c],
                     'main_content': ' '.join(words)})
    pd.DataFrame(rows).sample(frac=1, random_state=1).to_parquet(path)


def _same(a, b):
    if sparse.issparse(a):
        return a.shape == b.shape and (a != b).nnz == 0
    return a.equals(b)


def test_data_dir_cache_round_trip(tmp_path):
    """prepare -> data_dir cache -> --restore_previous_data gives the same matrices and labels, under the reference's file names."""
    import main_autoencoder as cli
    _tiny_corpus(tmp_path / 'corpus.snappy.parquet')
    F = cli.check_flags(cli.build_parser().parse_args(['--model_name', 'm', '--train_row', '40', '--validate_row', '15', '--max_features',
                                                        '80', '--data_path', str(tmp_path / 'corpus.snappy.parquet')]))
    model = _Dirs(tmp_path)
    d = cli.prepare_uci(F, model)
    expected = ['article.snappy.parquet', 'article_validate.snappy.parquet', 'article_label_category_publish_name.pkl',
                'article_label_category_publish_name_validate.pkl', 'article_label_story.pkl', 'article_label_story_validate.pkl',
                'article_count_vectorized.npz', 'article_count_vectorized_validate.npz', 'article_binary_count_vectorized.npz',
                'article_binary_count_vectorized_validate.npz', 'article_tfidf_vectorized.npz', 'article_tfidf_vectorized_validate.npz',
                'count_vectorizer.joblib', 'tfidf_transformer.joblib']          # main_autoencoder.py:223-244
    assert sorted(os.listdir(model.data_dir)) == sorted(expected)
    assert d['binary'][0].shape == (40, d['binary'][0].shape[1]) and d['binary'][1].shape[0] == 15
    assert set(np.unique(d['binary'][0].data)) == {1} and d['binary'][0].shape[1] <= 80
    assert (d['articles'].article_id.values == np.sort(d['articles'].article_id.values)).all()      # ascending ids, newest 55 kept
    assert d['articles'].article_id.min() > 1000 + 3 * 4 and d['articles_validate'].article_id.min() > d['articles'].article_id.max()
    r = cli.restore_uci(model)
    for key in ('binary', 'tfidf', 'label_story', 'label_category_publish_name'):
        assert _same(d[key][0], r[key][0]) and _same(d[key][1], r[key][1]), key
    assert d['articles'].equals(r['articles']) and d['articles_validate'].equals(r['articles_validate'])
    assert r['count_vectorizer'].vocabulary_ == d['count_vectorizer'].vocabulary_
    assert np.allclose(r['tfidf_transformer'].idf_, d['tfidf_transformer'].idf_)
    counts = read_file(model.data_dir + 'article_count_vectorized.npz')
    assert counts.max() > 1 and (counts != 0).nnz == d['binary'][0].nnz       # raw counts kept next to the binarised matrix

    enc, enc_v = np.random.RandomState(0).rand(40, 4), np.random.RandomState(1).rand(15, 4)
    cli.save_tsv(model, d, enc, enc_v)
    assert sorted(os.listdir(model.tsv_dir)) == sorted([
        'article_tfidf_vectorized.tsv', 'article_tfidf_vectorized_validate.tsv', 'article_binary_count_vectorized.tsv',
        'article_binary_count_vectorized_validate.tsv', 'article_label.tsv', 'article_label_validate.tsv', 'article_encoded.tsv',
        'article_encoded_validate.tsv'])                                         # main_autoencoder.py:294-301
    assert np.allclose(read_file(model.tsv_dir + 'article_encoded.tsv', data_type='numpy'), enc)
    assert (read_file(model.tsv_dir + 'article_binary_count_vectorized_validate.tsv', data_type='scipy') != d['binary'][1]).nnz == 0
    lab = read_file(model.tsv_dir + 'article_label.tsv')
    assert list(lab.columns) == ['label_story', 'label_category_publish_name', 'title', 'story', 'category_publish_name'] and len(lab) == 40


def test_uci_preparation_matches_the_reference_configuration(tmp_path):
    """C1 of BASELINE.json: 8000 x 10000 binary CSR from the UCI corpus (SURVEY 8d quotes nnz 1 241 293).  The preparation runs on
    the newest 300 articles of the corpus (tests/golden/uci_news_sample.parquet) and must give exactly what the reference's own
    vectoriser gives (tests/golden/uci_prep_sample.npz, oracle/gen_golden_uci_sample.py); the full-size matrices are the
    committed fixture tests/golden/uci_c1.npz, which the same preparation wrote from the whole corpus with the default flags."""
    import main_autoencoder as cli
    from helpers import load_uci_c1
    gold = np.load(os.path.join(ROOT, 'tests', 'golden', 'uci_prep_sample.npz'))
    F = cli.check_flags(cli.build_parser().parse_args([
        '--model_name', 'uci', '--data_path', os.path.join(ROOT, 'tests', 'golden', 'uci_news_sample.parquet'),
        '--train_row', str(int(gold['train_row'])), '--validate_row', str(int(gold['validate_row'])),
        '--max_features', str(int(gold['max_features']))]))
    d = cli.prepare_uci(F, None)
    assert list(d['count_vectorizer'].get_feature_names_out()) == list(gold['vocabulary'])
    for k, split in enumerate(('train', 'validate')):
        X, Xt = d['binary'][k].tocsr(), d['tfidf'][k].tocsr()
        X.sort_indices()
        Xt.sort_indices()
        assert X.shape == tuple(gold[split + '_shape'])
        assert (X.indptr == gold[split + '_indptr']).all() and (X.indices == gold[split + '_indices']).all()
        assert (X.data == 1).all() and (Xt.indptr == X.indptr).all() and (Xt.indices == X.indices).all()
        assert np.allclose(Xt.data, gold[split + '_tfidf'], rtol=1e-12, atol=0)
        assert (d['articles' if k == 0 else 'articles_validate'].article_id.values == gold[split + '_article_id']).all()
        for lab in ('category_publish_name', 'story'):
            assert (np.asarray(d['label_' + lab][k]) == gold['%s_label_%s' % (split, lab)]).all(), (split, lab)

    defaults = cli.check_flags(cli.build_parser().parse_args(['--model_name', 'uci']))
    assert (defaults.train_row, defaults.validate_row, defaults.max_features) == (8000, 2000, 10000)
    full = load_uci_c1()
    X, Xv = full['train'], full['validate']
    assert X.shape == (8000, 10000) and Xv.shape == (2000, 10000)
    assert abs(X.nnz - 1241293) <= 0.01 * 1241293
    assert len(np.unique(full['train_label_category_publish_name'])) == 4
