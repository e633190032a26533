#!/usr/bin/env python
"""Generate tests/golden/uci_news_sample.parquet and tests/golden/uci_prep_sample.npz (test infrastructure).

    python oracle/gen_golden_uci_sample.py <reference checkout>

The sample is the newest SAMPLE_ROWS articles of the reference's UCI news corpus (datasets/uci_news.snappy.parquet), with
the columns the preparation reads and main_content cut to CONTENT_CHARS characters so that the fixture stays small.  The
golden arrays are what the reference's own datasets/articles.py (read_articles, count_vectorize, tfidf_transform; imported
unmodified, with its unused `jieba` import stubbed) makes of that sample, selected and ordered as main_autoencoder.py:177-224
does for the CLI defaults (triplet strategy batch_all, label category_publish_name, min_df 0, max_df 0.99) at the small sizes
below.  tests/test_io_formats.py runs the CLI's prepare_uci on the sample and compares.
"""
import os
import sys
import types

import numpy as np
import pandas as pd

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
OUT = os.path.join(ROOT, 'tests', 'golden')
SAMPLE_ROWS, CONTENT_CHARS = 300, 400
TRAIN_ROW, VALIDATE_ROW, MAX_FEATURES = 220, 60, 800
COLUMNS = ['article_id', 'title', 'story', 'category_publish_name', 'main_content']


def main(ref):
    sys.modules.setdefault('jieba', types.ModuleType('jieba'))    # only articles.tokenizer_chinese uses it; tokenizer=None below
    sys.path.insert(0, ref)
    from datasets import articles as ref_articles  # noqa: E402  (reference code)

    corpus = pd.read_parquet(os.path.join(ref, 'datasets', 'uci_news.snappy.parquet'), columns=COLUMNS)
    sample = corpus.loc[corpus.article_id.nlargest(SAMPLE_ROWS).index].sort_index().reset_index(drop=True)
    sample['main_content'] = sample.main_content.str.slice(0, CONTENT_CHARS)
    sample_path = os.path.join(OUT, 'uci_news_sample.parquet')
    sample.to_parquet(sample_path, compression='gzip', index=False)

    df = ref_articles.read_articles(path=sample_path)
    df.index.name = None          # pandas >= 2 refuses to sort by a name that is both the index and a column
    df = df.sort_index(ascending=False)
    df['label_story'] = pd.factorize(df.story)[0]
    df['label_category_publish_name'] = pd.factorize(df.category_publish_name.apply(lambda s: s.lstrip('即時')))[0]
    df = df.loc[df.category_publish_name.notna()]                  # label_category_publish_name_valid == 1
    df = df.iloc[0:TRAIN_ROW + VALIDATE_ROW].sort_values('article_id')
    cv, X, _, _ = ref_articles.count_vectorize(df.main_content[0:TRAIN_ROW], tokenizer=None, stop_words='english', min_df=0.0,
                                               max_df=0.99, max_features=MAX_FEATURES, binary=False)
    Xv = cv.transform(df.main_content[TRAIN_ROW:TRAIN_ROW + VALIDATE_ROW])
    tf, Xt = ref_articles.tfidf_transform(X)
    out = {'train_row': np.int64(TRAIN_ROW), 'validate_row': np.int64(VALIDATE_ROW), 'max_features': np.int64(MAX_FEATURES),
           'vocabulary': np.array(cv.get_feature_names_out()).astype(str)}
    for split, sl, counts, tfidf in (('train', slice(0, TRAIN_ROW), X, Xt),
                                     ('validate', slice(TRAIN_ROW, TRAIN_ROW + VALIDATE_ROW), Xv, tf.transform(Xv))):
        counts, tfidf = counts.tocsr(), tfidf.tocsr()
        counts.sort_indices()
        tfidf.sort_indices()
        out[split + '_shape'] = np.array(counts.shape)
        out[split + '_indptr'] = counts.indptr.astype(np.int32)
        out[split + '_indices'] = counts.indices.astype(np.int32)
        out[split + '_counts'] = counts.data.astype(np.int32)
        out[split + '_tfidf'] = tfidf.data.astype(np.float64)
        out[split + '_article_id'] = df.article_id.values[sl].astype(np.int64)
        for lab in ('category_publish_name', 'story'):
            out['%s_label_%s' % (split, lab)] = df['label_' + lab].values[sl].astype(np.int32)
    np.savez_compressed(os.path.join(OUT, 'uci_prep_sample.npz'), **out)
    print({k: v.shape for k, v in out.items()}, 'nnz', X.nnz, Xv.nnz)


if __name__ == '__main__':
    main(sys.argv[1])
