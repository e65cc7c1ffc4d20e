"""Rank the gene pairs a trained digenic model has not seen: exhaustive top-N over all pairs of a gene set, on the device.

    python -m trigenicinteractionpredictor_b200.predict_pairs -t train_mixed.dat -e test_mixed.dat \\
        -p results/Sample_0_K10.npz [-p results/Sample_1_K10.npz ...] [-n 100] [-g genes.txt] [-q queries.txt] \\
        [--include-known] [-o predictions.tsv] [--device cuda:0]

The mixed train / test files rebuild the digenic model's digestion (TrigenicInteractionPredictor_23.Model.get_train_test);
every parameter file (the .npz that the digenic command line writes with --save-params) must belong to it.  With several
files the score of a pair is the mean of the models' scores (DESIGN §4.11).  Pairs that are pair keys of the train or
test file are left out unless --include-known.  -g: one gene name per line, the candidates (default: all genes).

Output: a header line "Predicted Interaction<TAB>ID of genes<TAB>Genes", then one line per pair, best first: the score,
the id key "a_b" in slot order, and the two gene names sorted by name.

-q: one query gene name per line.  Then -n counts per query: for every query, in file order, the -n best pairs that
contain it, the partner taken from the -g genes plus the queries (default: all genes).  The header is
"Query gene<TAB>Predicted Interaction<TAB>ID of genes<TAB>Genes" and every line starts with its query's name."""
from __future__ import annotations

import contextlib
import getopt
import os
import sys

HEADER = "Predicted Interaction\tID of genes\tGenes\n"
QUERY_HEADER = "Query gene\t" + HEADER


def _fail(msg: str) -> int:
    print("ERROR: " + msg, file=sys.stderr)
    return 2


def main(argv=None) -> int:
    argv = sys.argv[1:] if argv is None else argv
    train = test = out = device = genes_file = queries_file = None
    params: list[str] = []
    top, include_known = 100, False
    try:
        opts, rest = getopt.getopt(argv, "ht:e:p:n:g:q:o:", ["help", "train=", "test=", "params=", "top=", "genes=",
                                                             "queries=", "include-known", "out=", "device="])
    except getopt.GetoptError as exc:
        return _fail("argument error: %s" % exc)
    if rest:
        return _fail("unexpected arguments: %s" % " ".join(rest))
    for opt, arg in opts:
        if opt in ("-h", "--help"):
            print(__doc__)
            return 0
        if opt in ("-t", "--train"):
            train = arg
        elif opt in ("-e", "--test"):
            test = arg
        elif opt in ("-p", "--params"):
            params.append(arg)
        elif opt in ("-n", "--top"):
            try:
                top = int(arg)
            except ValueError:
                return _fail("--top must be an integer (got %r)" % arg)
        elif opt in ("-g", "--genes"):
            genes_file = arg
        elif opt in ("-q", "--queries"):
            queries_file = arg
        elif opt == "--include-known":
            include_known = True
        elif opt in ("-o", "--out"):
            out = arg
        elif opt == "--device":
            device = arg
    if top < 1:
        return _fail("--top must be positive (got %d)" % top)
    if train is None or test is None or not params:
        return _fail("-t/--train, -e/--test and at least one -p/--params are required")
    for path in [train, test, *params] + [f for f in (genes_file, queries_file) if f]:
        if not os.path.isfile(path):
            return _fail("the file %s does not exist" % path)
    if out is not None and os.path.dirname(os.path.abspath(out)) and not os.path.isdir(os.path.dirname(os.path.abspath(out))):
        return _fail("the directory of %s does not exist" % out)

    from .TrigenicInteractionPredictor_23 import Model
    model = Model(device=device)
    with contextlib.redirect_stdout(sys.stderr):      # the digestion's "READ DATA" lines are not part of the table
        model.get_train_test(train, test)
    genes = None
    if genes_file:
        with open(genes_file, encoding="utf-8") as fh:
            genes = [line.strip() for line in fh if line.strip()]
        unknown = [g for g in genes if g not in model.gene_id]
        if unknown:
            return _fail("genes not in the train / test files: %s" % ", ".join(unknown))
    queries = None
    if queries_file:
        with open(queries_file, encoding="utf-8") as fh:
            queries = [line.strip() for line in fh if line.strip()]
        if not queries:
            return _fail("the query file %s names no gene" % queries_file)
        unknown = [g for g in queries if g not in model.gene_id]
        if unknown:
            return _fail("query genes not in the train / test files: %s" % ", ".join(unknown))
        seen, twice = set(), []
        for g in queries:
            if g in seen and g not in twice:
                twice.append(g)
            seen.add(g)
        if twice:
            return _fail("query genes listed twice: %s" % ", ".join(twice))
    sets = []
    for path in params:
        try:
            th, _, q = model.check_parameters_file(path)
        except ValueError as exc:
            return _fail(str(exc))
        sets.append((th, q))
    if len({th.shape[1] for th, _ in sets}) != 1:
        return _fail("the parameter files have different K")

    if queries is None:
        rows = model.predict_top_pairs(top, genes=genes, exclude_known=not include_known, params=sets)
        text = HEADER + "".join(str(s) + "\t" + key + "\t" + names + "\n" for s, key, names in rows)
    else:
        per = model.predict_top_pairs_per_gene(queries, top, genes=genes, exclude_known=not include_known, params=sets)
        text = QUERY_HEADER + "".join(q + "\t" + str(s) + "\t" + key + "\t" + names + "\n"
                                      for q in queries for s, key, names in per[q])
    if out is None:
        sys.stdout.write(text)
    else:
        with open(out, "w", encoding="utf-8") as fh:
            fh.write(text)
    return 0


if __name__ == "__main__":
    sys.exit(main())
