"""Rank the triplets a trained model has not seen: exhaustive top-N over all triplets of a gene set, on the device.

    python -m trigenicinteractionpredictor_b200.predict -t train0.dat -e test0.dat \\
        -p results/Sample_0_K10.npz [-p results/Sample_1_K10.npz ...] [-n 100] [-g genes.txt] [--include-known] \\
        [-o predictions.tsv] [--device cuda:0]

The train / test files rebuild the model's digestion (gene ids in order of first appearance, TIP.py:321-423); every
parameter file (the .npz that training with --save-params writes) must belong to it.  With several files the score of a
triplet is the mean of the models' scores.  Triplets that are keys of the train or test file are left out unless
--include-known.  -g: one gene name per line, the candidates (default: all genes).

Output: a header line "Predicted Interaction<TAB>ID of genes<TAB>Genes", then one line per triplet, best first: the score,
the id key as in the report's "ID of genes" column, and the gene names sorted by name (the fold-file format)."""
from __future__ import annotations

import contextlib
import getopt
import os
import sys

HEADER = "Predicted Interaction\tID of genes\tGenes\n"


def _fail(msg: str) -> int:
    print("ERROR: " + msg, file=sys.stderr)
    return 2


def main(argv=None) -> int:
    argv = sys.argv[1:] if argv is None else argv
    train = test = out = device = genes_file = None
    params: list[str] = []
    top, include_known = 100, False
    try:
        opts, rest = getopt.getopt(argv, "ht:e:p:n:g:o:", ["help", "train=", "test=", "params=", "top=", "genes=",
                                                           "include-known", "out=", "device="])
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
            if top < 1:
                return _fail("--top must be positive (got %d)" % top)
        elif opt in ("-g", "--genes"):
            genes_file = arg
        elif opt == "--include-known":
            include_known = True
        elif opt in ("-o", "--out"):
            out = arg
        elif opt == "--device":
            device = arg
    if train is None or test is None or not params:
        return _fail("-t/--train, -e/--test and at least one -p/--params are required")
    for path in [train, test, *params] + ([genes_file] if genes_file else []):
        if not os.path.isfile(path):
            return _fail("the file %s does not exist" % path)
    if out is not None and os.path.dirname(os.path.abspath(out)) and not os.path.isdir(os.path.dirname(os.path.abspath(out))):
        return _fail("the directory of %s does not exist" % out)

    from .TrigenicInteractionPredictor import Model
    model = Model(device=device)
    with contextlib.redirect_stdout(sys.stderr):      # the digestion's "READ DATA" lines are not part of the table
        model.get_traintest(train, test)
    genes = None
    if genes_file:
        with open(genes_file, encoding="utf-8") as fh:
            genes = [line.strip() for line in fh if line.strip()]
        unknown = [g for g in genes if g not in model.gene_id]
        if unknown:
            return _fail("genes not in the train / test files: %s" % ", ".join(unknown))
    sets = []
    for path in params:
        try:
            sets.append(model.check_parameters_file(path))
        except ValueError as exc:
            return _fail(str(exc))
    if len({th.shape[1] for th, _ in sets}) != 1:
        return _fail("the parameter files have different K")

    rows = model.predict_top_triplets(top, genes=genes, exclude_known=not include_known, params=sets)
    text = HEADER + "".join(str(s) + "\t" + key + "\t" + names + "\n" for s, key, names in rows)
    if out is None:
        sys.stdout.write(text)
    else:
        with open(out, "w", encoding="utf-8") as fh:
            fh.write(text)
    return 0


if __name__ == "__main__":
    sys.exit(main())
