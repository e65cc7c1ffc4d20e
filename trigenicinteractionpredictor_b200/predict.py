"""Rank the triplets a trained model has not seen: exhaustive top-N over all triplets of a gene set, on the device.

    python -m trigenicinteractionpredictor_b200.predict -t train0.dat -e test0.dat \\
        -p results/Sample_0_K10.npz [-p results/Sample_1_K10.npz ...] [-n 100] [-g genes.txt] \\
        [-q queries.txt | -r pairs.txt | --held-out | --held-out-pairs [-r pairs.txt] | --held-out-genes [-q queries.txt]]
        [--include-known] [-o predictions.tsv] [--device cuda:0]

The train / test files rebuild the model's digestion (gene ids in order of first appearance, TIP.py:321-423); every
parameter file (the .npz that training with --save-params writes) must belong to it.  With several files the score of a
triplet is the mean of the models' scores.  Triplets that are keys of the train or test file are left out unless
--include-known.  -g: one gene name per line, the candidates (default: all genes).

Output: a header line "Predicted Interaction<TAB>ID of genes<TAB>Genes", then one line per triplet, best first: the score,
the id key as in the report's "ID of genes" column, and the gene names sorted by name (the fold-file format).

-q: one query gene name per line.  Then -n counts per query: for every query, in file order, the -n best triplets that
contain it, the two partners taken from the -g genes plus the queries (default: all genes).  The header is
"Query gene<TAB>Predicted Interaction<TAB>ID of genes<TAB>Genes" and every line starts with its query's name.

-r: one query pair per line, written nameA+nameB (the raw screens' notation for a double-mutant query) or as two
whitespace-separated names.  Then -n counts per pair: for every pair, in file order, the -n best triplets that contain
both genes, the third taken from the -g genes plus the pairs' genes (default: all genes).  The header is
"Query pair<TAB>Predicted Interaction<TAB>ID of genes<TAB>Genes" and every line starts with its pair, written nameA+nameB.
-q and -r exclude each other.

--held-out: where the test file's triplets land among all unseen triplets (Model.rank_held_out, DESIGN §4.8): the
universe is every triplet of the -g genes (default: all genes) that is not a key of the train file, ranked by score, and
-n is the number of its best triplets ranked exactly (default 100000).  Below them a rank is an interval lo-hi that holds
the exact rank.  Output: summary lines "Name:<TAB>value" (universe size, counts, recall at N for the positives and the
negatives, the positives' median rank and AUC against the universe, each as lo or lo-hi), then the header
"Rank<TAB>Predicted Interaction<TAB>Real Interaction<TAB>ID of genes<TAB>Genes" and one line per ranked test triplet, best
first.  --held-out excludes -q, -r and --include-known.

--held-out-pairs: where each test triplet lands among its query pair's unseen partners (Model.rank_held_out_per_pair,
DESIGN §4.9).  Without -r every test triplet of the -g genes gives three views, one per pair of its genes; with -r a view
is a listed pair and a test triplet that contains both of its genes, the third taken from the -g genes plus the pairs'
genes.  A pair's universe is every partner whose triplet is not a key of the train file, and every rank is exact.
Output: summary lines "Name:<TAB>value" (counts, hits at N for the positives and the negatives, the positives' median
rank, MRR and AUC against the pair universes), then the header "Query pair<TAB>Rank<TAB>Pair universe<TAB>Predicted
Interaction<TAB>Real Interaction<TAB>ID of genes<TAB>Genes" and one line per view, by pair (file order, or sorted names)
and rank.  --held-out-pairs excludes -q, -n, --held-out and --include-known.

--held-out-genes: where each test triplet lands among its query gene's unseen triplets (Model.rank_held_out_per_gene,
DESIGN §4.10).  Without -q every test triplet of the -g genes gives three views, one per gene; with -q a view is a listed
query and a test triplet that contains it, the partners taken from the -g genes plus the queries.  A query's universe is
every pair of other genes whose triplet is not a key of the train file, and every rank is exact.  Output: summary lines
"Name:<TAB>value" (counts, hits at N for the positives and the negatives, the positives' median rank, MRR and AUC against
the gene universes), then the header "Query gene<TAB>Rank<TAB>Gene universe<TAB>Predicted Interaction<TAB>Real
Interaction<TAB>ID of genes<TAB>Genes" and one line per view, by query (file order, or sorted names) and rank.
--held-out-genes excludes -r, -n, --held-out, --held-out-pairs and --include-known."""
from __future__ import annotations

import contextlib
import getopt
import os
import sys

HEADER = "Predicted Interaction\tID of genes\tGenes\n"
QUERY_HEADER = "Query gene\t" + HEADER
PAIR_HEADER = "Query pair\t" + HEADER
HELD_OUT_HEADER = "Rank\tPredicted Interaction\tReal Interaction\tID of genes\tGenes\n"
HELD_OUT_PAIRS_HEADER = "Query pair\tRank\tPair universe\tPredicted Interaction\tReal Interaction\tID of genes\tGenes\n"
HELD_OUT_GENES_HEADER = "Query gene\tRank\tGene universe\tPredicted Interaction\tReal Interaction\tID of genes\tGenes\n"
RECALL_AT = (100, 1000, 10000, 100000)
HITS_AT = (1, 5, 10, 20, 50, 100)
GENE_HITS_AT = (1, 10, 20, 100, 1000, 10000)


def _fail(msg: str) -> int:
    print("ERROR: " + msg, file=sys.stderr)
    return 2


def main(argv=None) -> int:
    argv = sys.argv[1:] if argv is None else argv
    train = test = out = device = genes_file = queries_file = pairs_file = None
    params: list[str] = []
    top, include_known, held_out, held_out_pairs, held_out_genes = None, False, False, False, False
    try:
        opts, rest = getopt.getopt(argv, "ht:e:p:n:g:q:r:o:", ["help", "train=", "test=", "params=", "top=", "genes=",
                                                               "queries=", "pairs=", "include-known", "held-out",
                                                               "held-out-pairs", "held-out-genes", "out=", "device="])
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
        elif opt in ("-r", "--pairs"):
            pairs_file = arg
        elif opt == "--include-known":
            include_known = True
        elif opt == "--held-out":
            held_out = True
        elif opt == "--held-out-pairs":
            held_out_pairs = True
        elif opt == "--held-out-genes":
            held_out_genes = True
        elif opt in ("-o", "--out"):
            out = arg
        elif opt == "--device":
            device = arg
    if held_out_genes:
        if pairs_file or top is not None or held_out or held_out_pairs or include_known:
            return _fail("--held-out-genes excludes -r/--pairs, -n/--top, --held-out, --held-out-pairs and --include-known")
    elif held_out_pairs:
        if queries_file or held_out or include_known or top is not None:
            return _fail("--held-out-pairs excludes -q/--queries, -n/--top, --held-out and --include-known")
    elif held_out:
        if queries_file or pairs_file or include_known:
            return _fail("--held-out excludes -q/--queries, -r/--pairs and --include-known")
        top = 100000 if top is None else top
        if top < 0:
            return _fail("--top must be >= 0 with --held-out (got %d)" % top)
    else:
        top = 100 if top is None else top
        if top < 1:
            return _fail("--top must be positive (got %d)" % top)
    if train is None or test is None or not params:
        return _fail("-t/--train, -e/--test and at least one -p/--params are required")
    if queries_file and pairs_file:
        return _fail("-q/--queries and -r/--pairs exclude each other")
    for path in [train, test, *params] + [f for f in (genes_file, queries_file, pairs_file) if f]:
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
    pairs = None
    if pairs_file:
        pairs = []
        with open(pairs_file, encoding="utf-8") as fh:
            for no, line in enumerate(fh, 1):
                if not line.strip():
                    continue
                pair = line.strip().split("+") if "+" in line else line.split()
                if len(pair) != 2 or not all(g.strip() for g in pair) or any(len(g.split()) != 1 for g in pair):
                    return _fail("line %d of %s is not a pair nameA+nameB or nameA nameB: %r" % (no, pairs_file, line.strip()))
                pairs.append((pair[0].strip(), pair[1].strip()))
        if not pairs:
            return _fail("the pair file %s names no pair" % pairs_file)
        unknown = list(dict.fromkeys(g for p in pairs for g in p if g not in model.gene_id))
        if unknown:
            return _fail("pair genes not in the train / test files: %s" % ", ".join(unknown))
        single = [p for p in pairs if p[0] == p[1]]
        if single:
            return _fail("a pair of one gene: %s" % "+".join(single[0]))
        seen, twice = set(), []
        for p in pairs:
            if frozenset(p) in seen and "+".join(p) not in twice:
                twice.append("+".join(p))
            seen.add(frozenset(p))
        if twice:
            return _fail("pairs listed twice: %s" % ", ".join(twice))
    sets = []
    for path in params:
        try:
            sets.append(model.check_parameters_file(path))
        except ValueError as exc:
            return _fail(str(exc))
    if len({th.shape[1] for th, _ in sets}) != 1:
        return _fail("the parameter files have different K")

    if held_out_genes:
        try:
            res = model.rank_held_out_per_gene(queries, genes=genes, params=sets, hits_at=GENE_HITS_AT)
        except ValueError as exc:
            return _fail(str(exc))
        text = held_out_genes_text(res)
    elif held_out_pairs:
        try:
            res = model.rank_held_out_per_pair(pairs, genes=genes, params=sets, hits_at=HITS_AT)
        except ValueError as exc:
            return _fail(str(exc))
        text = held_out_pairs_text(res)
    elif held_out:
        try:
            res = model.rank_held_out(top, genes=genes, params=sets, recall_at=RECALL_AT)
        except ValueError as exc:
            return _fail(str(exc))
        text = held_out_text(res)
    elif pairs is not None:
        per = model.predict_top_triplets_per_pair(pairs, top, genes=genes, exclude_known=not include_known, params=sets)
        text = PAIR_HEADER + "".join(p[0] + "+" + p[1] + "\t" + str(s) + "\t" + key + "\t" + names + "\n"
                                     for p in pairs for s, key, names in per[p])
    elif queries is None:
        rows = model.predict_top_triplets(top, genes=genes, exclude_known=not include_known, params=sets)
        text = HEADER + "".join(str(s) + "\t" + key + "\t" + names + "\n" for s, key, names in rows)
    else:
        per = model.predict_top_triplets_per_gene(queries, top, genes=genes, exclude_known=not include_known, params=sets)
        text = QUERY_HEADER + "".join(q + "\t" + str(s) + "\t" + key + "\t" + names + "\n"
                                      for q in queries for s, key, names in per[q])
    if out is None:
        sys.stdout.write(text)
    else:
        with open(out, "w", encoding="utf-8") as fh:
            fh.write(text)
    return 0


def _interval(v) -> str:
    if v is None:
        return "n/a"
    lo, hi = v
    return str(lo) if lo == hi else "%s-%s" % (lo, hi)


def held_out_text(res: dict) -> str:
    """Summary lines and the table of ranked test triplets of Model.rank_held_out."""
    lines = ["Universe size:\t%d" % res["universe"], "Exactly ranked:\t%d" % res["n_exact"],
             "Ranked positives:\t%d" % res["positives"], "Ranked negatives:\t%d" % res["negatives"],
             "Excluded train keys:\t%d" % res["excluded_train"], "Excluded outside the genes:\t%d" % res["excluded_genes"]]
    for N, r in res["recall_at"].items():
        lines.append("Recall at %d:\t%s" % (N, _interval(r["positives"])))
        lines.append("Negatives at %d:\t%s" % (N, _interval(r["negatives"])))
    lines.append("Median rank of positives:\t%s" % _interval(res["median_rank"]))
    lines.append("Universe AUC:\t%s" % _interval(res["auc"]))
    body = "".join("%s\t%s\t%d\t%s\t%s\n" % (_interval((lo, hi)), score, label, key, names)
                   for key, names, label, score, lo, hi in res["rows"])
    return "\n".join(lines) + "\n" + HELD_OUT_HEADER + body


def _value(v) -> str:
    return "n/a" if v is None else str(v)


def held_out_pairs_text(res: dict) -> str:
    """Summary lines and the table of views of Model.rank_held_out_per_pair."""
    lines = ["Query pairs:\t%d" % len(res["pairs"]), "Views:\t%d" % res["views"], "Positive views:\t%d" % res["positives"],
             "Negative views:\t%d" % res["negatives"], "Excluded train keys:\t%d" % res["excluded_train"],
             "Excluded outside the genes:\t%d" % res["excluded_genes"]]
    for N, r in res["hits_at"].items():
        lines.append("Hits at %d:\t%s" % (N, _value(r["positives"])))
        lines.append("Negatives at %d:\t%s" % (N, _value(r["negatives"])))
    lines += ["Median rank of positives:\t%s" % _value(res["median_rank"]), "MRR:\t%s" % _value(res["mrr"]),
              "Pair AUC (micro):\t%s" % _value(res["auc_micro"]), "Pair AUC (macro):\t%s" % _value(res["auc_macro"])]
    body = "".join("%s\t%d\t%d\t%s\t%d\t%s\t%s\n" % (pair, rank, universe, score, label, key, names)
                   for pair, key, names, label, score, rank, universe in res["rows"])
    return "\n".join(lines) + "\n" + HELD_OUT_PAIRS_HEADER + body


def held_out_genes_text(res: dict) -> str:
    """Summary lines and the table of views of Model.rank_held_out_per_gene."""
    lines = ["Query genes:\t%d" % len(res["genes"]), "Views:\t%d" % res["views"], "Positive views:\t%d" % res["positives"],
             "Negative views:\t%d" % res["negatives"], "Excluded train keys:\t%d" % res["excluded_train"],
             "Excluded outside the genes:\t%d" % res["excluded_genes"]]
    for N, r in res["hits_at"].items():
        lines.append("Hits at %d:\t%s" % (N, _value(r["positives"])))
        lines.append("Negatives at %d:\t%s" % (N, _value(r["negatives"])))
    lines += ["Median rank of positives:\t%s" % _value(res["median_rank"]), "MRR:\t%s" % _value(res["mrr"]),
              "Gene AUC (micro):\t%s" % _value(res["auc_micro"]), "Gene AUC (macro):\t%s" % _value(res["auc_macro"])]
    body = "".join("%s\t%d\t%d\t%s\t%d\t%s\t%s\n" % (gene, rank, universe, score, label, key, names)
                   for gene, key, names, label, score, rank, universe in res["rows"])
    return "\n".join(lines) + "\n" + HELD_OUT_GENES_HEADER + body


if __name__ == "__main__":
    sys.exit(main())
