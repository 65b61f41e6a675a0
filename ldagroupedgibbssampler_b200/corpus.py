"""Corpus containers on the host side of the drop-in boundary.

The reference hands the sampler a MALLET ``InstanceList`` whose instances carry a ``FeatureSequence``
of type ids (reference: src/main/java/cc/mallet/util/LDAUtils.java:136-182,233-330).  This module
holds the minimum of that: an ``InstanceList`` mirror that flattens to CSR (``doc_offsets`` int64[D+1],
``tokens`` int32[N]), a reader for the reference's ``name<TAB>label<TAB>text`` files that is enough for
corpora (tokenizer classes, stop list, rare-word and TF-IDF pruning as LDAUtils.loadDataset applies
them), the named benchmark shapes of SURVEY section 8, and the token-balanced document sharding of
section 8(e).
"""
from __future__ import annotations

import re
from dataclasses import dataclass, field
from typing import Iterable, List, Optional, Sequence, Tuple

import numpy as np


class Alphabet:
    """First-seen-order vocabulary (MALLET Alphabet as StringList2FeatureSequence fills it)."""

    def __init__(self, entries: Optional[Iterable[str]] = None):
        self._list: List[str] = []
        self._index = {}
        for e in entries or []:
            self.lookupIndex(e)

    def lookupIndex(self, entry: str, add: bool = True) -> int:
        i = self._index.get(entry)
        if i is None:
            if not add:
                return -1
            i = len(self._list)
            self._index[entry] = i
            self._list.append(entry)
        return i

    def lookupObject(self, i: int) -> str:
        return self._list[i]

    def size(self) -> int:
        return len(self._list)

    def __len__(self) -> int:
        return len(self._list)

    def __eq__(self, other) -> bool:
        return isinstance(other, Alphabet) and self._list == other._list


@dataclass
class InstanceList:
    """Documents as arrays of type ids plus the alphabets, like MALLET's InstanceList of FeatureSequences."""

    docs: List[np.ndarray] = field(default_factory=list)
    alphabet: Alphabet = field(default_factory=Alphabet)
    names: List[str] = field(default_factory=list)
    labels: List[str] = field(default_factory=list)
    num_types: Optional[int] = None   # for synthetic corpora that have no strings

    def size(self) -> int:
        return len(self.docs)

    def getDataAlphabet(self) -> Alphabet:
        return self.alphabet

    def getNumTypes(self) -> int:
        return self.num_types if self.num_types is not None else self.alphabet.size()

    def to_csr(self) -> Tuple[np.ndarray, np.ndarray]:
        if getattr(self, "_csr", None) is not None:
            return self._csr
        lens = np.fromiter((len(d) for d in self.docs), np.int64, len(self.docs))
        off = np.zeros(len(self.docs) + 1, np.int64)
        np.cumsum(lens, out=off[1:])
        tokens = (np.concatenate([np.asarray(d, np.int32) for d in self.docs]) if off[-1] > 0
                  else np.zeros(0, np.int32))
        return off, np.ascontiguousarray(tokens, np.int32)

    @staticmethod
    def from_csr(doc_offsets: np.ndarray, tokens: np.ndarray, num_types: int) -> "InstanceList":
        il = InstanceList(num_types=int(num_types))
        il._csr = (np.ascontiguousarray(doc_offsets, np.int64), np.ascontiguousarray(tokens, np.int32))
        il.docs = _CsrDocs(*il._csr)
        return il


class _CsrDocs(Sequence):
    """Sequence view over a CSR corpus (so million-document synthetic corpora are not split into lists)."""

    def __init__(self, off, tokens):
        self.off, self.tokens = off, tokens

    def __len__(self):
        return len(self.off) - 1

    def __getitem__(self, d):
        if isinstance(d, slice):
            return [self[i] for i in range(*d.indices(len(self)))]
        return self.tokens[self.off[d]: self.off[d + 1]]


_LINE = re.compile(r"^(\S*)[\s,]*([^\t]+)[\s,]*(.*)$")   # LDAUtils.java:236

# Unicode general categories as the reference's tokenizers classify code points
# (pipe/SimpleTokenizerLarge.java:69-119, pipe/NumericAlsoTokenizer.java:59-100,
#  pipe/KeepConnectorPunctuationTokenizerLarge.java:69-110, pipe/KeepConnectorPunctuationNumericAlsoTokenizer.java:59-100)
_WORD = {"Ll", "Lu", "Mc", "Me", "Mn", "Lt", "Lm", "Lo"}
_DELIM = {"Zs", "Zl", "Zp", "Pe", "Pd", "Pc", "Ps", "Pi", "Pf", "Po"}


def tokenize(text: str, stop: Optional[set] = None, keep_numbers: bool = True, keep_connectors: bool = False,
             max_token_buffer: int = 10000) -> List[str]:
    """The reference's four tokenizer classes (LDAUtils.initTokenizer, util/LDAUtils.java:532-561) as one
    function.  Letters and marks build a token; separators and punctuation end it; with ``keep_numbers``
    decimal digits build tokens too (NumericAlsoTokenizer), with ``keep_connectors`` connector
    punctuation ("_", category Pc) does (KeepConnectorPunctuation*).  Every other code point -- digits
    without ``keep_numbers``, control characters such as TAB, symbols -- is skipped WITHOUT ending the
    token (SimpleTokenizerLarge.java:113-118), so "ab1c" is one token "abc" when numbers are dropped.
    A finished token is dropped when the stop list contains it.  A token longer than ``max_token_buffer``
    code points raises IndexError, the reference's ArrayIndexOutOfBoundsException on its fixed token buffer
    (``max_doc_buf_size``, SimpleTokenizerLarge.java:59; SimpleTokenizerLargeTest.java:48-75).  (The reference indexes
    ``Character.codePointAt`` with a code-point counter, SimpleTokenizerLarge.java:66-68, so it misreads text
    beyond the Basic Multilingual Plane; that quirk is not reproduced.)"""
    import unicodedata
    stop = stop if stop is not None else set()
    out: List[str] = []
    buf: List[str] = []
    for ch in text:
        cat = unicodedata.category(ch)
        if cat in _WORD or (keep_numbers and cat == "Nd") or (keep_connectors and cat == "Pc"):
            if len(buf) >= max_token_buffer:
                raise IndexError(f"token longer than the token buffer ({max_token_buffer})")
            buf.append(ch)
        elif cat in _DELIM:
            if buf:
                tok = "".join(buf)
                if tok not in stop:
                    out.append(tok)
                buf = []
    if buf:
        tok = "".join(buf)
        if tok not in stop:
            out.append(tok)
    return out


def _read_stoplist(stoplist) -> set:
    """A stop list file holds one word per line (MALLET SimpleTokenizer(File)); an iterable is taken as is."""
    if stoplist is None:
        return set()
    if isinstance(stoplist, str):
        with open(stoplist, "r", encoding="utf-8") as f:
            return {ln.strip() for ln in f if ln.strip()}
    return set(stoplist)


def _read_lines(path: str):
    """(name, label, lower-cased text) per line, CsvIterator with LDAUtils.java:236's regex + CharSequenceLowercase."""
    with open(path, "r", encoding="utf-8") as f:
        for line in f:
            line = line.rstrip("\n")
            if not line.strip():
                continue
            m = _LINE.match(line)
            if not m:
                continue
            yield m.group(1), m.group(2).strip(), m.group(3).lower()


def corpus_statistics(path: str, stop: set, keep_numbers: bool, keep_connectors: bool, alphabet: Alphabet,
                      max_token_buffer: int = 10000):
    """First pass of loadInstancesPrune / loadInstancesKeep: per word id its corpus count (tf,
    TfIdfPipe.getTf) and the number of documents containing it (df, TfIdfPipe.getIdf); returns (tf, df, D)."""
    tf: dict = {}
    df: dict = {}
    n_docs = 0
    for _, _, text in _read_lines(path):
        seen = set()
        for tok in tokenize(text, stop, keep_numbers, keep_connectors, max_token_buffer):
            i = alphabet.lookupIndex(tok)
            tf[i] = tf.get(i, 0) + 1
            if i not in seen:
                seen.add(i)
                df[i] = df.get(i, 0) + 1
        n_docs += 1
    return tf, df, n_docs


def tfidf_ranking(tf: dict, df: dict, n_docs: int, n_types: int) -> List[int]:
    """Word ids by ``tf * ln(D / df)`` descending (pipe/TfIdfPipe.java:75-104); ties: higher id first, MALLET's
    IDSorter order, which is what TfIdfPipeTest.java:118-137 expects ("a" 3, "is" 4, "this" 5)."""
    import math
    score = [(tf.get(i, 0) * math.log(n_docs / df[i]) if tf.get(i, 0) and df.get(i, 0) else 0.0) for i in range(n_types)]
    return sorted(range(n_types), key=lambda i: (-score[i], -i))


def load_dataset(path: str, stoplist=None, keep_numbers: bool = True, alphabet: Optional[Alphabet] = None,
                 rare_threshold: int = 0, keep_connectors: bool = False, tfidf_vocab_size: int = -1,
                 max_token_buffer: int = 10000, frozen_alphabet: bool = False) -> InstanceList:
    """``LDAUtils.loadDataset`` for a ``name<TAB>label<TAB>text`` file (util/LDAUtils.java:136-182):

    * ``tfidf_vocab_size > 0``: ``loadInstancesKeep`` (util/LDAUtils.java:353-460) -- a first pass counts, per
      word, its occurrences (tf) and the documents containing it (df); words are ranked by
      ``tf * ln(D / df)`` descending (pipe/TfIdfPipe.java:75-104) and everything from rank
      ``tfidf_vocab_size`` on joins the stop list (TfIdfPipe.java:162-172);
    * otherwise ``loadInstancesPrune`` (util/LDAUtils.java:233-330): with ``rare_threshold > 0`` a first pass
      counts the words and those seen fewer than ``rare_threshold`` times join the stop list (MALLET
      FeatureCountPipe.addPrunedWordsToStoplist; its source is not in the reference tree: restated from the
      2.0.8 release);
    * second pass: lower-case, tokenise, drop stop words, first-seen vocabulary order
      (StringList2FeatureSequence).  With a caller-supplied ``alphabet`` both passes share it, as in the
      reference, so pruned words keep their ids.

    Ties of the TF-IDF ranking follow MALLET's IDSorter (higher id first; restated from memory of 2.0.8).

    ``frozen_alphabet`` (a test set read with the training alphabet): the alphabet does not grow, words it does not
    hold are dropped as MALLET's pipes drop them once the alphabet is frozen, and the pruning passes are skipped (they
    are the training set's)."""
    stop = _read_stoplist(stoplist)
    if frozen_alphabet:
        if alphabet is None:
            raise ValueError("frozen_alphabet needs the training alphabet")
        il = InstanceList(alphabet=alphabet)
        for name, label, text in _read_lines(path):
            ids = [i for i in (alphabet.lookupIndex(tok, add=False)
                               for tok in tokenize(text, stop, keep_numbers, keep_connectors, max_token_buffer)) if i >= 0]
            il.docs.append(np.asarray(ids, np.int32))
            il.names.append(name)
            il.labels.append(label)
        return il
    if tfidf_vocab_size > 0 or rare_threshold > 0:
        first = alphabet if alphabet is not None else Alphabet()
        tf, df, n_docs = corpus_statistics(path, stop, keep_numbers, keep_connectors, first, max_token_buffer)
        stop = set(stop)
        if tfidf_vocab_size > 0:
            for i in tfidf_ranking(tf, df, n_docs, first.size())[tfidf_vocab_size:]:
                stop.add(first.lookupObject(i))
        else:
            for i in range(first.size()):
                if tf.get(i, 0) < rare_threshold:
                    stop.add(first.lookupObject(i))
    il = InstanceList(alphabet=alphabet if alphabet is not None else Alphabet())
    for name, label, text in _read_lines(path):
        ids = [il.alphabet.lookupIndex(tok) for tok in tokenize(text, stop, keep_numbers, keep_connectors, max_token_buffer)]
        il.docs.append(np.asarray(ids, np.int32))
        il.names.append(name)
        il.labels.append(label)
    return il


# --------------------------------------------------------------------------------------------
# named shapes (SURVEY section 8 size table; reference: src/main/resources/datasets/README.txt:3-31)
# --------------------------------------------------------------------------------------------
SHAPES = {
    # name: (D, V, mean document length, K, scheme, alpha, beta)
    "nips": dict(D=1500, V=12419, mean_len=1267.0, K=100, scheme="gpu_ggs", alpha=1.0, beta=0.01),
    "enron": dict(D=39861, V=28102, mean_len=161.0, K=400, scheme="gpu_pcgs", alpha=50.0 / 400, beta=0.01),
    "pubmed": dict(D=8200000, V=141043, mean_len=90.0, K=1000, scheme="gpu_ggs", alpha=50.0 / 1000, beta=0.01),
}


def shard_documents_by_tokens(doc_offsets: np.ndarray, world: int) -> List[Tuple[int, int]]:
    """Contiguous document ranges with (nearly) equal token counts, one per rank (SURVEY 8e:
    balance by tokens, not by document count as the reference's EvenSplitBatchBuilder does,
    topics/randomscan/document/EvenSplitBatchBuilder.java:30-44).  Returns [(d0, d1)] per rank."""
    off = np.asarray(doc_offsets, np.int64)
    D, N = len(off) - 1, int(off[-1])
    cuts = [0]
    for r in range(1, world):
        target = N * r // world
        d = int(np.searchsorted(off, target, side="left"))
        d = min(max(d, cuts[-1]), D)
        cuts.append(d)
    cuts.append(D)
    return [(cuts[r], cuts[r + 1]) for r in range(world)]


def take_shard(doc_offsets: np.ndarray, tokens: np.ndarray, d0: int, d1: int):
    """Local CSR of documents [d0, d1) plus the global bases the library keys its counters with."""
    off = np.asarray(doc_offsets, np.int64)
    t0, t1 = int(off[d0]), int(off[d1])
    return (off[d0: d1 + 1] - t0).astype(np.int64), np.ascontiguousarray(tokens[t0:t1], np.int32), d0, t0


def write_synthetic_corpus(path: str, D: int, V: int, mean_len: float, seed: int = 20190529, chunk: int = 100000):
    """Write a synthetic corpus of a BASELINE shape (SURVEY 8d, the generator of ``synth_corpus``) in the reference's
    ``name<TAB>label<TAB>text`` format (util/LDAUtils.java:233-330) so that the Java driver can read the very corpus the
    GPU benchmark samples (scripts/run_java_baseline.sh).  Type w becomes the word ``w<id>``."""
    from ._lib import synth_corpus
    with open(path, "w") as f:
        for d0 in range(0, D, chunk):
            n = min(chunk, D - d0)
            off, tokens = synth_corpus(n, V, mean_len, seed=seed, doc_first=d0)
            for d in range(n):
                f.write("doc%d\tX\t%s\n" % (d0 + d, " ".join("w%d" % t for t in tokens[off[d]:off[d + 1]])))
