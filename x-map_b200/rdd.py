"""A minimal local stand-in for the RDD surface the pipelines hand to callers.

The reference returns PySpark RDDs from every pipeline (assist.py:9-150).  When
the caller passes a real SparkContext the facades wrap their results with
``sc.parallelize``; when ``sc`` is None (no Spark installed -- the case on the
GPU boxes) they return a ``LocalRDD``: an eager, single-partition, list-backed
object with the transformations downstream code uses (the recommender stages
call map / flatMap / filter / mapPartitions / reduceByKey / join / collect /
collectAsMap on the AlterEgo RDD, recommenderSim.py:15-75).

``LazyRDD`` defers building Python records until somebody actually looks at
them, so that device-resident results (hundreds of millions of similarity
pairs) can flow from one pipeline stage to the next without ever becoming
Python tuples.
"""
import numpy as np


class Broadcast(object):
    def __init__(self, value):
        self.value = value


class LocalRDD(object):
    def __init__(self, records=()):
        self._records = list(records)

    # subclasses may compute lazily
    def _data(self):
        return self._records

    def _new(self, it):
        return LocalRDD(it)

    def cache(self):
        return self

    persist = cache

    def collect(self):
        return list(self._data())

    def collectAsMap(self):
        return dict(self._data())

    def take(self, n):
        return list(self._data()[:n])

    def first(self):
        return self._data()[0]

    def count(self):
        return len(self._data())

    def map(self, f):
        return self._new(f(x) for x in self._data())

    def flatMap(self, f):
        return self._new(y for x in self._data() for y in f(x))

    def filter(self, f):
        return self._new(x for x in self._data() if f(x))

    def mapPartitions(self, f):
        return self._new(f(iter(self._data())))

    def keys(self):
        return self._new(k for k, _ in self._data())

    def values(self):
        return self._new(v for _, v in self._data())

    def union(self, other):
        return self._new(list(self._data()) + list(other.collect()))

    def distinct(self):
        return self._new(dict.fromkeys(self._data()))

    def intersection(self, other):
        theirs = set(other.collect())
        return self._new(x for x in dict.fromkeys(self._data()) if x in theirs)

    def combineByKey(self, create, merge_value, merge_combiners=None):
        acc = {}
        for k, v in self._data():
            acc[k] = merge_value(acc[k], v) if k in acc else create(v)
        return self._new(acc.items())

    def reduceByKey(self, f):
        return self.combineByKey(lambda v: v, f)

    def groupByKey(self):
        return self.combineByKey(lambda v: [v], lambda a, v: a + [v])

    def join(self, other):
        right = {}
        for k, v in other.collect():
            right.setdefault(k, []).append(v)
        return self._new((k, (v, w)) for k, v in self._data() for w in right.get(k, ()))

    def reduce(self, f):
        it = iter(self._data())
        acc = next(it)
        for x in it:
            acc = f(acc, x)
        return acc

    def randomSplit(self, weights, seed=None):
        cell = split_cells(weights, seed, len(self._data()))
        return [self._new(x for x, c in zip(self._data(), cell) if c == i) for i in range(len(weights))]


class LazyRDD(LocalRDD):
    """Records are produced by ``builder()`` on first use; ``handle`` carries the
    device-resident result for the next pipeline stage."""

    def __init__(self, builder, handle=None):
        self._builder = builder
        self._records = None
        self.handle = handle

    def _data(self):
        if self._records is None:
            self._records = list(self._builder())
        return self._records


def split_cells(weights, seed, n):
    """The part randomSplit puts each of n records in: one RandomState(seed % 2**32) uniform per record."""
    w = np.asarray(weights, dtype=np.float64)
    edges = np.cumsum(w / w.sum())
    rng = np.random.RandomState(None if seed is None else seed % (2 ** 32))
    return np.minimum(np.searchsorted(edges, rng.random_sample(n), side="right"), len(w) - 1)


class LocalContext(object):
    """What the pipelines need from a SparkContext when none is supplied."""

    def parallelize(self, data, numSlices=None):
        return LocalRDD(data)

    def broadcast(self, value):
        return Broadcast(value)

    def textFile(self, path, minPartitions=None):
        if path.startswith("file:"):
            path = path[5:]
        with open(path) as f:
            return LocalRDD(line.rstrip("\n") for line in f if line.strip())


def context_of(sc):
    return LocalContext() if sc is None else sc


def records_of(rdd):
    """Records of a LocalRDD, a real RDD, or any iterable."""
    return rdd.collect() if hasattr(rdd, "collect") else list(rdd)
